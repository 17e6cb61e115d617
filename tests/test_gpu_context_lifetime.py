"""Lifetime of a C ABI context: closing it gives back all of its device memory, and a Gram matrix is only read back while it
is still the last Gram result (the IBS and KING calls reuse its buffer)."""
import numpy as np
import pytest

import oracle_py as O

pytestmark = pytest.mark.gpu

KGL_B200_ERR_STATE = 2


def test_close_frees_device_memory():
    """A process that opens a context per analysis must not lose device memory each time: IBS and KING on the tensor cores
    (their Gram blocks) and the iterative estimators (the moment tables) allocate the most."""
    import torch
    from kgl_gene_b200.capi import KglB200
    from kgl_gene_b200.synth import make_population

    pop, _ = make_population(2048, 20000, seed=11, missing_rate=0.002)      # indexed code-3 cells: the tensor-core IBS form
    free = []
    for _ in range(4):
        gpu = KglB200(0)
        gpu.upload_population(pop)
        gpu.ibs()
        assert gpu.ibs_used_tensor_cores()
        gpu.king()
        gpu.select_loci(spacing=0)
        gpu.inbreed("HallME", hall_sweeps=20)
        assert gpu.used_moment_tables() > 0
        gpu.inbreed("Loglikelihood")
        gpu.close()
        torch.cuda.synchronize()
        free.append(torch.cuda.mem_get_info()[0])
    drift = free[0] - free[3]
    assert drift < (4 << 20), f"{drift / 2**20:.1f} MiB of device memory lost over three create / close cycles"


def test_gram_not_readable_after_ibs():
    from kgl_gene_b200.capi import KglB200, KglError
    from kgl_gene_b200.synth import make_population

    pop, _ = make_population(300, 5000, seed=12, missing_rate=0.002)
    gpu = KglB200(0)
    try:
        gpu.upload_population(pop)
        gpu.enqueue_gram()
        gpu.ibs()
        assert gpu.ibs_used_tensor_cores()
        with pytest.raises(KglError, match=rf"\[{KGL_B200_ERR_STATE}\]: enqueue_gram first"):
            gpu.fetch_gram()
        gpu.enqueue_gram()
        assert np.array_equal(gpu.fetch_gram(), O.gram(pop)[0])
    finally:
        gpu.close()
