"""Launch limits of the persistent per-item kernels (ESS, beta) that outlive one sampler: they are prepared once per
(kernel, launch shape) and re-used by every later sampler in the process."""
import pytest

from conftest import make_problem

pytestmark = pytest.mark.gpu
ITEM_PERSISTENT = 1


def test_persistent_item_kernels_after_a_smaller_shape():
    """The dynamic shared-memory limit belongs to the kernel, not to a launch shape.  n = 4096 and n = 2304 run the same
    8-values-per-thread instantiation with 512 and 288 threads.  Preparing the smaller shape must not take the limit below
    what the larger one, prepared earlier, launches with."""
    import gpirt_b200.sampler as G
    from gpirt_b200 import _lib
    assert _lib.load().gpirt_b200_device_count() > 0, "no CUDA device"
    for n, m in ((4096, 160), (2304, 6), (4096, 160)):
        p = make_problem(n, m, seed=n + m, missing=0.0)
        s = G.Sampler(p["y"], p["theta"], p["pm"], p["psd"], p["pstep"], seed=3)
        s.init_draws()
        s.sweep(1)
        if m > 6:
            assert s.uses(2) == ITEM_PERSISTENT
        s.close()
