"""CPU-side checks of the denoiser on every device (rt_multi_render_denoised): argument errors without a device, the
binding, and the ghost-zone arithmetic the band windows use."""
import ctypes as C

import numpy as np

from mcp_raytracer_b200.scene_data import rt_denoise_opts, rt_region, rt_stats


def test_null_multi_is_an_invalid_argument():
    from mcp_raytracer_b200 import _native

    L = _native.lib()
    buf = np.zeros(12, np.uint8)
    reg = rt_region(0, 0, 2, 2)
    opts = rt_denoise_opts(5, 0, 0, 0)
    st = rt_stats()
    assert L.rt_multi_render_denoised(None, C.byref(reg), buf.ctypes.data, buf.nbytes, None, C.byref(opts), C.byref(st)) == 1
    assert L.rt_multi_render_denoised(None, None, None, 0, None, None, None) == 1
    assert "null argument" in _native.last_error()


def test_multi_denoised_is_bound():
    from mcp_raytracer_b200 import MultiCamera, _native

    assert "rt_multi_render_denoised" in _native.EXPORTS
    assert callable(getattr(MultiCamera, "renderDenoised"))


def _reach(K):
    """Rows above and below a row of the last pass's output that the filter's inputs are read from, stage by stage:
    pass k reads 2^(k+1) rows away (taps at +-2 * 2^k, variance blur +-1); prepare's depth gradient reads +-1."""
    r, out = 0, []
    for k in reversed(range(K)):
        r += 2 << k
        out.append(r)
    return out[::-1], r + 1


def test_ghost_zones_cover_what_each_stage_reads():
    """h_k = 2^(K+1) - 2^(k+2) rows beyond the band for pass k, 2^(K+1) - 2 for prepare, one more for the features
    (dn_halo in rt_types.h): each stage computes exactly the rows the later stages read, no more."""
    for K in range(9):
        h = [(1 << (K + 1)) - (1 << (k + 2)) for k in range(K)]
        prepare = (1 << (K + 1)) - 2
        reach, features = _reach(K)
        # pass k's outputs are read by the passes after it: the rows the last pass reads through passes k+1..K-1
        for k in range(K):
            assert h[k] == (reach[k + 1] if k + 1 < K else 0)
        assert prepare == (reach[0] if K else 0)
        assert features == prepare + 1
    assert (1 << 6) - 2 == 62 and (1 << 9) - 2 == 510  # prepare's halo at the default K = 5 and at K = 8
