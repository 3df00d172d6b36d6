"""CPU-side checks of the progressive renders on every device (rt_multi_render_progressive / _denoised): argument errors
without a device, the bindings, and the cap schedule that every progressive call shares (rt_progressive_caps)."""
import ctypes as C

import numpy as np
import pytest

from mcp_raytracer_b200.scene_data import rt_denoise_opts, rt_region, rt_stats


def test_null_multi_is_an_invalid_argument():
    from mcp_raytracer_b200 import _native

    L = _native.lib()
    buf = np.zeros(12, np.uint8)
    reg = rt_region(0, 0, 2, 2)
    opts = rt_denoise_opts(5, 0, 0, 0)
    st = rt_stats()
    assert L.rt_multi_render_progressive(None, C.byref(reg), buf.ctypes.data, buf.nbytes, None, 4, None, None, C.byref(st)) == 1
    assert "null argument" in _native.last_error()
    assert L.rt_multi_render_progressive(None, None, None, 0, None, 1, None, None, None) == 1
    assert "null argument" in _native.last_error()
    assert L.rt_multi_render_progressive_denoised(None, C.byref(reg), buf.ctypes.data, buf.nbytes, None, None, 4, C.byref(opts),
                                                  None, None, C.byref(st)) == 1
    assert "null argument" in _native.last_error()
    assert L.rt_multi_render_progressive_denoised(None, None, None, 0, None, None, 1, None, None, None, None) == 1
    assert "null argument" in _native.last_error()


def test_multi_progressive_is_bound():
    from mcp_raytracer_b200 import MultiCamera, _native

    for name, n_args in (("rt_multi_render_progressive", 9), ("rt_multi_render_progressive_denoised", 11)):
        assert name in _native.EXPORTS
        assert len(getattr(_native.lib(), name).argtypes) == n_args
    assert callable(getattr(MultiCamera, "renderProgressive"))
    assert callable(getattr(MultiCamera, "renderProgressiveDenoised"))


def _parent_caps(S, batch, n_passes):
    """The loop of progressive_host before the schedule was shared: (pass, cap) of every pass that runs."""
    out, prev = [], 0
    for k in range(1, n_passes + 1):
        cap = (S * k + n_passes - 1) // n_passes
        cap = min(S, (cap + batch - 1) // batch * batch) if k < n_passes else S
        if cap <= prev and not (S <= 0 and k == n_passes):
            continue
        out.append((k, cap))
        prev = cap
    return out


def _caps(S, batch, n_passes):
    from mcp_raytracer_b200 import _native

    caps = np.full(n_passes, -7, np.int32)
    run = _native.lib().rt_progressive_caps(S, batch, n_passes, caps.ctypes.data)
    got = [(k + 1, int(c)) for k, c in enumerate(caps) if c >= 0]
    assert run == len(got) and np.all((caps >= 0) | (caps == -1))
    return got


@pytest.mark.parametrize("S,batch", [(40, 1), (50, 1), (7, 1), (1, 1), (0, 1), (100, 10), (64, 8), (30, 10), (5, 8), (0, 4),
                                     (2048, 64), (13, 3)])
def test_cap_schedule_is_progressive_hosts(S, batch):
    """Fixed spp (batch 1) and adaptive sampling (batch = aBatch), S = 0, more passes than samples."""
    for n_passes in (1, 2, 3, 4, 7, 8, S + 3, 3 * S + 1):
        got = _caps(S, batch, n_passes)
        assert got == _parent_caps(S, batch, n_passes), (S, batch, n_passes)
        assert got[-1][1] == S and len(got) <= max(1, min(n_passes, S))  # ends at S; passes with no new samples are skipped
        caps = [c for _, c in got]
        assert caps == sorted(set(caps))


def test_cap_schedule_examples_and_errors():
    from mcp_raytracer_b200 import _native

    assert _caps(40, 1, 8)[:3] == [(1, 5), (2, 10), (3, 15)]
    assert _caps(32, 1, 4) == [(1, 8), (2, 16), (3, 24), (4, 32)]
    assert _caps(3, 1, 6) == [(1, 1), (3, 2), (5, 3)]
    assert _caps(0, 1, 5) == [(5, 0)]
    assert _caps(30, 10, 4) == [(1, 10), (2, 20), (3, 30)]
    buf = np.zeros(4, np.int32)
    L = _native.lib()
    for args in ((-1, 1, 4), (8, 0, 4), (8, 1, 0)):
        assert L.rt_progressive_caps(*args, buf.ctypes.data) == -1
    assert L.rt_progressive_caps(8, 1, 4, None) == -1
