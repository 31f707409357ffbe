"""GPU parity: hb_filter_unsharp_cuda / hb_filter_chroma_smooth_cuda vs the reference's hb_filter_unsharp /
hb_filter_chroma_smooth wrapped in mt_frame (SURVEY.md 8 f2), bit-exact."""
import numpy as np
import pytest

from handbrake_b200 import synth
from reference_runs import differing_frames
from test_oracle import UNSHARP_CASES, CHROMA_SMOOTH_CASES

pytestmark = pytest.mark.gpu

FMT = {8: synth.PIX_FMT_YUV420P, 10: synth.PIX_FMT_YUV420P10}
UP, DOWN = "hb_filter_hbcu_upload", "hb_filter_hbcu_download"


def same(r, g):
    assert g.saw_eof and r.saw_eof
    assert g.frames.shape == r.frames.shape
    assert np.array_equal(g.start, r.start)
    if not np.array_equal(g.frames, r.frames):
        raise AssertionError(f"frames {differing_frames(g.frames, r.frames)[:8]} differ")


@pytest.mark.parametrize("settings", [c[0] for c in UNSHARP_CASES])
@pytest.mark.parametrize("depth,w,h", [(8, 333, 211), (10, 330, 210)])
def test_unsharp(ref, cuda_filters, settings, depth, w, h):
    """ragged sizes (tiles end inside the picture, odd chroma), sizes 3..15 incl. the uint32 wrap at size 15"""
    clip = synth.progressive_clip(FMT[depth], w, h, 9, seed=61)
    same(ref.run("hb_filter_unsharp_mt", settings, clip, FMT[depth], w, h),
         cuda_filters.run("hb_filter_unsharp_cuda", settings, clip, FMT[depth], w, h))
    assert cuda_filters.buffers_alive() == 0


@pytest.mark.parametrize("settings", [c[0] for c in CHROMA_SMOOTH_CASES])
@pytest.mark.parametrize("depth,w,h", [(8, 333, 211), (10, 330, 210)])
def test_chroma_smooth(ref, cuda_filters, settings, depth, w, h):
    clip = synth.progressive_clip(FMT[depth], w, h, 9, seed=63)
    r = ref.run("hb_filter_chroma_smooth_mt", settings, clip, FMT[depth], w, h)
    g = cuda_filters.run("hb_filter_chroma_smooth_cuda", settings, clip, FMT[depth], w, h)
    same(r, g)
    yb = w * h * (2 if depth > 8 else 1)
    assert np.array_equal(g.frames[:, :yb], clip[:, :yb])            # luma passes through


def test_extreme_content(ref, cuda_filters):
    """flat 0 / flat max / full-range noise: the clamp bounds and the wrap-around sums"""
    w, h = 192, 112
    for depth in (8, 10):
        n = synth.frame_bytes(FMT[depth], w, h) // (2 if depth > 8 else 1)
        mx = (1 << depth) - 1
        dt = np.uint16 if depth > 8 else np.uint8
        rng = np.random.default_rng(7)
        clip = np.stack([np.zeros(n, dt), np.full(n, mx, dt), rng.integers(0, mx + 1, n).astype(dt),
                         (rng.integers(0, 2, n) * mx).astype(dt)]).view(np.uint8).reshape(4, -1)
        for name, s in (("unsharp", "y-strength=1.5:y-size=15"), ("unsharp", "y-strength=1.5:y-size=3"),
                        ("chroma_smooth", "cb-strength=3:cb-size=15"), ("chroma_smooth", "cb-strength=3:cb-size=3")):
            same(ref.run(f"hb_filter_{name}_mt", s, clip, FMT[depth], w, h),
                 cuda_filters.run(f"hb_filter_{name}_cuda", s, clip, FMT[depth], w, h))


def test_1080p_and_device_chain(ref, cuda_filters):
    """full HD through the filters alone and inside a device-resident chain with lapsharp behind them"""
    w, h = 1920, 1080
    clip = synth.progressive_clip(FMT[8], w, h, 4, seed=65)
    su, sc, sl = "y-strength=0.5:y-size=7", "cb-strength=1.2:cb-size=7", "y-strength=0.2:y-kernel=isolap"
    r = ref.run(["hb_filter_chroma_smooth_mt", "hb_filter_unsharp_mt", "hb_filter_lapsharp_mt"], [sc, su, sl], clip, FMT[8], w, h)
    g = cuda_filters.run(["hb_filter_chroma_smooth_cuda", "hb_filter_unsharp_cuda", "hb_filter_lapsharp_cuda"], [sc, su, sl], clip, FMT[8], w, h)
    same(r, g)
    d = cuda_filters.run([UP, "hb_filter_chroma_smooth_cuda", "hb_filter_unsharp_cuda", "hb_filter_lapsharp_cuda", DOWN],
                         [None, sc, su, sl, None], clip, FMT[8], w, h)
    same(r, d)
    assert cuda_filters.buffers_alive() == 0
