"""GPU parity: hb_filter_denoise_cuda (hqdn3d) vs the reference's hb_filter_denoise (SURVEY.md 8 f4), bit-exact."""
import numpy as np
import pytest

from handbrake_b200 import synth
from reference_runs import differing_frames
from test_oracle import HQDN3D_CASES

pytestmark = pytest.mark.gpu

FMT = {8: synth.PIX_FMT_YUV420P, 10: synth.PIX_FMT_YUV420P10, 12: synth.PIX_FMT_YUV420P12}
UP, DOWN = "hb_filter_hbcu_upload", "hb_filter_hbcu_download"


def same(r, g):
    assert g.saw_eof and r.saw_eof
    assert g.frames.shape == r.frames.shape
    assert np.array_equal(g.start, r.start)
    if not np.array_equal(g.frames, r.frames):
        raise AssertionError(f"frames {differing_frames(g.frames, r.frames)[:8]} differ")


@pytest.mark.parametrize("settings", [c[0] for c in HQDN3D_CASES])
@pytest.mark.parametrize("depth,w,h", [(8, 333, 211), (10, 330, 210),
                                       # widths the warp-specialised kernels take (multiples of 8; 328: luma only, chroma 164 stays on
                                       # the round-1 kernels), heights that end inside a 32-row tile, more than one 128-column tile
                                       (8, 328, 211), (10, 400, 130), (12, 272, 75)])
def test_hqdn3d(ref, cuda_filters, settings, depth, w, h):
    """ragged sizes (rows and columns that do not fill the 32-sample tiles), a dozen frames of temporal state,
    temporal-only planes, the default chain of strengths"""
    clip = synth.progressive_clip(FMT[depth], w, h, 12, seed=93)
    same(ref.run("hb_filter_denoise", settings, clip, FMT[depth], w, h),
         cuda_filters.run("hb_filter_denoise_cuda", settings, clip, FMT[depth], w, h))
    assert cuda_filters.buffers_alive() == 0


def test_extreme_content(ref, cuda_filters):
    w, h = 192, 112
    for depth in (8, 10):
        n = synth.frame_bytes(FMT[depth], w, h) // (2 if depth > 8 else 1)
        mx = (1 << depth) - 1
        dt = np.uint16 if depth > 8 else np.uint8
        rng = np.random.default_rng(11)
        clip = np.stack([np.zeros(n, dt), np.full(n, mx, dt), rng.integers(0, mx + 1, n).astype(dt),
                         (rng.integers(0, 2, n) * mx).astype(dt), np.zeros(n, dt)]).view(np.uint8).reshape(5, -1)
        for s in (None, "y-spatial=12:y-temporal=15", "y-spatial=0.5:y-temporal=0.5"):
            same(ref.run("hb_filter_denoise", s, clip, FMT[depth], w, h),
                 cuda_filters.run("hb_filter_denoise_cuda", s, clip, FMT[depth], w, h))


def test_1080p_and_device_chain(ref, cuda_filters):
    w, h = 1920, 1080
    clip = synth.progressive_clip(FMT[8], w, h, 6, seed=95)
    sd, sl = "y-spatial=3:cb-spatial=2:y-temporal=4", "y-strength=0.2:y-kernel=isolap"
    r = ref.run(["hb_filter_denoise", "hb_filter_lapsharp_mt"], [sd, sl], clip, FMT[8], w, h)
    same(r, cuda_filters.run(["hb_filter_denoise_cuda", "hb_filter_lapsharp_cuda"], [sd, sl], clip, FMT[8], w, h))
    same(r, cuda_filters.run([UP, "hb_filter_denoise_cuda", "hb_filter_lapsharp_cuda", DOWN], [None, sd, sl, None], clip, FMT[8], w, h))
    assert cuda_filters.buffers_alive() == 0


def test_round1_kernels_still_agree(ref, cuda_filters, monkeypatch):
    """HBCU_HQDN3D_V1=1 forces the one-warp-does-everything kernels (still used for odd widths and 16-bit depth)"""
    monkeypatch.setenv("HBCU_HQDN3D_V1", "1")
    w, h = 384, 130
    for depth in (8, 10):
        clip = synth.progressive_clip(FMT[depth], w, h, 6, seed=97)
        same(ref.run("hb_filter_denoise", HQDN3D_CASES[0][0], clip, FMT[depth], w, h),
             cuda_filters.run("hb_filter_denoise_cuda", HQDN3D_CASES[0][0], clip, FMT[depth], w, h))
