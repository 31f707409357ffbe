"""GPU parity: hb_filter_nlmeans_cuda vs the reference's hb_filter_nlmeans (bit-exact)."""
import numpy as np
import pytest

from handbrake_b200 import synth
from reference_runs import differing_frames

pytestmark = pytest.mark.gpu

FMT8, FMT10 = synth.PIX_FMT_YUV420P, synth.PIX_FMT_YUV420P10


def run_both(ref, cuda, settings, clip, fmt, w, h, ref_threads=2):
    r = ref.run("hb_filter_nlmeans", settings + f":threads={ref_threads}", clip, fmt, w, h)
    g = cuda.run("hb_filter_nlmeans_cuda", settings, clip, fmt, w, h)
    return r, g


def assert_same(r, g):
    assert g.saw_eof and r.saw_eof
    assert g.frames.shape == r.frames.shape
    assert np.array_equal(g.start, r.start)
    if not np.array_equal(g.frames, r.frames):
        raise AssertionError(f"mismatch: frames {differing_frames(g.frames, r.frames)[:8]} differ")


@pytest.mark.parametrize("strength", [3, 6, 10])
def test_config1_640x360_presets(ref, cuda_filters, strength):
    """BASELINE config 1 (light) + medium/strong on the same clip: 10 frames, bit-exact."""
    w, h = 640, 360
    clip = synth.progressive_clip(FMT8, w, h, 10)
    r, g = run_both(ref, cuda_filters, f"y-strength={strength}", clip, FMT8, w, h)
    assert_same(r, g)
    assert cuda_filters.buffers_alive() == 0


def test_ragged_geometry_and_chroma_params(ref, cuda_filters):
    """width/height not multiples of the tile, odd chroma size, per-plane parameters"""
    w, h = 333, 211
    clip = synth.progressive_clip(FMT8, w, h, 6, seed=7)
    s = "y-strength=6:y-origin-tune=0.8:y-patch-size=7:y-range=3:y-frame-count=2:cb-strength=4:cb-patch-size=5:cb-range=5:cb-frame-count=3"
    r, g = run_both(ref, cuda_filters, s, clip, FMT8, w, h)
    assert_same(r, g)


def test_10bit(ref, cuda_filters):
    w, h = 320, 192
    clip = synth.progressive_clip(FMT10, w, h, 5)
    r, g = run_both(ref, cuda_filters, "y-strength=6", clip, FMT10, w, h)
    assert_same(r, g)


def test_generic_kernel_matches(ref, cuda_filters):
    """patch 11 does not fit the tiled kernel (n/2 <= 4): exercises the generic kernel"""
    w, h = 200, 120
    clip = synth.progressive_clip(FMT8, w, h, 4)
    r, g = run_both(ref, cuda_filters, "y-strength=6:y-patch-size=11:y-range=5", clip, FMT8, w, h)
    assert_same(r, g)


def test_strength_zero_bypass_and_single_frame(ref, cuda_filters):
    w, h = 160, 96
    clip = synth.progressive_clip(FMT8, w, h, 3)
    r, g = run_both(ref, cuda_filters, "y-strength=0:cb-strength=5:y-frame-count=1", clip, FMT8, w, h)
    assert_same(r, g)
    assert np.array_equal(g.frames[:, : w * h], clip[:, : w * h])   # luma untouched


def test_fewer_frames_than_window(ref, cuda_filters):
    """EOF before the look-ahead window ever fills: shrinking window only (nlmeans.c:636-640)"""
    w, h = 160, 96
    clip = synth.progressive_clip(FMT8, w, h, 2)
    r, g = run_both(ref, cuda_filters, "y-strength=6:y-frame-count=4", clip, FMT8, w, h)
    assert_same(r, g)


@pytest.mark.parametrize("mode", [1, 2, 4, 8, 16, 32, 1 + 256, 2 + 512, 4 + 256 + 512, 2049, 2048 + 8 + 512, 2048, 256, 1024,
                                  1 + 1024, 16 + 1024, 2 + 1024 + 256, 8 + 1024 + 2048 + 512])
@pytest.mark.parametrize("fmt", [FMT8, FMT10])
def test_prefilter_modes(ref, cuda_filters, mode, fmt):
    """mean / median / csm prefilters (3x3, 5x5), reduce 25/50/75, edgeboost (a raster-order recurrence, solved as a
    fixed-point iteration), passthru, the no-op modes; chroma inherits luma.
    The reference with threads=1: with more workers it races on frame[0].image_pre (SURVEY.md 8a a5, DESIGN.md)."""
    w, h = 200, 120
    clip = synth.progressive_clip(fmt, w, h, 4, seed=81)
    s = f"y-strength=6:y-patch-size=5:y-range=3:y-frame-count=2:cb-frame-count=1:y-prefilter={mode}"
    r = ref.run("hb_filter_nlmeans", s + ":threads=1", clip, fmt, w, h)
    g = cuda_filters.run("hb_filter_nlmeans_cuda", s, clip, fmt, w, h)
    assert_same(r, g)


@pytest.mark.parametrize("impl", ["1", "3"])
def test_other_kernels_agree(ref, cuda_filters, monkeypatch, impl):
    """generic (1) and integer-tiled (3) kernels on the same 8-bit clip the v3 kernel handles by default"""
    monkeypatch.setenv("HBCU_NLMEANS_IMPL", impl)
    w, h = 300, 150
    clip = synth.progressive_clip(FMT8, w, h, 4, seed=21)
    r, g = run_both(ref, cuda_filters, "y-strength=6:cb-strength=3:cb-range=5", clip, FMT8, w, h)
    assert_same(r, g)


def test_flat_and_extreme_content(ref, cuda_filters):
    """all-zero frames (result==0 -> source pixel fallback), saturated frames, and full-range noise"""
    w, h = 192, 112
    fb = synth.frame_bytes(FMT8, w, h)
    rng = np.random.default_rng(5)
    clip = np.stack([np.zeros(fb, np.uint8), np.full(fb, 255, np.uint8),
                     rng.integers(0, 256, fb, dtype=np.uint8), rng.integers(0, 256, fb, dtype=np.uint8),
                     np.zeros(fb, np.uint8)])
    for s in ("y-strength=3", "y-strength=10:y-origin-tune=0.15", "y-strength=1.5"):
        r, g = run_both(ref, cuda_filters, s, clip, FMT8, w, h)
        assert_same(r, g)


def test_golden_digests(cuda_filters):
    """the committed digests of the reference output (tests/golden), no reference needed at run time"""
    import hashlib, json
    from pathlib import Path
    golden = json.loads((Path(__file__).parent / "golden" / "nlmeans_golden.json").read_text())
    for name, c in golden.items():
        fmt = FMT8 if c["depth"] == 8 else FMT10
        clip = synth.progressive_clip(fmt, c["width"], c["height"], c["frames"], seed=c["seed"])
        g = cuda_filters.run("hb_filter_nlmeans_cuda", c["settings"], clip, fmt, c["width"], c["height"])
        assert [hashlib.sha256(f.tobytes()).hexdigest() for f in g.frames] == c["sha256"], name


@pytest.mark.parametrize("s", ["y-strength=6:y-patch-size=7:cb-strength=5:cb-patch-size=5:cb-range=5:cr-patch-size=3",
                               "y-strength=8:y-patch-size=9:y-range=5:y-frame-count=3"])
def test_patch_sizes_3_5_7_9(ref, cuda_filters, s):
    """patch sizes 3/5/7/9 over the three planes: per-plane launches where the patch sizes differ, the 8-warp shape of
    patch 9"""
    w, h = 300, 170
    clip = synth.progressive_clip(FMT8, w, h, 4, seed=23)
    r, g = run_both(ref, cuda_filters, s, clip, FMT8, w, h)
    assert_same(r, g)


@pytest.mark.parametrize("s", ["y-strength=6", "y-strength=10:y-patch-size=5:y-range=5:y-frame-count=3"])
@pytest.mark.parametrize("fmt", [FMT8, FMT10])
def test_ragged_clip_8_and_10bit(ref, cuda_filters, fmt, s):
    """a 330 x 210 clip (ragged against every tile shape) in 8 and 10 bit, default kernels"""
    w, h = 330, 210
    clip = synth.progressive_clip(fmt, w, h, 4, seed=33)
    r, g = run_both(ref, cuda_filters, s, clip, fmt, w, h)
    assert_same(r, g)


def clip10_extreme(w, h, seed=9):
    """full-range 10-bit noise, flat 0 and flat 1023 frames (worst case for the fp32-exact row sums: d = 1023 everywhere)"""
    n = synth.frame_bytes(FMT10, w, h) // 2
    rng = np.random.default_rng(seed)
    frames = [rng.integers(0, 1024, n, dtype=np.uint16), np.zeros(n, np.uint16), np.full(n, 1023, np.uint16),
              rng.integers(0, 2, n, dtype=np.uint16) * 1023, rng.integers(0, 1024, n, dtype=np.uint16)]
    return np.stack(frames).view(np.uint8).reshape(len(frames), -1)


@pytest.mark.parametrize("impl", ["0", "3", "1"])
def test_10bit_kernels_agree(ref, cuda_filters, monkeypatch, impl):
    """default 10-bit kernel (0), integer tiled kernel (3), generic kernel (1): patch 7/5/3, ranges 3/5/7, every alignment
    of the compare window (dx0 mod 4), 3-frame window, ragged size; the second setting gives luma and chroma different
    patch sizes, so by default each plane runs its own launch"""
    monkeypatch.setenv("HBCU_NLMEANS_IMPL", impl)
    w, h = 330, 210
    clip = synth.progressive_clip(FMT10, w, h, 4, seed=31)
    for s in ("y-strength=6", "y-strength=10:y-patch-size=5:y-range=7:y-frame-count=3:cb-strength=4:cb-patch-size=3:cb-range=5"):
        r, g = run_both(ref, cuda_filters, s, clip, FMT10, w, h)
        assert_same(r, g)


def test_10bit_extreme_content(ref, cuda_filters):
    w, h = 256, 128
    clip = clip10_extreme(w, h)
    for s in ("y-strength=3", "y-strength=10:y-origin-tune=0.15", "y-strength=1.5:y-patch-size=5"):
        r, g = run_both(ref, cuda_filters, s, clip, FMT10, w, h)
        assert_same(r, g)


def test_10bit_container_with_out_of_range_samples(ref, cuda_filters):
    """a yuv420p10 stream whose 16-bit words exceed 1023 from the third frame on: the border kernel raises the range
    flag, the v3 kernel stands down and the integer kernel produces the frames -- still the reference's output"""
    w, h = 256, 128
    clip = synth.progressive_clip(FMT10, w, h, 5, seed=33).copy()
    v = clip.view(np.uint16).reshape(5, -1)
    v[2, 1000:1040] = 4095
    v[3, ::97] = 3000
    r, g = run_both(ref, cuda_filters, "y-strength=6", clip, FMT10, w, h)
    assert_same(r, g)


def test_edgeboost_long_dependency_chain(ref, cuda_filters):
    """a diagonal line of isolated edge pairs: clearing the first one clears the next ... one Jacobi round per sample"""
    w, h = 96, 80
    n = synth.frame_bytes(FMT8, w, h)
    frame = np.full(n, 60, np.uint8)
    y = frame[: w * h].reshape(h, w)
    for i in range(2, 70, 2):                     # isolated bright dots on a diagonal
        y[i, i] = 220
    clip = np.stack([frame, frame.copy(), frame.copy()])
    clip[1, : w * h].reshape(h, w)[5:40:3, 50] = 200
    s = "y-strength=6:y-patch-size=5:y-frame-count=2:y-prefilter=1025:cb-prefilter=0"
    r = ref.run("hb_filter_nlmeans", s + ":threads=1", clip, FMT8, w, h)
    g = cuda_filters.run("hb_filter_nlmeans_cuda", s, clip, FMT8, w, h)
    assert_same(r, g)
