"""GPU parity at BASELINE.json's full frame sizes (few frames each, so the CPU side finishes in seconds):
the CUDA filters against the reference itself, bit for bit, plus size-independent properties."""
import numpy as np
import pytest

from handbrake_b200 import synth
from reference_runs import differing_frames
from test_oracle import decomb_inputs

pytestmark = pytest.mark.gpu
FMT = {8: synth.PIX_FMT_YUV420P, 10: synth.PIX_FMT_YUV420P10}


def same(r, g):
    assert g.frames.shape == r.frames.shape
    if not np.array_equal(g.frames, r.frames):
        raise AssertionError(f"frames {differing_frames(g.frames, r.frames)[:8]} differ")
    assert np.array_equal(g.start, r.start) and list(g.combed) == list(r.combed)


def test_config2_1080p_nlmeans_medium(ref, cuda_filters):
    w, h = 1920, 1080
    clip = synth.progressive_clip(FMT[8], w, h, 5)
    same(ref.run("hb_filter_nlmeans", "y-strength=6:threads=5", clip, FMT[8], w, h),
         cuda_filters.run("hb_filter_nlmeans_cuda", "y-strength=6", clip, FMT[8], w, h))


def test_config4_4k_nlmeans_strong(ref, cuda_filters):
    w, h = 3840, 2160
    clip = synth.progressive_clip(FMT[8], w, h, 4)
    r = ref.run("hb_filter_nlmeans", "y-strength=10:threads=4", clip, FMT[8], w, h)
    g = cuda_filters.run("hb_filter_nlmeans_cuda", "y-strength=10", clip, FMT[8], w, h)
    same(r, g)
    # property: denoising shrinks the frame-to-frame noise energy but keeps the mean level
    yb = w * h
    assert abs(float(g.frames[:, :yb].mean()) - float(clip[:, :yb].mean())) < 2.0
    assert np.var(g.frames[0, :yb].astype(np.float32) - g.frames[1, :yb]) < np.var(clip[0, :yb].astype(np.float32) - clip[1, :yb])


def test_4k_10bit_nlmeans_medium(ref, cuda_filters):
    w, h = 3840, 2160
    clip = synth.progressive_clip(FMT[10], w, h, 3)
    same(ref.run("hb_filter_nlmeans", "y-strength=6:threads=3", clip, FMT[10], w, h),
         cuda_filters.run("hb_filter_nlmeans_cuda", "y-strength=6", clip, FMT[10], w, h))


def test_4k_nlmeans_large_window(ref, cuda_filters):
    """'strong + animation tune': patch 5, range 7, 4 frames (the large search window of BASELINE config 4)"""
    w, h = 3840, 2160
    clip = synth.progressive_clip(FMT[8], w, h, 5)[:, :]
    s = "y-strength=10:y-origin-tune=0.15:y-patch-size=5:y-range=7:y-frame-count=4"
    r = ref.run("hb_filter_nlmeans", s + ":threads=5", clip[:3], FMT[8], w, h)
    g = cuda_filters.run("hb_filter_nlmeans_cuda", s, clip[:3], FMT[8], w, h)
    same(r, g)


def test_config3_4k_10bit_comb_detect_decomb_eedi2bob(ref, cuda_filters):
    w, h = 3840, 2160
    clip, flags, _ = decomb_inputs(10, w, h, 2, seed=21)          # 2 interlaced + 3 progressive-noise frames
    s = ["mode=3:spatial-metric=2:motion-thresh=1:spatial-thresh=1:filter-mode=2:block-thresh=40:block-width=16:block-height=16",
         "mode=63"]                                                # eedi2bob (31) + selective (32), as work.c sets it
    r = ref.run(["hb_filter_comb_detect", "hb_filter_decomb"], s, clip, FMT[10], w, h, flags=flags)
    g = cuda_filters.run(["hb_filter_comb_detect_cuda", "hb_filter_decomb_cuda"], s, clip, FMT[10], w, h, flags=flags)
    same(r, g)
    assert g.vrate == (60000, 1001)
    # property of any deinterlacer here: the lines of the kept field are the input's lines
    dims = synth.plane_dims(w, h)
    n_bobbed = 0
    out_i = 0
    for t in range(clip.shape[0]):
        if r.combed[out_i] == 0:
            out_i += 1
            continue
        src_y = synth.split_planes(clip[t], FMT[10], w, h)[0]
        tff = 1 if (flags[t] & synth.PIC_FLAG_PROGRESSIVE_FRAME) else int(bool(flags[t] & synth.PIC_FLAG_TOP_FIELD_FIRST))
        for field in range(2):
            parity = field ^ tff ^ 1
            out_y = synth.split_planes(g.frames[out_i], FMT[10], w, h)[0]
            kept = slice(1, None, 2) if parity else slice(0, None, 2)    # parity 1 rebuilds even rows -> odd rows kept
            assert np.array_equal(out_y[kept], src_y[kept])
            out_i += 1
            n_bobbed += 1
    assert n_bobbed >= 2


def test_4k_lapsharp(ref, cuda_filters):
    w, h = 3840, 2160
    clip = synth.progressive_clip(FMT[10], w, h, 3, noise=20)
    same(ref.run("hb_filter_lapsharp", "y-strength=0.2:y-kernel=isolap", clip, FMT[10], w, h),
         cuda_filters.run("hb_filter_lapsharp_cuda", "y-strength=0.2:y-kernel=isolap", clip, FMT[10], w, h))


def test_config5_8k_10bit_chain(ref, cuda_filters):
    """BASELINE config 5: 7680x4320 yuv420p10, decomb -> NLMeans medium -> lapsharp, in libhb's enforced filter
    order (hb.c:1701-1720).  A 99.5 MB frame is above the buffer pool's largest size class (fifo.c:111-112)."""
    w, h = 7680, 4320
    clip, flags, _ = decomb_inputs(10, w, h, 1, seed=5)
    clip, flags = clip[:3], flags[:3]
    names_r = ["hb_filter_decomb", "hb_filter_nlmeans", "hb_filter_lapsharp_mt"]
    names_g = ["hb_filter_decomb_cuda", "hb_filter_nlmeans_cuda", "hb_filter_lapsharp_cuda"]
    s = ["mode=7", "y-strength=6", "y-strength=0.2:y-kernel=isolap"]
    r = ref.run(names_r, [s[0], s[1] + ":threads=3", s[2]], clip, FMT[10], w, h, flags=flags)
    g = cuda_filters.run(names_g, s, clip, FMT[10], w, h, flags=flags)
    same(r, g)
    assert g.frames.shape[0] == 3
