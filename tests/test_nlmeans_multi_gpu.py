"""GPU parity of multi-device dealing: hb_filter_nlmeans_cuda with `devices=...` vs its own single-device run and vs the
reference (bit-exact).  `devices=0,0` deals the ordered stream to TWO handles on one GPU -- every piece of the path
(owners, per-device index spaces, halo by device-to-device copy, event ordering between the handles, in-order harvest)
runs on a 1-GPU box; `devices=0,1` runs when a second GPU is visible (gpurun --gpus 2; NVLink peer copy).
VERDICT r1 item 4; the reference's frame-parallel dealing is mt_frame_filter.c:169-237."""
import ctypes as C

import numpy as np
import pytest

import handbrake_b200
from handbrake_b200 import synth
from reference_runs import differing_frames

pytestmark = pytest.mark.gpu

FMT8, FMT10 = synth.PIX_FMT_YUV420P, synth.PIX_FMT_YUV420P10


def device_count():
    return C.CDLL(str(handbrake_b200.LIBHBCU)).hbcu_device_count()


def same(a, b):
    assert a.saw_eof and b.saw_eof and not a.init_failed and not b.init_failed
    assert a.frames.shape == b.frames.shape
    assert np.array_equal(a.start, b.start) and np.array_equal(a.stop, b.stop)
    if not np.array_equal(a.frames, b.frames):
        raise AssertionError(f"frames {differing_frames(a.frames, b.frames)[:8]} differ")


CASES = [
    ("y-strength=3", "devices=0,0:block=4", 640, 360, 10, FMT8),                                   # BASELINE config 1
    ("y-strength=10", "devices=0,0,0:block=2", 640, 360, 10, FMT8),
    ("y-strength=6:y-patch-size=5:y-range=5:y-frame-count=4", "devices=0,0:block=3", 333, 211, 11, FMT8),
    ("y-strength=6:y-frame-count=3", "devices=0,0:block=1", 320, 192, 7, FMT10),                   # block raised to 2
    ("y-strength=6:y-prefilter=1:y-frame-count=2", "devices=0,0:block=2", 200, 120, 7, FMT8),      # start-of-stream rule
    ("y-strength=6:y-frame-count=3", "devices=0,0,0,0:block=2", 128, 96, 3, FMT8),                 # shorter than one round
]


@pytest.mark.parametrize("settings,multi,w,h,n,fmt", CASES)
def test_two_handles_on_one_gpu_equal_one_handle_and_reference(ref, cuda_filters, settings, multi, w, h, n, fmt):
    clip = synth.progressive_clip(fmt, w, h, n, seed=31)
    one = cuda_filters.run("hb_filter_nlmeans_cuda", settings, clip, fmt, w, h)
    many = cuda_filters.run("hb_filter_nlmeans_cuda", settings + ":" + multi, clip, fmt, w, h)
    # the prefilter modes follow the reference's single-worker behaviour (DESIGN.md 4.1)
    r = ref.run("hb_filter_nlmeans", settings + (":threads=1" if "prefilter" in settings else ":threads=2"), clip, fmt, w, h)
    same(r, one)
    same(r, many)
    same(one, many)
    assert cuda_filters.buffers_alive() == 0


def test_long_stream_many_blocks(cuda_filters):
    """enough frames to go round every ring several times with all queues full"""
    w, h, n = 256, 144, 70
    clip = synth.progressive_clip(FMT8, w, h, n, seed=3)
    s = "y-strength=6:y-patch-size=3:y-frame-count=3"
    one = cuda_filters.run("hb_filter_nlmeans_cuda", s, clip, FMT8, w, h)
    many = cuda_filters.run("hb_filter_nlmeans_cuda", s + ":devices=0,0,0:block=4:threads=2", clip, FMT8, w, h)
    same(one, many)


@pytest.mark.parametrize("settings,block", [("y-strength=3", 8), ("y-strength=6:y-frame-count=4:y-patch-size=5", 3),
                                            ("y-strength=6:y-prefilter=1", 2)])
def test_two_gpus_equal_one(ref, cuda_filters, settings, block):
    """config 1 over two real devices == one device == the reference (the halo crosses NVLink)"""
    if device_count() < 2:
        pytest.skip("needs two GPUs (gpurun --gpus 2)")
    w, h, n = 640, 360, 21
    clip = synth.progressive_clip(FMT8, w, h, n, seed=12)
    one = cuda_filters.run("hb_filter_nlmeans_cuda", settings, clip, FMT8, w, h)
    two = cuda_filters.run("hb_filter_nlmeans_cuda", settings + f":devices=0,1:block={block}", clip, FMT8, w, h)
    same(one, two)
    r = ref.run("hb_filter_nlmeans", settings + (":threads=1" if "prefilter" in settings else ":threads=2"), clip[:10], FMT8, w, h)
    assert np.array_equal(r.frames[:6], two.frames[:6])        # frames whose look-ahead window (<= 4 frames) lies inside the first 10
    if device_count() >= 4:
        four = cuda_filters.run("hb_filter_nlmeans_cuda", settings + f":devices=0,1,2,3:block={block}", clip, FMT8, w, h)
        same(one, four)


def test_frame_parallel_filters_over_devices(ref, cuda_filters):
    """lapsharp / unsharp / chroma smooth with `devices=`: round-robin over handles (two on one GPU; two GPUs when visible)"""
    w, h, n = 640, 360, 19
    clip = synth.progressive_clip(FMT8, w, h, n, seed=7)
    lists = ["0,0", "0,0,0"] + (["0,1"] if device_count() >= 2 else []) + (["0,1,2,3"] if device_count() >= 4 else [])
    for ref_name, name, settings in (("hb_filter_lapsharp_mt", "hb_filter_lapsharp_cuda", "y-strength=0.3:y-kernel=isolap"),
                                     ("hb_filter_unsharp_mt", "hb_filter_unsharp_cuda", "y-strength=0.5:y-size=5"),
                                     ("hb_filter_chroma_smooth_mt", "hb_filter_chroma_smooth_cuda", "cb-strength=0.8:cb-size=5")):
        r = ref.run(ref_name, settings, clip, FMT8, w, h)
        for devs in lists:
            same(r, cuda_filters.run(name, settings + ":devices=" + devs, clip, FMT8, w, h))
    assert cuda_filters.buffers_alive() == 0


def test_decomb_over_devices(ref, cuda_filters):
    """decomb without EEDI2 dealt over two handles of one GPU (and two GPUs when visible) == the reference"""
    from test_oracle import decomb_inputs
    w, h = 352, 288
    clip, flags, combed = decomb_inputs(8, w, h, 13, seed=6)
    lists = [("0,0", 3), ("0,0,0", 1)] + ([("0,1", 4)] if device_count() >= 2 else [])
    for mode, tags in ((7, None), (39, combed), (23, None)):
        r = ref.run("hb_filter_decomb", f"mode={mode}", clip, FMT8, w, h, flags=flags, combed=tags)
        for devs, block in lists:
            g = cuda_filters.run("hb_filter_decomb_cuda", f"mode={mode}:devices={devs}:block={block}", clip, FMT8, w, h, flags=flags, combed=tags)
            same(r, g)
    assert cuda_filters.buffers_alive() == 0
