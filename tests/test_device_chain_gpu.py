"""GPU parity of device-resident filter chains (SURVEY.md 8 f3): between two CUDA filters the frame stays in HBM
(HBCU_DEVICE hb_buffer_t backing), hb_filter_hbcu_upload / hb_filter_hbcu_download are the two ends.  The output must be
the reference chain's output, bit for bit, and no device frame or hb_buffer_t may leak."""
import ctypes as C

import numpy as np
import pytest

from handbrake_b200 import LIBHBCU, synth
from reference_runs import differing_frames
from test_oracle import decomb_inputs

pytestmark = pytest.mark.gpu

FMT = {8: synth.PIX_FMT_YUV420P, 10: synth.PIX_FMT_YUV420P10}
UP, DOWN = "hb_filter_hbcu_upload", "hb_filter_hbcu_download"


def frames_alive():
    core = C.CDLL(str(LIBHBCU))
    core.hbcu_frames_alive.restype = C.c_long
    return core.hbcu_frames_alive()


def same(r, g):
    assert g.saw_eof and r.saw_eof
    assert g.frames.shape == r.frames.shape, (g.frames.shape, r.frames.shape)
    assert np.array_equal(g.start, r.start)
    if not np.array_equal(g.frames, r.frames):
        raise AssertionError(f"frames {differing_frames(g.frames, r.frames)[:8]} differ")


@pytest.mark.parametrize("depth,w,h", [(8, 333, 211), (10, 330, 210), (8, 640, 360)])
def test_nlmeans_between_adapters(ref, cuda_filters, depth, w, h):
    clip = synth.progressive_clip(FMT[depth], w, h, 7, seed=41)
    r = ref.run("hb_filter_nlmeans", "y-strength=6:threads=2", clip, FMT[depth], w, h)
    g = cuda_filters.run([UP, "hb_filter_nlmeans_cuda", DOWN], [None, "y-strength=6", None], clip, FMT[depth], w, h)
    same(r, g)
    assert frames_alive() == 0 and cuda_filters.buffers_alive() == 0


@pytest.mark.parametrize("depth", [8, 10])
def test_lapsharp_device_frames_with_padded_stride(ref, cuda_filters, depth):
    """width*bps not a multiple of 64: lapsharp reads the mirrored stride padding (lapsharp.c:333), which for a device
    frame is produced in HBM"""
    w, h = 300, 150
    clip = synth.progressive_clip(FMT[depth], w, h, 5, seed=43)
    for s in ("y-strength=0.2:y-kernel=isolap", "y-strength=0.5:y-kernel=log:cb-strength=0.3:cb-kernel=lap"):
        r = ref.run("hb_filter_lapsharp_mt", s, clip, FMT[depth], w, h)
        g = cuda_filters.run([UP, "hb_filter_lapsharp_cuda", DOWN], [None, s, None], clip, FMT[depth], w, h)
        same(r, g)
    assert frames_alive() == 0 and cuda_filters.buffers_alive() == 0


@pytest.mark.parametrize("depth", [8, 10])
def test_full_chain_device_resident(ref, cuda_filters, depth):
    """comb_detect -> decomb (selective: uncombed frames pass through as references to the same device frame) ->
    nlmeans -> lapsharp, one upload and one download per frame"""
    w, h = 256, 144
    clip, flags, _ = decomb_inputs(depth, w, h, 8, seed=3)
    names_r = ["hb_filter_comb_detect", "hb_filter_decomb", "hb_filter_nlmeans", "hb_filter_lapsharp_mt"]
    names_g = [UP, "hb_filter_comb_detect_cuda", "hb_filter_decomb_cuda", "hb_filter_nlmeans_cuda", "hb_filter_lapsharp_cuda", DOWN]
    s = [None, "mode=39", "y-strength=6", "y-strength=0.2:y-kernel=isolap"]
    r = ref.run(names_r, [s[0], s[1], s[2] + ":threads=2", s[3]], clip, FMT[depth], w, h, flags=flags)
    g = cuda_filters.run(names_g, [None] + s + [None], clip, FMT[depth], w, h, flags=flags)
    same(r, g)
    assert list(g.combed) == list(r.combed)
    assert frames_alive() == 0 and cuda_filters.buffers_alive() == 0


def test_eedi2_bob_device_resident(ref, cuda_filters):
    w, h = 320, 192
    clip, flags, _ = decomb_inputs(10, w, h, 5, seed=9)
    r = ref.run(["hb_filter_comb_detect", "hb_filter_decomb"], [None, "mode=63"], clip, FMT[10], w, h, flags=flags)
    g = cuda_filters.run([UP, "hb_filter_comb_detect_cuda", "hb_filter_decomb_cuda", DOWN], [None, None, "mode=63", None],
                         clip, FMT[10], w, h, flags=flags)
    same(r, g)
    assert g.vrate == r.vrate == (60000, 1001)
    assert frames_alive() == 0 and cuda_filters.buffers_alive() == 0


def test_mixed_host_and_device_segments(ref, cuda_filters):
    """device segment, back to host, a host-side CUDA filter behind it: every filter takes either kind of buffer"""
    w, h = 256, 144
    clip, flags, _ = decomb_inputs(8, w, h, 6, seed=13)
    r = ref.run(["hb_filter_decomb", "hb_filter_nlmeans"], ["mode=7", "y-strength=3:threads=2"], clip, FMT[8], w, h, flags=flags)
    g = cuda_filters.run([UP, "hb_filter_decomb_cuda", DOWN, "hb_filter_nlmeans_cuda"], [None, "mode=7", None, "y-strength=3"],
                         clip, FMT[8], w, h, flags=flags)
    same(r, g)
    assert frames_alive() == 0 and cuda_filters.buffers_alive() == 0


def test_chain_without_download_adapter_fails_loudly(cuda_filters):
    w, h = 160, 96
    clip = synth.progressive_clip(FMT[8], w, h, 3)
    with pytest.raises(RuntimeError):
        cuda_filters.run([UP, "hb_filter_lapsharp_cuda"], [None, "y-strength=0.2"], clip, FMT[8], w, h)
    assert frames_alive() == 0 and cuda_filters.buffers_alive() == 0
