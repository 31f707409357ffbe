"""GPU parity: hb_filter_decomb_cuda vs the reference's hb_filter_decomb (bit-exact pictures, timestamps, counts)."""
import numpy as np
import pytest

from handbrake_b200 import synth
from reference_runs import differing_frames
from test_oracle import DECOMB_CASES, decomb_inputs

pytestmark = pytest.mark.gpu
FMT = {8: synth.PIX_FMT_YUV420P, 10: synth.PIX_FMT_YUV420P10}


def compare(ref, cuda, s, clip, fmt, w, h, flags, combed):
    r = ref.run("hb_filter_decomb", s, clip, fmt, w, h, flags=flags, combed=combed)
    g = cuda.run("hb_filter_decomb_cuda", s, clip, fmt, w, h, flags=flags, combed=combed)
    assert not g.init_failed and g.saw_eof
    assert g.frames.shape == r.frames.shape, (g.frames.shape, r.frames.shape)
    assert np.array_equal(g.start, r.start) and np.array_equal(g.stop, r.stop)
    assert np.array_equal(g.flags, r.flags) and np.array_equal(g.combed, r.combed)
    assert g.vrate == r.vrate
    if not np.array_equal(g.frames, r.frames):
        raise AssertionError(f"{s}: frames {differing_frames(g.frames, r.frames)[:8]} differ")


@pytest.mark.parametrize("mode,parity,tags", DECOMB_CASES)
@pytest.mark.parametrize("depth", [8, 10])
def test_line_filters_match_reference(ref, cuda_filters, mode, parity, tags, depth):
    w, h = 200, 106          # ragged width (not a multiple of 4*64), odd chroma height
    clip, flags, combed = decomb_inputs(depth, w, h, 7)
    compare(ref, cuda_filters, f"mode={mode}:parity={parity}", clip, FMT[depth], w, h, flags, combed if tags else None)
    assert cuda_filters.buffers_alive() == 0


def test_comb_detect_then_decomb_chain(ref, cuda_filters):
    """the pipeline libhb builds: comb_detect tags frames, decomb (selective) acts on the tags"""
    w, h = 320, 180
    clip, flags, _ = decomb_inputs(8, w, h, 10, seed=9)
    s = [None, "mode=39"]
    r = ref.run(["hb_filter_comb_detect", "hb_filter_decomb"], s, clip, FMT[8], w, h, flags=flags)
    g = cuda_filters.run(["hb_filter_comb_detect_cuda", "hb_filter_decomb_cuda"], s, clip, FMT[8], w, h, flags=flags)
    assert g.frames.shape == r.frames.shape and np.array_equal(g.frames, r.frames)
    assert list(g.combed) == list(r.combed) and len(set(r.combed)) > 1


def test_short_clips(ref, cuda_filters):
    w, h = 96, 64
    for n in (1, 2):
        clip, flags, combed = decomb_inputs(8, w, h, n)
        clip, flags = clip[:n], flags[:n]
        compare(ref, cuda_filters, "mode=23", clip, FMT[8], w, h, flags, None)


# ---------------------------------------------------------------- EEDI2
EEDI2_CASES = [
    (8, False), (24, False), (9, False), (25, False), (31, False), (31 | 32, True), (15, True), (10, True),
]


@pytest.mark.parametrize("mode,tags", EEDI2_CASES)
@pytest.mark.parametrize("depth", [8, 10])
def test_eedi2_matches_reference(ref, cuda_filters, mode, tags, depth):
    """EEDI2 alone, bobbed, feeding yadif; incl. the edge-mask state carried from field to field"""
    w, h = 208, 120          # stride 256 > width: the linear-address reads of EEDI2 see the stride padding
    clip, flags, combed = decomb_inputs(depth, w, h, 6, seed=11)
    compare(ref, cuda_filters, f"mode={mode}", clip, FMT[depth], w, h, flags, combed if tags else None)


def test_eedi2_stride_equals_width(ref, cuda_filters):
    """width a multiple of 64 (as at every BASELINE config): row ends wrap into the next row's pixels"""
    w, h = 256, 96
    clip, flags, combed = decomb_inputs(8, w, h, 5, seed=12)
    compare(ref, cuda_filters, "mode=31", clip, FMT[8], w, h, flags, None)
    compare(ref, cuda_filters, "mode=24:magnitude-thresh=6:variance-thresh=10:laplacian-thresh=12:noise-thresh=30:search-distance=16",
            clip, FMT[8], w, h, flags, None)


def test_eedi2_odd_plane_height_is_refused(cuda_filters):
    w, h = 208, 122          # chroma height 61 is odd: the reference copies a line from beyond the plane
    clip, flags, combed = decomb_inputs(8, w, h, 3)
    g = cuda_filters.run("hb_filter_decomb_cuda", "mode=24", clip, FMT[8], w, h, flags=flags)
    assert g.init_failed == 1


# ---------------------------------------------------------------- EEDI2 postproc 2/3 (corner filter, SURVEY.md 8a a28)
@pytest.mark.parametrize("pp", [2, 3, 0])
@pytest.mark.parametrize("mode", [24, 31])
@pytest.mark.parametrize("depth,w,h", [(8, 208, 120), (10, 208, 120), (8, 256, 128)])
def test_eedi2_postproc_matches_port(cuda_filters, pp, mode, depth, w, h):
    """The reference's corner filter shares scratch arrays between its plane threads (a race) and reads memory nothing
    wrote, so the pin is the C restatement (every stage checked against the reference's exported functions and the
    race-free part of its luma output, tests/test_oracle.py); 256x128 has pitch == width: the blur's one out-of-row
    read lands in the next row"""
    from oracle_port import OraclePort
    port = OraclePort()
    clip, flags, combed = decomb_inputs(depth, w, h, 5, seed=11)
    o, _ = port.decomb_clip(clip, w, h, depth, mode, -1, flags, None, postproc=pp)
    g = cuda_filters.run("hb_filter_decomb_cuda", f"mode={mode}:postproc={pp}", clip, FMT[depth], w, h, flags=flags)
    assert not g.init_failed and g.saw_eof and g.frames.shape == o.shape
    if not np.array_equal(g.frames, o):
        d = g.frames != o
        raise AssertionError(f"postproc={pp}: {np.count_nonzero(d)} bytes differ in frames {np.argwhere(d.any(axis=1)).ravel()[:8]}")
    if pp == 3 or (pp == 2 and w == 256):         # the corner filter did change pictures (it rarely fires without postproc 1's map)
        base, _ = port.decomb_clip(clip, w, h, depth, mode, -1, flags, None, postproc=pp - 2)
        assert not np.array_equal(base, o)


def test_eedi2_postproc_small_planes_are_refused(cuda_filters):
    w, h = 96, 40            # chroma planes 48x20: the reference's spelled-out blur edges would overlap
    clip, flags, combed = decomb_inputs(8, w, h, 3)
    g = cuda_filters.run("hb_filter_decomb_cuda", "mode=24:postproc=2", clip, FMT[8], w, h, flags=flags)
    assert g.init_failed == 1
