"""CPU tests of the detelecine (pullup) drop-in, SURVEY.md 8 f4.

oracle/_ref/libhostlogic.so is the PRODUCT's host-side state machine (handbrake_b200/libhb/detelecine_cuda.c,
compiled untouched) with its device calls redirected to the plain-C restatement oracle/port/detelecine_port.c.  Pinned
here, frame for frame, against the stored runs of the reference's own hb_filter_detelecine (tests/reference_runs.py).  On
the GPU box the same host code drives the CUDA kernels and tests/test_detelecine_gpu.py compares that with the reference."""
import numpy as np
import pytest

from handbrake_b200 import synth
from conftest import ORACLE_DIR
from reference_runs import differing_frames

FMT = {8: synth.PIX_FMT_YUV420P, 10: synth.PIX_FMT_YUV420P10}
HOSTLOGIC_SO = ORACLE_DIR / "_ref" / "libhostlogic.so"      # see tests/test_hostlogic.py

# (telecined_clip keywords, settings)
DETELECINE_CASES = [
    (dict(), None),
    (dict(tff=False), None),
    (dict(soft=True), None),
    (dict(soft=True, tff=False, video_tail=5), None),
    (dict(video_tail=7), None),                                   # the cadence breaks into interlaced video
    (dict(noise=12), "strict-breaks=0"),
    (dict(noise=0), "strict-breaks=1"),
    (dict(tff=False), "parity=0"),                                # user says TFF, the pictures are BFF
    (dict(), "parity=1"),
    (dict(), "plane=1"),
    (dict(noise=6), "plane=2:skip-left=2:skip-right=3:skip-top=6:skip-bottom=5"),
    (dict(), "skip-left=0:skip-top=0:plane=7"),                    # clamped to the safety margins / plane 0
]


@pytest.fixture(scope="session")
def hostlogic():
    from handbrake_b200.hblib import FilterLib
    if not HOSTLOGIC_SO.exists():
        pytest.skip("oracle/_ref/libhostlogic.so not built")
    return FilterLib(HOSTLOGIC_SO)


def compare(r, g):
    assert not g.init_failed and g.saw_eof
    assert g.frames.shape == r.frames.shape, (g.frames.shape, r.frames.shape)
    assert np.array_equal(g.start, r.start) and np.array_equal(g.stop, r.stop) and np.array_equal(g.flags, r.flags)
    if not np.array_equal(g.frames, r.frames):
        raise AssertionError(f"frames {differing_frames(g.frames, r.frames)[:8]} differ")


@pytest.mark.parametrize("kw,settings", DETELECINE_CASES)
@pytest.mark.parametrize("depth,w,h", [(8, 160, 96), (10, 160, 96), (8, 200, 90)])
def test_detelecine_hostlogic_equals_reference(ref, hostlogic, kw, settings, depth, w, h):
    clip, flags = synth.telecined_clip(FMT[depth], w, h, 16, seed=71, **kw)
    r = ref.run("hb_filter_detelecine", settings, clip, FMT[depth], w, h, flags=flags)
    g = hostlogic.run("hb_filter_detelecine_cuda", settings, clip, FMT[depth], w, h, flags=flags)
    compare(r, g)
    assert hostlogic.buffers_alive() == 0


def test_detelecine_removes_the_pulldown(ref, hostlogic):
    """hard 2:3 pulldown of noiseless film: every output after the pass-through is one of the film frames again, each
    once, in order -- 4 out of 5 pictures survive"""
    w, h = 160, 96
    n_film = 24
    clip, flags = synth.telecined_clip(FMT[8], w, h, n_film, seed=3, noise=2)
    film = [synth.progressive_frame(FMT[8], w, h, 3 * t, 3, 2) for t in range(n_film)]
    g = hostlogic.run("hb_filter_detelecine_cuda", None, clip, FMT[8], w, h, flags=flags)
    assert clip.shape[0] == 30 and 22 <= g.frames.shape[0] <= 25
    which = []
    for f in g.frames[1:]:
        hits = [t for t in range(n_film) if np.array_equal(f, film[t])]
        assert len(hits) == 1
        which.append(hits[0])
    assert which == sorted(set(which))


def test_detelecine_static_and_repeated_pictures(ref, hostlogic):
    """identical pictures in a row (all metrics zero), then motion, then a picture repeated by RFF"""
    w, h = 160, 96
    a = synth.progressive_frame(FMT[8], w, h, 0, 5, 4)
    moving = synth.progressive_clip(FMT[8], w, h, 6, seed=5, noise=4, t0=4)
    clip = np.stack([a, a, a, a] + list(moving) + [a, a])
    flags = np.full(clip.shape[0], synth.PIC_FLAG_TOP_FIELD_FIRST, np.uint16)
    flags[6] |= synth.PIC_FLAG_REPEAT_FIRST_FIELD
    flags[7] = 0
    for settings in (None, "strict-breaks=1"):
        r = ref.run("hb_filter_detelecine", settings, clip, FMT[8], w, h, flags=flags)
        g = hostlogic.run("hb_filter_detelecine_cuda", settings, clip, FMT[8], w, h, flags=flags)
        compare(r, g)


def test_detelecine_long_clip_every_picture_flagged_rff(ref, hostlogic):
    """three fields submitted per picture for a whole clip"""
    w, h = 96, 64
    clip = synth.progressive_clip(FMT[8], w, h, 40, seed=9, noise=5)
    flags = np.full(40, synth.PIC_FLAG_TOP_FIELD_FIRST | synth.PIC_FLAG_REPEAT_FIRST_FIELD, np.uint16)
    flags[1::2] = synth.PIC_FLAG_REPEAT_FIRST_FIELD                   # alternate field order so no field is dropped
    r = ref.run("hb_filter_detelecine", None, clip, FMT[8], w, h, flags=flags)
    g = hostlogic.run("hb_filter_detelecine_cuda", None, clip, FMT[8], w, h, flags=flags)
    compare(r, g)


def test_detelecine_too_small_for_metric_blocks_is_refused(hostlogic):
    w, h = 32, 24                 # (24 - 16) >> 3 = 1 block row, (32 - 16) >> 3 = 2: fine; 16 lines leave none
    clip = synth.progressive_clip(FMT[8], 32, 16, 3)
    g = hostlogic.run("hb_filter_detelecine_cuda", None, clip, FMT[8], 32, 16)
    assert g.init_failed == 1


@pytest.mark.parametrize("seed", range(48))
def test_detelecine_random_streams(ref, hostlogic, seed):
    """random mixtures of film pictures, woven field pairs and repeated pictures under random TFF / RFF flags and
    settings: whatever the state machine decides, it decides what the reference decides"""
    w, h = 64, 48
    fmt = FMT[8 if seed % 3 else 10]
    rng = np.random.default_rng(seed)
    film = [synth.progressive_frame(fmt, w, h, 3 * t, seed, int(rng.integers(0, 10))) for t in range(12)]
    frames, flags = [], []
    for i in range(40):
        k = rng.integers(0, 4)
        a, b = film[rng.integers(0, 12)], film[rng.integers(0, 12)]
        if k == 0:
            f = a
        elif k == 1:
            f = synth.weave(a, b, fmt, w, h)
        elif k == 2 and frames:
            f = frames[-1]
        else:
            f = film[i % 12]
        frames.append(f)
        flags.append((synth.PIC_FLAG_TOP_FIELD_FIRST if rng.random() < 0.6 else 0) | (synth.PIC_FLAG_REPEAT_FIRST_FIELD if rng.random() < 0.4 else 0))
    clip, flags = np.stack(frames), np.array(flags, np.uint16)
    settings = [None, "strict-breaks=0", "strict-breaks=1", "parity=0", "parity=1", "plane=1"][seed % 6]
    r = ref.run("hb_filter_detelecine", settings, clip, fmt, w, h, flags=flags)
    g = hostlogic.run("hb_filter_detelecine_cuda", settings, clip, fmt, w, h, flags=flags)
    compare(r, g)
