"""GPU parity: hb_filter_detelecine_cuda (host state machine + CUDA metrics / reductions / field weaving) against the
reference's hb_filter_detelecine (its stored runs, tests/reference_runs.py) -- pictures, timestamps, flags, which frames are dropped."""
import numpy as np
import pytest

from handbrake_b200 import synth
from test_detelecine import DETELECINE_CASES, FMT, compare

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("kw,settings", DETELECINE_CASES)
@pytest.mark.parametrize("depth,w,h", [(8, 160, 96), (10, 160, 96), (8, 200, 90), (10, 328, 122)])
def test_detelecine_matches_reference(ref, cuda_filters, kw, settings, depth, w, h):
    clip, flags = synth.telecined_clip(FMT[depth], w, h, 16, seed=71, **kw)
    r = ref.run("hb_filter_detelecine", settings, clip, FMT[depth], w, h, flags=flags)
    g = cuda_filters.run("hb_filter_detelecine_cuda", settings, clip, FMT[depth], w, h, flags=flags)
    compare(r, g)
    assert cuda_filters.buffers_alive() == 0


@pytest.mark.parametrize("seed", range(12))
def test_detelecine_random_streams(ref, cuda_filters, seed):
    w, h = 136, 80                     # 15 x 6 metric blocks; stride 192 > width
    fmt = FMT[8 if seed % 3 else 10]
    rng = np.random.default_rng(seed)
    film = [synth.progressive_frame(fmt, w, h, 3 * t, seed, int(rng.integers(0, 10))) for t in range(12)]
    frames, flags = [], []
    for i in range(40):
        k = rng.integers(0, 4)
        a, b = film[rng.integers(0, 12)], film[rng.integers(0, 12)]
        f = a if k == 0 else synth.weave(a, b, fmt, w, h) if k == 1 else frames[-1] if (k == 2 and frames) else film[i % 12]
        frames.append(f)
        flags.append((synth.PIC_FLAG_TOP_FIELD_FIRST if rng.random() < 0.6 else 0) | (synth.PIC_FLAG_REPEAT_FIRST_FIELD if rng.random() < 0.4 else 0))
    clip, flags = np.stack(frames), np.array(flags, np.uint16)
    settings = [None, "strict-breaks=0", "strict-breaks=1", "parity=0", "parity=1", "plane=1"][seed % 6]
    r = ref.run("hb_filter_detelecine", settings, clip, fmt, w, h, flags=flags)
    g = cuda_filters.run("hb_filter_detelecine_cuda", settings, clip, fmt, w, h, flags=flags)
    compare(r, g)


def test_detelecine_1080p_matches_reference_and_removes_the_pulldown(ref, cuda_filters):
    w, h = 1920, 1080
    n_film = 12
    clip, flags = synth.telecined_clip(FMT[8], w, h, n_film, seed=3, noise=2)
    film = [synth.progressive_frame(FMT[8], w, h, 3 * t, 3, 2) for t in range(n_film)]
    r = ref.run("hb_filter_detelecine", None, clip, FMT[8], w, h, flags=flags)
    g = cuda_filters.run("hb_filter_detelecine_cuda", None, clip, FMT[8], w, h, flags=flags)
    compare(r, g)
    for f in g.frames[1:]:
        assert sum(np.array_equal(f, film[t]) for t in range(n_film)) == 1       # a film frame again, not a woven mixture


def test_detelecine_4k_10bit_removes_the_pulldown(cuda_filters):
    """BASELINE config 3's geometry: size-independent property instead of a reference run"""
    w, h = 3840, 2160
    n_film = 8
    clip, flags = synth.telecined_clip(FMT[10], w, h, n_film, seed=4, noise=2, tff=False)
    film = [synth.progressive_frame(FMT[10], w, h, 3 * t, 4, 2) for t in range(n_film)]
    g = cuda_filters.run("hb_filter_detelecine_cuda", None, clip, FMT[10], w, h, flags=flags)
    assert not g.init_failed and g.saw_eof and 6 <= g.frames.shape[0] <= clip.shape[0]
    which = []
    for f in g.frames[1:]:
        hits = [t for t in range(n_film) if np.array_equal(f, film[t])]
        assert len(hits) == 1
        which.append(hits[0])
    assert which == sorted(set(which))


def test_detelecine_too_small_is_refused(cuda_filters):
    clip = synth.progressive_clip(FMT[8], 32, 16, 3)
    g = cuda_filters.run("hb_filter_detelecine_cuda", None, clip, FMT[8], 32, 16)
    assert g.init_failed == 1


@pytest.mark.parametrize("depth", [8, 10])
def test_detelecine_device_resident(ref, cuda_filters, depth):
    """pullup inside a device-resident chain: device frames in, device frames out (hbcu_detelecine_upload_frame /
    download_frame), bit-identical to the reference's host chain; nothing leaks"""
    import ctypes as C
    from handbrake_b200 import LIBHBCU
    UP, DOWN = "hb_filter_hbcu_upload", "hb_filter_hbcu_download"
    w, h = 720, 480
    clip, flags = synth.telecined_clip(FMT[depth], w, h, 12, seed=8, noise=2)
    r = ref.run(["hb_filter_detelecine", "hb_filter_lapsharp_mt"], [None, "y-strength=0.3"], clip, FMT[depth], w, h, flags=flags)
    g = cuda_filters.run([UP, "hb_filter_detelecine_cuda", "hb_filter_lapsharp_cuda", DOWN], [None, None, "y-strength=0.3", None],
                         clip, FMT[depth], w, h, flags=flags)
    compare(r, g)
    core = C.CDLL(str(LIBHBCU))
    core.hbcu_frames_alive.restype = C.c_long
    assert core.hbcu_frames_alive() == 0 and cuda_filters.buffers_alive() == 0
