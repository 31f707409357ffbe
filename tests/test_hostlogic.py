"""CPU tests of the product's HOST-SIDE filter code (SURVEY.md 8a a1-a3, a8: settings cascade and sanitising, weight
tables, look-ahead buffering, EOF flush, output order and properties).

oracle/_ref/libhostlogic.so is handbrake_b200/libhb/*_cuda.c compiled UNTOUCHED, with every hbcu_* device call renamed to
a plain-C stand-in built on the restatement (oracle/port/hostlogic_*.c).  Compared here with the stored runs of the
reference's own filter objects (tests/reference_runs.py).  On the GPU box the same host code drives the CUDA kernels
(tests/test_*_gpu.py)."""
import ctypes as C
import hashlib
import json
from pathlib import Path

import numpy as np
import pytest

from handbrake_b200 import synth
from conftest import ORACLE_DIR
from reference_runs import differing_frames

FMT = {8: synth.PIX_FMT_YUV420P, 10: synth.PIX_FMT_YUV420P10}
HOSTLOGIC_SO = ORACLE_DIR / "_ref" / "libhostlogic.so"


@pytest.fixture(scope="module")
def hostlogic():
    from handbrake_b200.hblib import FilterLib
    if not HOSTLOGIC_SO.exists():
        pytest.skip("oracle/_ref/libhostlogic.so not built")
    return FilterLib(HOSTLOGIC_SO)


def same_stream(r, g):
    assert not g.init_failed and g.saw_eof
    assert g.frames.shape == r.frames.shape, (g.frames.shape, r.frames.shape)
    assert np.array_equal(g.start, r.start) and np.array_equal(g.stop, r.stop) and np.array_equal(g.flags, r.flags)
    if not np.array_equal(g.frames, r.frames):
        raise AssertionError(f"frames {differing_frames(g.frames, r.frames)[:8]} differ")


NLMEANS_SETTINGS = [
    None,                                                        # filter defaults (nlmeans.c:58-69)
    "y-strength=1.5", "y-strength=3", "y-strength=6", "y-strength=10",          # presets ultralight .. strong (param.c:408-428)
    "y-strength=6:y-origin-tune=0.8:y-patch-size=5:y-range=7:y-frame-count=4",  # tune animation-like (param.c:501-523)
    "y-strength=4:cb-strength=8:cb-range=5:cr-strength=2:cr-patch-size=9",      # cascade Cr <- Cb <- Y, per-plane overrides
    "y-strength=6:y-patch-size=4:y-range=6:y-frame-count=99:y-origin-tune=7",   # sanitised: odd sizes, frames <= 32, tune in [0.01, 1]
    "y-strength=0:cb-strength=5:cr-strength=0",                                 # bypassed planes are copied
    "y-strength=6:y-frame-count=1",                                             # no temporal window
    "y-strength=6:threads=3",
    "y-strength=6:y-prefilter=1:threads=1", "y-strength=6:y-prefilter=1032:cb-prefilter=272:threads=1",
    "y-strength=5:y-prefilter=2048:threads=1",                                  # passthru
]


@pytest.mark.parametrize("settings", NLMEANS_SETTINGS)
@pytest.mark.parametrize("depth", [8, 10])
def test_nlmeans_host_filter_equals_reference(ref, hostlogic, settings, depth):
    w, h = 48, 32
    clip = synth.progressive_clip(FMT[depth], w, h, 6, seed=40 + depth)
    ref_settings = settings
    if settings and "frame-count=99" in settings:
        clip = clip[:3]                               # 32 look-ahead frames of a naive O(n^2 r^2) restatement: keep it small
    r = ref.run("hb_filter_nlmeans", ref_settings, clip, FMT[depth], w, h)
    g = hostlogic.run("hb_filter_nlmeans_cuda", settings, clip, FMT[depth], w, h)
    same_stream(r, g)
    assert hostlogic.buffers_alive() == 0


@pytest.mark.parametrize("n", [1, 2, 3, 23])
def test_nlmeans_host_filter_clip_lengths(ref, hostlogic, n):
    """shorter than the temporal window (EOF flush with a shrinking window from the first frame on) and long enough to go
    round the device ring several times"""
    w, h = 32, 32
    clip = synth.progressive_clip(FMT[8], w, h, n, seed=7)
    s = "y-strength=6:y-frame-count=3:y-range=3:y-patch-size=3"
    r = ref.run("hb_filter_nlmeans", s, clip, FMT[8], w, h)
    g = hostlogic.run("hb_filter_nlmeans_cuda", s, clip, FMT[8], w, h)
    same_stream(r, g)


MULTI_CASES = [
    # (extra settings, frames): `devices` lists the handles the ordered stream is dealt to, `block` the frames per turn
    ("y-strength=6:y-patch-size=3:y-frame-count=2:devices=0,0:block=3", 11),
    ("y-strength=6:y-patch-size=3:y-frame-count=3:devices=0,0,0:block=2", 13),        # halo of 2 = the whole next block
    ("y-strength=6:y-patch-size=3:y-frame-count=4:devices=0,0:block=1", 9),           # block raised to nframes - 1
    ("y-strength=6:y-patch-size=3:y-frame-count=2:devices=0,0,0,0:block=2", 5),       # fewer blocks than devices' turns
    ("y-strength=6:y-patch-size=3:y-frame-count=3:devices=0,0:block=4", 2),           # shorter than the window: EOF flush only
    ("y-strength=6:y-patch-size=3:y-frame-count=2:y-prefilter=1:devices=0,0:block=2:threads=1", 8),   # start-of-stream rule on frame 0 only
    ("y-strength=6:y-patch-size=3:y-frame-count=3:y-prefilter=1032:cb-prefilter=272:devices=0,0,0:block=3:threads=1", 10),
    ("y-strength=6:y-patch-size=3:y-frame-count=1:devices=0,0:block=2", 7),           # no temporal window: no halo at all
    ("y-strength=0:cb-strength=5:cb-patch-size=3:devices=0,0:block=2", 6),            # bypassed planes
]


@pytest.mark.parametrize("settings,n", MULTI_CASES)
def test_nlmeans_multi_device_dealing_equals_reference(ref, hostlogic, settings, n):
    """VERDICT r1 item 4: one ordered stream dealt block-cyclically to several device handles (mt_frame_filter.c:169-237
    deals frames to threads the same way), halo by peer copy, harvested in order == the reference's single stream.  The
    stand-in handles are CPU rings, so this pins the host side: owners, local indices, halo frames, window at block ends,
    the EOF flush, the start-of-stream rule staying with frame 0."""
    w, h = 40, 32
    clip = synth.progressive_clip(FMT[8], w, h, n, seed=90 + n)
    ref_settings = ":".join(kv for kv in settings.split(":") if not kv.startswith(("devices=", "block=")))
    r = ref.run("hb_filter_nlmeans", ref_settings, clip, FMT[8], w, h)
    g = hostlogic.run("hb_filter_nlmeans_cuda", settings, clip, FMT[8], w, h)
    same_stream(r, g)
    assert hostlogic.buffers_alive() == 0


def test_nlmeans_multi_device_env_and_bad_lists(hostlogic, monkeypatch):
    w, h = 40, 32
    clip = synth.progressive_clip(FMT[8], w, h, 7, seed=5)
    s = "y-strength=6:y-patch-size=3"
    one = hostlogic.run("hb_filter_nlmeans_cuda", s, clip, FMT[8], w, h)
    monkeypatch.setenv("HBCU_DEVICES", "0,0,0")
    monkeypatch.setenv("HBCU_BLOCK", "2")
    three = hostlogic.run("hb_filter_nlmeans_cuda", s, clip, FMT[8], w, h)
    assert np.array_equal(one.frames, three.frames) and np.array_equal(one.start, three.start)
    monkeypatch.delenv("HBCU_DEVICES")
    bad = hostlogic.run("hb_filter_nlmeans_cuda", s + ":devices=0,x", clip, FMT[8], w, h)
    assert bad.init_failed


def test_nlmeans_host_filter_reproduces_golden_digests(hostlogic):
    golden = json.loads((Path(__file__).parent / "golden" / "nlmeans_golden.json").read_text())
    for name in ("tiny_light_96x64", "tiny_tuned_10bit_64x48"):
        c = golden[name]
        clip = synth.progressive_clip(FMT[c["depth"]], c["width"], c["height"], c["frames"], seed=c["seed"])
        g = hostlogic.run("hb_filter_nlmeans_cuda", c["settings"], clip, FMT[c["depth"]], c["width"], c["height"])
        assert [hashlib.sha256(f.tobytes()).hexdigest() for f in g.frames] == c["sha256"], name


# ---------------------------------------------------------------- comb-detect, decomb, lapsharp host filters
from test_oracle import COMB_SETTINGS, DECOMB_CASES, LAPSHARP_CASES, decomb_inputs, mixed_interlaced_clip  # noqa: E402


@pytest.mark.parametrize("settings", COMB_SETTINGS)
@pytest.mark.parametrize("depth", [8, 10])
def test_comb_detect_host_filter_equals_reference(ref, hostlogic, settings, depth):
    """the three-frame window: first frame duplicated (HB_FILTER_DELAY), exhaustive check at both ends, buffers passed
    through with their verdict; also that the host's gamma table and shifted thresholds are the reference's"""
    w, h = 176, 112
    clip = mixed_interlaced_clip(FMT[depth], w, h, 9)
    flags = np.full(clip.shape[0], synth.PIC_FLAG_TOP_FIELD_FIRST, np.uint16)
    r = ref.run("hb_filter_comb_detect", settings, clip, FMT[depth], w, h, flags=flags)
    g = hostlogic.run("hb_filter_comb_detect_cuda", settings, clip, FMT[depth], w, h, flags=flags)
    same_stream(r, g)
    assert list(g.combed) == list(r.combed)
    assert hostlogic.buffers_alive() == 0


def test_comb_detect_host_filter_short_clips(ref, hostlogic):
    w, h = 96, 64
    for n in (1, 2, 3):
        clip = synth.interlaced_clip(FMT[8], w, h, n, seed=3, static_every=0)
        r = ref.run("hb_filter_comb_detect", None, clip, FMT[8], w, h)
        g = hostlogic.run("hb_filter_comb_detect_cuda", None, clip, FMT[8], w, h)
        same_stream(r, g)
        assert list(g.combed) == list(r.combed)


@pytest.mark.parametrize("mode,parity,tags", DECOMB_CASES + [(24, -1, False), (31, -1, False), (63, -1, True), (15, 1, True)])
@pytest.mark.parametrize("depth", [8, 10])
def test_decomb_host_filter_equals_reference(ref, hostlogic, mode, parity, tags, depth):
    """per-frame mode from the combed tag, parity / field order from flags and the setting, bob timestamps and frame
    rate, one EEDI2 call per rebuilt field with the mask state carried along"""
    w, h = (96, 52) if not mode & 8 else (112, 64)
    clip, flags, combed = decomb_inputs(depth, w, h, 6)
    s = f"mode={mode}:parity={parity}"
    r = ref.run("hb_filter_decomb", s, clip, FMT[depth], w, h, flags=flags, combed=combed if tags else None)
    g = hostlogic.run("hb_filter_decomb_cuda", s, clip, FMT[depth], w, h, flags=flags, combed=combed if tags else None)
    same_stream(r, g)
    assert list(g.combed) == list(r.combed) and g.vrate == r.vrate
    assert hostlogic.buffers_alive() == 0


def test_comb_detect_then_decomb_host_chain(ref, hostlogic):
    w, h = 160, 96
    clip, flags, _ = decomb_inputs(8, w, h, 8, seed=9)
    s = [None, "mode=39"]
    r = ref.run(["hb_filter_comb_detect", "hb_filter_decomb"], s, clip, FMT[8], w, h, flags=flags)
    g = hostlogic.run(["hb_filter_comb_detect_cuda", "hb_filter_decomb_cuda"], s, clip, FMT[8], w, h, flags=flags)
    same_stream(r, g)
    assert list(g.combed) == list(r.combed) and len(set(r.combed)) > 1


@pytest.mark.parametrize("settings,strengths,kernels", LAPSHARP_CASES + [("y-strength=9:y-kernel=nonsense", None, None)])
@pytest.mark.parametrize("depth", [8, 10])
def test_lapsharp_host_filter_equals_reference(ref, hostlogic, settings, strengths, kernels, depth):
    w, h = 200, 90
    clip = synth.progressive_clip(FMT[depth], w, h, 5, seed=31, noise=20)
    r = ref.run("hb_filter_lapsharp_mt", settings, clip, FMT[depth], w, h)
    g = hostlogic.run("hb_filter_lapsharp_cuda", settings, clip, FMT[depth], w, h)
    same_stream(r, g)


# ---------------------------------------------------------------- unsharp, chroma smooth, hqdn3d host filters
from test_oracle import CHROMA_SMOOTH_CASES, UNSHARP_CASES  # noqa: E402


@pytest.mark.parametrize("settings", [c[0] for c in UNSHARP_CASES])
@pytest.mark.parametrize("depth", [8, 10])
def test_unsharp_host_filter_equals_reference(ref, hostlogic, settings, depth):
    w, h = 150, 98
    clip = synth.progressive_clip(FMT[depth], w, h, 4, seed=51)
    same_stream(ref.run("hb_filter_unsharp_mt", settings, clip, FMT[depth], w, h),
                hostlogic.run("hb_filter_unsharp_cuda", settings, clip, FMT[depth], w, h))


@pytest.mark.parametrize("settings", [c[0] for c in CHROMA_SMOOTH_CASES])
@pytest.mark.parametrize("depth", [8, 10])
def test_chroma_smooth_host_filter_equals_reference(ref, hostlogic, settings, depth):
    w, h = 150, 98
    clip = synth.progressive_clip(FMT[depth], w, h, 4, seed=53)
    same_stream(ref.run("hb_filter_chroma_smooth_mt", settings, clip, FMT[depth], w, h),
                hostlogic.run("hb_filter_chroma_smooth_cuda", settings, clip, FMT[depth], w, h))


@pytest.mark.parametrize("settings", [None, "y-spatial=2", "y-spatial=7:cb-spatial=7:cr-spatial=7:y-temporal=7:cb-temporal=5:cr-temporal=5",
                                      "y-spatial=0:y-temporal=4", "y-spatial=3:cb-spatial=0:cr-temporal=0", "y-spatial=300:y-temporal=300"])
@pytest.mark.parametrize("depth", [8, 10])
def test_hqdn3d_host_filter_equals_reference(ref, hostlogic, settings, depth):
    """the default chain of denoise.c:237-266 and the coefficient tables the host computes (hqdn3d_precalc_coef)"""
    w, h = 96, 64
    clip = synth.progressive_clip(FMT[depth], w, h, 6, seed=61, noise=10)
    same_stream(ref.run("hb_filter_denoise", settings, clip, FMT[depth], w, h),
                hostlogic.run("hb_filter_denoise_cuda", settings, clip, FMT[depth], w, h))
    assert hostlogic.buffers_alive() == 0


@pytest.mark.parametrize("seed", range(16))
def test_random_settings_all_host_filters(ref, hostlogic, seed):
    """random (also out-of-range) settings for every filter object: whatever the reference's init() makes of them, the
    drop-in's init() makes the same"""
    rng = np.random.default_rng(seed)
    depth = 8 if rng.random() < 0.6 else 10
    fmt = FMT[depth]
    jobs = []
    mode = int(rng.integers(0, 64)) & ~8
    w, h = 96, 52
    clip, flags, combed = decomb_inputs(depth, w, h, 5, seed=seed)
    flags = np.array([int(rng.choice([0, 0x08, 0x10, 0x18])) for _ in range(clip.shape[0])], np.uint16)
    combed = rng.integers(0, 3, clip.shape[0]).astype(np.uint8)
    jobs.append(("hb_filter_decomb", "hb_filter_decomb_cuda", f"mode={mode}:parity={int(rng.integers(-1, 2))}", clip, w, h, dict(flags=flags, combed=combed)))
    s = (f"mode={int(rng.integers(0, 4))}:spatial-metric={int(rng.integers(0, 3))}:motion-thresh={int(rng.integers(0, 8))}:"
         f"spatial-thresh={int(rng.integers(0, 8))}:filter-mode={int(rng.integers(0, 3))}:block-thresh={int(rng.integers(1, 120))}:"
         f"block-width={int(rng.integers(4, 40))}:block-height={int(rng.integers(4, 40))}")
    w, h = 112, 80
    clip = mixed_interlaced_clip(fmt, w, h, 4, seed=seed)
    jobs.append(("hb_filter_comb_detect", "hb_filter_comb_detect_cuda", s, clip, w, h, dict(flags=np.full(clip.shape[0], 8, np.uint16))))
    parts = []
    for c in ("y", "cb", "cr"):
        if c == "y" or rng.random() < 0.5:
            parts.append(f"{c}-strength={rng.choice([0, 1.5, 3, 6, 10, 20])}")
        if rng.random() < 0.4:
            parts.append(f"{c}-patch-size={int(rng.integers(0, 12))}")
        if rng.random() < 0.4:
            parts.append(f"{c}-range={int(rng.integers(0, 8))}")
        if rng.random() < 0.4:
            parts.append(f"{c}-frame-count={int(rng.integers(0, 5))}")
        if rng.random() < 0.3:
            parts.append(f"{c}-origin-tune={rng.choice([0, 0.005, 0.3, 1, 2.5])}")
        if rng.random() < 0.3:
            parts.append(f"{c}-prefilter={int(rng.choice([1, 2, 4, 8, 16, 32, 257, 514, 1028, 2049, 1024, 256]))}")
    w, h = 40, 24
    jobs.append(("hb_filter_nlmeans", "hb_filter_nlmeans_cuda", ":".join(parts + ["threads=1"]), synth.progressive_clip(fmt, w, h, 5, seed=seed), w, h, {}))
    w, h = 88, 50
    clip = synth.progressive_clip(fmt, w, h, 3, seed=seed, noise=15)
    ks = ["lap", "isolap", "log", "isolog", "bogus"]
    jobs.append(("hb_filter_lapsharp_mt", "hb_filter_lapsharp_cuda", f"y-strength={rng.choice([0, 0.2, 1.5, 3])}:y-kernel={rng.choice(ks)}:cb-strength={rng.choice([0, 0.5, 9])}:cr-kernel={rng.choice(ks)}", clip, w, h, {}))
    jobs.append(("hb_filter_unsharp_mt", "hb_filter_unsharp_cuda", f"y-strength={rng.choice([-1, 0, 0.25, 1.5, 4])}:y-size={int(rng.integers(0, 20))}:cb-size={int(rng.integers(0, 20))}", clip, w, h, {}))
    jobs.append(("hb_filter_chroma_smooth_mt", "hb_filter_chroma_smooth_cuda", f"cb-strength={rng.choice([-1, 0, 0.25, 3, 8])}:cb-size={int(rng.integers(0, 20))}:cr-size={int(rng.integers(0, 20))}", clip, w, h, {}))
    jobs.append(("hb_filter_denoise", "hb_filter_denoise_cuda", f"y-spatial={rng.choice([0, 1, 4, 40, 300])}:cb-temporal={rng.choice([0, 2, 6, 100])}:cr-spatial={rng.choice([0, 3, 9])}", clip, w, h, {}))
    for rname, gname, settings, clip, w, h, kw in jobs:
        r = ref.run(rname, settings, clip, fmt, w, h, **kw)
        g = hostlogic.run(gname, settings, clip, fmt, w, h, **kw)
        assert r.init_failed == g.init_failed, (gname, settings)
        same_stream(r, g) if not r.init_failed else None
        assert list(g.combed) == list(r.combed) and g.vrate == r.vrate, (gname, settings)


@pytest.mark.parametrize("n", [0, 1, 2])
@pytest.mark.parametrize("w,h", [(96, 64), (70, 50)])
def test_empty_and_tiny_streams_all_host_filters(ref, hostlogic, n, w, h):
    """EOF as the first buffer, one picture, two pictures; a size whose chroma planes are odd"""
    fmt = FMT[8]
    clip = synth.progressive_clip(fmt, w, h, max(n, 1), seed=2)[:n]
    pairs = [("hb_filter_nlmeans", "hb_filter_nlmeans_cuda", "y-strength=6"), ("hb_filter_comb_detect", "hb_filter_comb_detect_cuda", None),
             ("hb_filter_decomb", "hb_filter_decomb_cuda", "mode=23"), ("hb_filter_lapsharp_mt", "hb_filter_lapsharp_cuda", None),
             ("hb_filter_unsharp_mt", "hb_filter_unsharp_cuda", None), ("hb_filter_chroma_smooth_mt", "hb_filter_chroma_smooth_cuda", None),
             ("hb_filter_denoise", "hb_filter_denoise_cuda", None), ("hb_filter_detelecine", "hb_filter_detelecine_cuda", None)]
    if (h // 2) % 2 == 0:
        pairs.append(("hb_filter_decomb", "hb_filter_decomb_cuda", "mode=31"))
    for rname, gname, settings in pairs:
        r = ref.run(rname, settings, clip, fmt, w, h)
        g = hostlogic.run(gname, settings, clip, fmt, w, h)
        same_stream(r, g)
    assert hostlogic.buffers_alive() == 0


# ---------------------------------------------------------------- device-resident chains, host side (SURVEY.md 8 f3)
UP, DOWN = "hb_filter_hbcu_upload", "hb_filter_hbcu_download"


def device_frames_alive(hostlogic):
    import ctypes as C
    hostlogic.lib.oracle_hbcu_frames_alive.restype = C.c_long
    return hostlogic.lib.oracle_hbcu_frames_alive()


@pytest.mark.parametrize("depth", [8, 10])
def test_device_resident_chain_host_side(ref, hostlogic, depth):
    """comb_detect -> decomb (selective) -> NLMeans -> lapsharp -> unsharp -> hqdn3d between the upload and download
    adapters: HBCU_DEVICE buffers, shallow dups of passed-through frames, hw_pix_fmt propagation, reference counts --
    with host memory standing in for device frames (oracle/port/hostlogic_frames.c).  Same pictures as the reference's
    plain chain, nothing left alive."""
    w, h = 144, 84                     # luma stride 192 > width: lapsharp reads the mirrored padding of a device frame
    clip, flags, _ = decomb_inputs(depth, w, h, 7, seed=3)
    names_r = ["hb_filter_comb_detect", "hb_filter_decomb", "hb_filter_denoise", "hb_filter_nlmeans", "hb_filter_chroma_smooth_mt", "hb_filter_lapsharp_mt",
               "hb_filter_unsharp_mt"]
    names_g = [UP] + [n.replace("_mt", "") + "_cuda" for n in names_r] + [DOWN]
    s = [None, "mode=39", "y-spatial=2", "y-strength=6:y-patch-size=3:y-range=3:threads=1", "cb-strength=0.8", "y-strength=0.2:y-kernel=isolap", "y-strength=0.4:y-size=5"]
    r = ref.run(names_r, s, clip, FMT[depth], w, h, flags=flags)
    g = hostlogic.run(names_g, [None] + s + [None], clip, FMT[depth], w, h, flags=flags)
    same_stream(r, g)
    assert list(g.combed) == list(r.combed) and len(set(r.combed)) > 1
    assert device_frames_alive(hostlogic) == 0 and hostlogic.buffers_alive() == 0


def test_mixed_host_and_device_segments_host_side(ref, hostlogic):
    w, h = 112, 64
    clip, flags, _ = decomb_inputs(8, w, h, 6, seed=13)
    r = ref.run(["hb_filter_comb_detect", "hb_filter_decomb", "hb_filter_nlmeans"], [None, "mode=63", "y-strength=3:y-patch-size=3:threads=1"], clip, FMT[8], w, h, flags=flags)
    g = hostlogic.run([UP, "hb_filter_comb_detect_cuda", "hb_filter_decomb_cuda", DOWN, "hb_filter_nlmeans_cuda"],
                      [None, None, "mode=63", None, "y-strength=3:y-patch-size=3"], clip, FMT[8], w, h, flags=flags)
    same_stream(r, g)
    assert g.vrate == r.vrate
    assert device_frames_alive(hostlogic) == 0 and hostlogic.buffers_alive() == 0


def test_device_chain_misuse_fails_loudly_host_side(hostlogic):
    w, h = 96, 64
    clip = synth.progressive_clip(FMT[8], w, h, 3)
    with pytest.raises(RuntimeError):                    # no download adapter: the sink refuses device buffers
        hostlogic.run([UP, "hb_filter_lapsharp_cuda"], [None, "y-strength=0.2"], clip, FMT[8], w, h)
    assert device_frames_alive(hostlogic) == 0 and hostlogic.buffers_alive() == 0


@pytest.mark.parametrize("depth", [8, 10])
def test_detelecine_inside_a_device_resident_chain(ref, hostlogic, depth):
    """VERDICT r1 missing 4: pullup between the adapters -- pictures arrive in and leave in device frames (frame twins of
    upload / download), pass-through pictures travel on as the device buffers they came in; == the reference's host chain"""
    w, h = 136, 80
    clip, flags = synth.telecined_clip(FMT[depth], w, h, 10, seed=6, noise=2)
    r = ref.run(["hb_filter_detelecine", "hb_filter_lapsharp_mt"], [None, "y-strength=0.3"], clip, FMT[depth], w, h, flags=flags)
    g = hostlogic.run([UP, "hb_filter_detelecine_cuda", "hb_filter_lapsharp_cuda", DOWN], [None, None, "y-strength=0.3", None], clip, FMT[depth], w, h, flags=flags)
    same_stream(r, g)
    g2 = hostlogic.run(["hb_filter_detelecine_cuda", UP, "hb_filter_lapsharp_cuda", DOWN], [None, None, "y-strength=0.3", None], clip, FMT[depth], w, h, flags=flags)
    same_stream(r, g2)
    assert device_frames_alive(hostlogic) == 0 and hostlogic.buffers_alive() == 0


def test_wrapped_decoder_surfaces_through_a_device_chain(ref, hostlogic, monkeypatch):
    """The NVDEC end of a zero-copy chain (VERDICT r1 item 8 / SURVEY.md 8 f4): with HBCU_UPLOAD_EXTERNAL the upload adapter
    plays a hardware decoder -- what goes downstream is hbcu_wrap_cuda_frame() around planes the "decoder" owns.  The chain's
    output equals the reference's, every surface goes back to its owner exactly once, nothing leaks."""
    w, h, n = 64, 48, 7
    clip = synth.progressive_clip(FMT[8], w, h, n, seed=77)
    r = ref.run(["hb_filter_nlmeans", "hb_filter_lapsharp_mt"], ["y-strength=6:y-patch-size=3:threads=1", "y-strength=0.3"], clip, FMT[8], w, h)
    monkeypatch.setenv("HBCU_UPLOAD_EXTERNAL", "1")
    hostlogic.lib.hbcu_test_surfaces_returned.restype = C.c_long
    before = hostlogic.lib.hbcu_test_surfaces_returned()
    g = hostlogic.run([UP, "hb_filter_nlmeans_cuda", "hb_filter_lapsharp_cuda", DOWN], [None, "y-strength=6:y-patch-size=3", "y-strength=0.3", None],
                      clip, FMT[8], w, h)
    same_stream(r, g)
    assert hostlogic.lib.hbcu_test_surfaces_returned() - before == n
    assert hostlogic.buffers_alive() == 0


@pytest.mark.parametrize("devices", ["0,0", "0,0,0", "0,0,0,0,0"])
def test_frame_parallel_filters_dealt_over_devices(ref, hostlogic, devices):
    """the mt_frame clients (lapsharp, unsharp, chroma smooth: frames are independent, mt_frame_filter.c:169-237) with
    `devices=`: frame t goes to handle t % n, outputs leave in stream order; == the reference"""
    w, h, n = 96, 64, 17
    clip = synth.progressive_clip(FMT[8], w, h, n, seed=21)
    for ref_name, name, settings in (("hb_filter_lapsharp_mt", "hb_filter_lapsharp_cuda", "y-strength=0.3:y-kernel=isolap"),
                                     ("hb_filter_unsharp_mt", "hb_filter_unsharp_cuda", "y-strength=0.5:y-size=5"),
                                     ("hb_filter_chroma_smooth_mt", "hb_filter_chroma_smooth_cuda", "cb-strength=0.8:cb-size=5")):
        r = ref.run(ref_name, settings, clip, FMT[8], w, h)
        g = hostlogic.run(name, settings + ":devices=" + devices, clip, FMT[8], w, h)
        same_stream(r, g)
    bad = hostlogic.run("hb_filter_lapsharp_cuda", "y-strength=0.3:devices=0,,1", clip, FMT[8], w, h)
    assert bad.init_failed
    assert hostlogic.buffers_alive() == 0


@pytest.mark.parametrize("devices,block", [("0,0", 3), ("0,0,0", 2), ("0,0", 1), ("0,0,0,0", 4)])
@pytest.mark.parametrize("depth", [8, 10])
def test_decomb_dealt_over_devices(ref, hostlogic, devices, block, depth):
    """decomb (yadif / blend / cubic / bob / selective, no EEDI2) with `devices=`: block-cyclic owners, the first and the
    last frame of a block also uploaded to the neighbouring block's device (prev / next), pictures out in order == the
    reference; EEDI2 modes refuse several devices at init"""
    w, h = 96, 64
    clip, flags, combed = decomb_inputs(depth, w, h, 11, seed=14)
    for mode, tags in ((7, None), (39, combed), (23, None), (4, None), (2, None), (55, combed)):
        r = ref.run("hb_filter_decomb", f"mode={mode}", clip, FMT[depth], w, h, flags=flags, combed=tags)
        g = hostlogic.run("hb_filter_decomb_cuda", f"mode={mode}:devices={devices}:block={block}", clip, FMT[depth], w, h, flags=flags, combed=tags)
        same_stream(r, g)
        assert r.vrate == g.vrate
    g = hostlogic.run("hb_filter_decomb_cuda", f"mode=15:devices={devices}", clip, FMT[depth], w, h, flags=flags)
    assert g.init_failed
    assert hostlogic.buffers_alive() == 0
