#!/usr/bin/env python
"""bench.py -- hot-path benchmark (contract in the task statement, section 4).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A *step* is one pass of the NLMeans hot path over one batch of `--batch` synthetic frames per GPU, taken from ONE
continuous frame stream per GPU (weak scaling: every rank filters its own block of the clip; the stream never
restarts between steps, so no step pays a pipeline fill or an EOF flush).  With the defaults (K = 20 steps of 768
frames) both timed regions last seconds, not milliseconds.

  value     frames/s, whole job, inputs already resident in HBM (border + NLMeans kernels, CUDA events on the
            compute streams; the step's inputs cycle through 32 distinct device frames = 398 MB > 126 MB L2)
  e2e       frames/s through hb_filter_nlmeans_cuda.work() with HOST hb_buffer_t frames: pinned H2D + kernels +
            D2H into fresh output buffers, all inside the timed region (hb_bench.c: decoder-style input buffers
            over a bounded ring of pinned payloads)
  roofline  algorithmic HBM bytes of the NLMeans kernel (3 x frame bytes per output frame, SURVEY.md 8d) / its
            CUDA-event time, against MEASURED_PEAKS.json; issue_frac = warp instructions of one launch (committed
            ncu capture) / (148 SMs x 4 schedulers x clock x kernel time) -- the roofline this kernel actually sits under
  cpu_baseline / --impl reference
            the reference's own nlmeans.c + nlmeans_x86.c (oracle/_ref/libhbref.so, compiled unmodified from
            /root/reference) on this box's host cores, same frames, same protocol, one continuous stream
  extra     (N = 1) the other BASELINE.json configurations, each with e2e / cpu_baseline / roofline:
            config 2 (1080p NLMeans medium), config 3 (4K 10-bit comb-detect + decomb EEDI2 bob), config 4 with the
            large search window (patch 5, range 7, frames 4), config 5 (8K 10-bit chain, frames device-resident
            between the filters)
  copy_only the e2e pipeline with every plane bypassed: the transfer ceiling of this box at this N
"""
import argparse
import ctypes as C
import json
import os
import re
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

from handbrake_b200 import synth  # noqa: E402

WORKLOADS = {
    # BASELINE.json configs[3]: the configuration the metric ("4K NLMeans frames/sec at 1/2/4/8 B200") is quoted on
    "4k_nlmeans_strong": dict(width=3840, height=2160, depth=8, settings="y-strength=10", nframes=2,
                              desc="3840x2160 yuv420p 8-bit, NLMeans 'strong' (strength 10, patch 7, range 3, frames 2)"),
    "4k_nlmeans_medium": dict(width=3840, height=2160, depth=8, settings="y-strength=6", nframes=2,
                              desc="3840x2160 yuv420p 8-bit, NLMeans 'medium'"),
    "4k_nlmeans_strong_animation": dict(width=3840, height=2160, depth=8, nframes=4,
                                        settings="y-strength=10:y-origin-tune=0.15:y-patch-size=5:y-range=7:y-frame-count=4",
                                        desc="3840x2160 8-bit, NLMeans strong + large search window (patch 5, range 7, frames 4)"),
    # BASELINE.json configs[1]
    "1080p_nlmeans_medium": dict(width=1920, height=1080, depth=8, settings="y-strength=6", nframes=2,
                                 desc="1920x1080 yuv420p 8-bit, NLMeans 'medium'"),
    # BASELINE.json configs[0] (the reference's CPU-runnable case)
    "360p_nlmeans_light": dict(width=640, height=360, depth=8, settings="y-strength=3", nframes=2,
                               desc="640x360 yuv420p 8-bit, NLMeans 'light'"),
    # diagnostic: every plane bypassed (strength 0) -> the transfer pipeline alone
    "4k_copy_only": dict(width=3840, height=2160, depth=8, settings="y-strength=0", nframes=2,
                         desc="3840x2160 yuv420p 8-bit, NLMeans strength 0 (bypass copy): transfer pipeline diagnostic"),
    # a prefilter mode (custom settings only, nlmeans.c:72-83): 8-bit planes run the prefilter variant of the v3 kernel
    "4k_nlmeans_medium_prefilter": dict(width=3840, height=2160, depth=8, settings="y-strength=6:y-prefilter=1", nframes=2,
                                        desc="3840x2160 yuv420p 8-bit, NLMeans 'medium' with the 3x3 mean prefilter"),
    "4k10_nlmeans_medium": dict(width=3840, height=2160, depth=10, settings="y-strength=6", nframes=2,
                                desc="3840x2160 yuv420p10 NLMeans 'medium'"),
}

COMB_DEFAULT = "mode=3:spatial-metric=2:motion-thresh=1:spatial-thresh=1:filter-mode=2:block-thresh=40:block-width=16:block-height=16"

# the other BASELINE.json configurations, reported in `extra` (N = 1).  alg_f = algorithmic HBM bytes per INPUT frame in
# units of the frame size F (SURVEY.md 8d): NLMeans (nframes + 1) F; comb-detect 3 Y (Y = 2/3 F at 4:2:0);
# decomb 4 F per output picture (bob: two pictures per input frame); lapsharp 2 F.
EXTRAS = [
    dict(name="cfg2_1080p_nlmeans_medium", config="BASELINE.json configs[1]", width=1920, height=1080, depth=8, interlaced=False,
         filters=["nlmeans"], settings=["y-strength=6"], frames=300, alg_f=3.0, nlm_workload="1080p_nlmeans_medium",
         desc="1920x1080 yuv420p 8-bit, NLMeans 'medium', 300-frame clip"),
    dict(name="cfg3_4k10_comb_detect_decomb_eedi2bob", config="BASELINE.json configs[2]", width=3840, height=2160, depth=10, interlaced=True,
         filters=["comb_detect", "decomb"], settings=[COMB_DEFAULT, "mode=63"], frames=300, alg_f=2.0 + 8.0 * 0.8,
         desc="3840x2160 yuv420p10 interlaced (1 static frame in 5), comb_detect -> decomb EEDI2 bob (mode 31 + selective), 300-frame clip",
         alg_note="comb-detect 3 Y = 2 F per frame + EEDI2 bob 8 F per combed frame (4 of 5 frames)"),
    dict(name="cfg4_4k_nlmeans_strong_large_window", config="BASELINE.json configs[3], 'large search window' variant", width=3840, height=2160,
         depth=8, interlaced=False, filters=["nlmeans"], settings=[WORKLOADS["4k_nlmeans_strong_animation"]["settings"]], frames=64,
         alg_f=5.0, nlm_workload="4k_nlmeans_strong_animation",
         desc="3840x2160 yuv420p 8-bit, NLMeans strong with the animation tune's window (patch 5, range 7, frames 4: 195 displacements per plane)"),
    dict(name="cfg5_8k10_chain_decomb_nlmeans_lapsharp", config="BASELINE.json configs[4]", width=7680, height=4320, depth=10, interlaced=True,
         filters=["decomb", "nlmeans", "lapsharp"], settings=["mode=7", "y-strength=6", "y-strength=0.2:y-kernel=isolap"], frames=64,
         alg_f=4.0 + 3.0 + 2.0, n_unique=3,
         desc="7680x4320 yuv420p10 interlaced: decomb (yadif, every frame) -> NLMeans medium -> lapsharp, frames device-resident between the filters "
              "(libhb orders filters by id: decomb runs before NLMeans)",
         alg_note="decomb 4 F + NLMeans 3 F + lapsharp 2 F per frame"),
]


# the reference's own filters (oracle/Makefile builds them from a HandBrake source tree); the CPU baseline runs them
REF_SO = REPO / "oracle" / "_ref" / "libhbref.so"
REF_HOWTO = "build it with `make -C oracle ref REF=<HandBrake source tree>`"


class BenchStats(C.Structure):
    _fields_ = [("seconds", C.c_double), ("frames_out", C.c_int64), ("bytes_in", C.c_int64),
                ("bytes_out", C.c_int64), ("checksum", C.c_uint64), ("ring_misses", C.c_int64)]


class NlmPlane(C.Structure):
    _fields_ = [("patch_size", C.c_int), ("range", C.c_int), ("nframes", C.c_int), ("bypass", C.c_int),
                ("origin_tune", C.c_double), ("weight_fact", C.c_float), ("diff_max", C.c_int),
                ("exptable", C.c_float * 128), ("prefilter", C.c_int)]


class NlmConfig(C.Structure):
    _fields_ = [("width", C.c_int), ("height", C.c_int), ("depth", C.c_int), ("chroma_shift_w", C.c_int),
                ("chroma_shift_h", C.c_int), ("device", C.c_int), ("ring_frames", C.c_int), ("out_slots", C.c_int),
                ("plane", NlmPlane * 3)]


class DecombConfig(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("width", "height", "depth", "chroma_shift_w", "chroma_shift_h", "device", "slots", "out_slots",
                                      "mode", "magnitude_threshold", "variance_threshold", "laplacian_threshold", "dilation_threshold",
                                      "erosion_threshold", "noise_threshold", "maximum_search_distance", "post_processing")]


def fmt_of(depth):
    return synth.PIX_FMT_YUV420P if depth == 8 else synth.PIX_FMT_YUV420P10


def bind_bench(lib):
    lib.hb_bench_open.restype = C.c_void_p
    lib.hb_bench_open.argtypes = [C.c_void_p, C.c_char_p, C.c_int, C.c_int, C.c_int]
    lib.hb_bench_open_chain.restype = C.c_void_p
    lib.hb_bench_open_chain.argtypes = [C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_char_p), C.c_int, C.c_int, C.c_int, C.c_int]
    lib.hb_bench_run.restype = C.c_int
    lib.hb_bench_run.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.POINTER(BenchStats)]
    lib.hb_bench_stream.restype = C.c_int
    lib.hb_bench_stream.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(BenchStats)]
    lib.hb_bench_finish.restype = C.c_int
    lib.hb_bench_finish.argtypes = [C.c_void_p, C.POINTER(BenchStats)]
    if hasattr(lib, "hb_bench_prefill"):
        lib.hb_bench_prefill.restype = C.c_int
        lib.hb_bench_prefill.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int]
    lib.hb_shim_set_log_level.argtypes = [C.c_int]
    lib.hb_shim_set_log_level(-1)
    lib.hb_shim_set_zero_buffers(0)     # like libhb's buffer pool: recycled, not zeroed
    lib.hb_get_cpu_count.restype = C.c_int


def open_chain(lib, names, settings, fmt, w, h, flags):
    protos = (C.c_void_p * len(names))(*[C.addressof(C.c_char.in_dll(lib, x)) for x in names])
    sets = (C.c_char_p * len(names))(*[(s.encode() if s else None) for s in settings])
    b = lib.hb_bench_open_chain(len(names), protos, sets, fmt, w, h, flags)
    if not b:
        raise RuntimeError(f"init of chain {names} failed")
    return b


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)"""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            p = [x.strip() for x in r.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1])); pw.append(float(p[2]))
            except ValueError:
                continue
            for n, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        # median over the samples taken under load (the sampler also sees the gaps between the two arms)
        busy = [s for s, w in zip(sm, pw) if w > 0.6 * max(pw)] if pw else sm
        return dict(sm_mhz=statistics.median(busy or sm) if sm else None, sm_max_mhz=max(mx) if mx else None,
                    power_w_max=max(pw) if pw else None, reasons=sorted(reasons), samples=len(sm))


def measured_peaks():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text()).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def gpu_numa_cpus(gpu_index):
    """CPU list of the NUMA node the GPU's PCIe link hangs off (sysfs, else the 'CPU Affinity' column of nvidia-smi topo -m)"""
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(gpu_index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip()
        bdf = out.lower()
        if bdf.startswith("00000000:"):
            bdf = bdf[4:]
        return Path(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read_text().strip() or None
    except Exception:
        pass
    try:
        topo = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=30).stdout
        for line in topo.splitlines():
            line = re.sub(r"\x1b\[[0-9;]*m", "", line)
            tok = line.split()
            if not tok or tok[0] != f"GPU{gpu_index}":
                continue
            for t in tok[1:]:
                if re.fullmatch(r"\d+(-\d+)?(,\d+(-\d+)?)*", t) and ("-" in t or "," in t):
                    return t
    except Exception:
        pass
    return None


def cpu_set(spec):
    ids = set()
    for part in spec.split(","):
        a, _, b = part.partition("-")
        ids.update(range(int(a), int(b or a) + 1))
    return ids


def bind_to_gpu_numa_node(gpu_index):
    """one process per GPU: keep the process (and the pinned frame buffers it is about to allocate: first touch) on the
    NUMA node of its GPU; best effort"""
    spec = gpu_numa_cpus(gpu_index)
    if not spec:
        return None
    try:
        ids = cpu_set(spec) & os.sched_getaffinity(0)
        if ids:
            os.sched_setaffinity(0, ids)
            return spec
    except Exception:
        pass
    return None


def pick_gpu(local_rank, world):
    """physical GPU of this rank.  Host memory bandwidth per socket, not PCIe, bounds the end-to-end arm once four
    GPUs stream through one socket (SCALE_r01: 39.8 -> 26 GB/s per GPU and direction), so a job smaller than the box
    spreads its ranks over both sockets: N = 2 -> GPUs 0, 4; N = 4 -> 0, 1, 4, 5.  HBCU_BENCH_GPUS=i,j,.. overrides."""
    env = os.environ.get("HBCU_BENCH_GPUS")
    if env:
        ids = [int(x) for x in env.split(",")]
        return ids[local_rank % len(ids)]
    try:
        import torch
        ndev = torch.cuda.device_count()
    except Exception:
        ndev = world
    if ndev >= 2 * world and ndev % 2 == 0 and world > 1:
        half = ndev // 2
        per = (world + 1) // 2
        return (local_rank // per) * half + (local_rank % per)
    return local_rank


def numa_of_pinned():
    """pages per NUMA node of this process's large mappings (the pinned frame pool among them), from
    /proc/self/numa_maps; evidence for where the pinned buffers live"""
    tot = {}
    try:
        for line in Path("/proc/self/numa_maps").read_text().splitlines():
            pages = {int(m.group(1)): int(m.group(2)) for m in re.finditer(r"\bN(\d+)=(\d+)", line)}
            if sum(pages.values()) * 4096 < (8 << 20):
                continue
            for k, v in pages.items():
                tot[k] = tot.get(k, 0) + v
    except Exception:
        return None
    return {f"node{k}_MB": round(v * 4096 / 1e6) for k, v in sorted(tot.items())} or None


def nlm_config(flt, wl, device, ring, out_slots):
    """device configuration from the settings string, built by the filter's own init code
    (hb_nlmeans_cuda_build_config in nlmeans_cuda.c: the numeric contract of nlmeans.c:343-358)"""
    cfg = NlmConfig()
    flt.hb_parse_filter_settings.restype = C.c_void_p
    flt.hb_parse_filter_settings.argtypes = [C.c_char_p]
    flt.hb_nlmeans_cuda_build_config.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.POINTER(NlmConfig),
                                                 C.c_void_p, C.c_void_p, C.c_void_p]
    d = flt.hb_parse_filter_settings(wl["settings"].encode())
    if flt.hb_nlmeans_cuda_build_config(d, fmt_of(wl["depth"]), wl["width"], wl["height"], C.byref(cfg), None, None, None) != 0:
        raise RuntimeError("bad NLMeans settings")
    cfg.device, cfg.ring_frames, cfg.out_slots = device, ring, out_slots
    return cfg


def plane_ptrs(t, dims, bps):
    base, off, ptrs, strides = t.data_ptr(), 0, [], []
    for (w, hh) in dims:
        ptrs.append(base + off); strides.append(w * bps); off += w * hh * bps
    return (C.c_void_p * 3)(*ptrs), (C.c_int * 3)(*strides)


class _DeviceBytes:
    """rows x pitch bytes of device memory, for torch.as_tensor"""

    def __init__(self, ptr, pitch, rows):
        self.__cuda_array_interface__ = {"shape": (rows, pitch), "typestr": "|u1", "data": (ptr, False), "version": 3}


def device_plane(torch, ptr, pitch, w, h, bps):
    """copy of an h x w plane (bps bytes a sample) at a device pointer with the given row pitch, as a numpy array"""
    rows = torch.as_tensor(_DeviceBytes(ptr, pitch, h), device="cuda").cpu().numpy()
    return np.ascontiguousarray(rows[:, : w * bps]).view(np.uint16 if bps == 2 else np.uint8)


DUMP_BYTES = 63 * 10**6          # payload; the three .npy headers stay inside 64 MB


def dump_outputs(out_dir, frames):
    """frames: the output frames, each [Y, U, V] planes.  Writes y.npy, u.npy, v.npy as float32 of shape (frames, h, w)
    when everything fits in DUMP_BYTES, else (frames, k) at the same k positions of every frame, k proportional to the
    plane's size and drawn without replacement by np.random.default_rng(plane number), in raster order."""
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    total = len(frames) * sum(p.size for p in frames[0]) * 4
    for i, name in enumerate(("y", "u", "v")):
        a = np.stack([f[i] for f in frames]).astype(np.float32)
        if total > DUMP_BYTES:
            k = a[0].size * DUMP_BYTES // total
            pos = np.sort(np.random.default_rng(i).choice(a[0].size, k, replace=False))
            a = a.reshape(len(frames), -1)[:, pos]
        np.save(out_dir / f"{name}.npy", a)


def ncu_capture(workload, depth):
    """numbers of the committed `ncu --set full` capture of this workload's kernel (never measured live: a run under
    ncu is not a bench value)"""
    names = {("4k_nlmeans_strong", 8): ["r02_nlmeans_v3_ncu.json", "r01g_nlmeans_fused_ncu.json"],
             ("4k10_nlmeans_medium", 10): ["r02_nlmeans_v3w_ncu.json"]}
    for n in names.get((workload, depth), []):
        p = REPO / "profiles" / n
        if p.exists():
            return json.loads(p.read_text()), f"profiles/{n}"
    return None, None


class Ours:
    """the CUDA libraries + torch, bound once per process"""

    def __init__(self, gpu):
        import torch
        import handbrake_b200
        handbrake_b200.require_native()
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; this path has no CPU fallback (use --impl reference for the CPU arm)")
        self.torch = torch
        self.gpu = gpu
        torch.cuda.set_device(gpu)
        os.environ["HBCU_DEVICE"] = str(gpu)
        self.core = C.CDLL(str(handbrake_b200.LIBHBCU))
        self.core.hbcu_last_error.restype = C.c_char_p
        self.core.hbcu_kernel_launches.restype = C.c_uint64
        self.core.hbcu_host_reserve.argtypes = [C.c_size_t, C.c_int]
        self.flt = C.CDLL(str(handbrake_b200.LIBHBCU_FILTERS))
        bind_bench(self.flt)
        self.flt.hbcu_use_pinned_buffers(1)

    def ck(self, rc):
        if rc != 0:
            raise RuntimeError(self.core.hbcu_last_error().decode())

    def nlmeans_device_arm(self, wl, host, B, K, Wm, barrier=lambda: None, clock=None, dump_dir=None):
        """kernel-only arm: one continuous stream whose raw frames are already in HBM.  Frame t+nf-1 is bordered
        (upload_device) just before frame t is filtered, like the filter object does.  Returns (ms, kernel stats).
        With dump_dir, the outputs of the last step still held in the handle's output slots are written there."""
        torch, core, ck = self.torch, self.core, self.ck
        W, H, depth, nf = wl["width"], wl["height"], wl["depth"], wl["nframes"]
        bps = 2 if depth > 8 else 1
        dims = synth.plane_dims(W, H)
        fb = host.shape[1]
        n_dev = max(8, min(32, int(420e6 // fb) + 1))                    # distinct device frames: > L2 (126 MB) in total
        dev = [torch.from_numpy(host[i % host.shape[0]]).cuda() for i in range(n_dev)]
        ptrs = [plane_ptrs(t, dims, bps) for t in dev]
        out_slots = 4
        cfg = nlm_config(self.flt, wl, self.gpu, ring=nf + 6, out_slots=out_slots)
        h = C.c_void_p()
        ck(core.hbcu_nlmeans_create(C.byref(h), C.byref(cfg)))
        state = {"t": 0}
        for i in range(nf - 1):
            ck(core.hbcu_nlmeans_upload_device(h, C.c_int64(i), ptrs[i % n_dev][0], ptrs[i % n_dev][1]))
        outp, outs = (C.c_void_p * 3)(), (C.c_int * 3)()
        kept = {}           # frame -> (plane pointers, strides) of the step's last out_slots results, which no later frame overwrites

        def step():
            t0 = state["t"]
            kept.clear()
            for t in range(t0, t0 + B):
                u = t + nf - 1
                ck(core.hbcu_nlmeans_upload_device(h, C.c_int64(u), ptrs[u % n_dev][0], ptrs[u % n_dev][1]))
                ck(core.hbcu_nlmeans_filter_device(h, C.c_int64(t), nf, outp, outs))
                if t >= t0 + B - out_slots:
                    kept[t] = (list(outp), list(outs))
            state["t"] = t0 + B

        for _ in range(Wm):
            step()
        ck(core.hbcu_nlmeans_sync(h))
        barrier()
        if clock is not None:
            clock.start()
        launches0 = core.hbcu_kernel_launches()
        ck(core.hbcu_nlmeans_mark(h, 0))
        for _ in range(K):
            step()
        ck(core.hbcu_nlmeans_mark(h, 1))
        ms = C.c_float()
        ck(core.hbcu_nlmeans_elapsed_ms(h, C.byref(ms)))
        ck(core.hbcu_nlmeans_sync(h))
        launches = int(core.hbcu_kernel_launches() - launches0)
        barrier()
        kms, kcalls = C.c_float(), C.c_int()
        ck(core.hbcu_nlmeans_kernel_ms(h, C.byref(kms), C.byref(kcalls)))
        if dump_dir is not None:
            dump_outputs(dump_dir, [[device_plane(torch, p, s, pw, ph, bps) for p, s, (pw, ph) in zip(*kept[t], dims)] for t in sorted(kept)])
        core.hbcu_nlmeans_destroy(h)
        del dev
        torch.cuda.empty_cache()
        return float(ms.value), dict(launches=launches, kernel_ms=float(kms.value), kernel_calls=int(kcalls.value),
                                     input_mb=n_dev * fb / 1e6)

    def stream_arm(self, names, settings, fmt, W, H, flags, host, warm_frames, timed_frames, ring=48, barrier=lambda: None):
        """e2e arm: host hb_buffer_t frames through the filter object(s); one continuous stream, warm-up then timed"""
        flt = self.flt
        b = open_chain(flt, names, settings, fmt, W, H, flags)
        st = BenchStats()
        fb = host.shape[1]
        self.core.hbcu_host_reserve(fb + 4096, ring + 48)
        if os.environ.get("HBCU_BENCH_WC_INPUT", "0") == "1":
            # decoder-style inputs in write-combined pinned memory (the CPU only writes them, the GPU only reads them)
            self.core.hbcu_host_set_write_combined(1)
            rc = flt.hb_bench_prefill(b, host.ctypes.data, host.shape[0], ring)
            self.core.hbcu_host_set_write_combined(0)
            if rc != 0:
                raise RuntimeError("input ring prefill failed")
        if flt.hb_bench_stream(b, host.ctypes.data, host.shape[0], warm_frames, ring, C.byref(st)) != 0:
            raise RuntimeError("warm-up stream failed: " + self.core.hbcu_last_error().decode())
        barrier()
        if flt.hb_bench_stream(b, host.ctypes.data, host.shape[0], timed_frames, ring, C.byref(st)) != 0:
            raise RuntimeError("timed stream failed: " + self.core.hbcu_last_error().decode())
        res = dict(seconds=st.seconds, frames_in=timed_frames, frames_out=int(st.frames_out), bytes_in=int(st.bytes_in),
                   bytes_out=int(st.bytes_out), checksum=int(st.checksum), ring_misses=int(st.ring_misses))
        barrier()
        flt.hb_bench_finish(b, None)
        return res


def nlm_roofline(wl, workload, ms, ks, frames, clocks_mhz=None):
    peak, peak_src = measured_peaks()
    fb = synth.frame_bytes(fmt_of(wl["depth"]), wl["width"], wl["height"])
    alg = (wl["nframes"] + 1) * fb
    # consecutive frames are launched on two alternating compute streams, so two launches are normally in flight:
    # the per-launch figure is the average event-pair duration divided by the measured concurrency
    launch_ms = ks["kernel_ms"] / max(ks["kernel_calls"], 1)
    in_flight = max(1.0, launch_ms * frames / ms) if ms > 0 else 1.0
    kern_ms = launch_ms / in_flight
    achieved = alg / (kern_ms / 1e3) / 1e9 if ks["kernel_calls"] else None
    cap, cap_src = ncu_capture(workload, wl["depth"])
    r = {"bound": "hbm", "achieved": round(achieved, 1) if achieved else None, "peak": peak, "unit": "GB/s",
         "frac": round(achieved / peak, 4) if achieved else None,
         "traffic": int(cap["dram_bytes_total"]) if cap else None, "traffic_source": cap_src,
         "kernel": ("nlmeans_v3_kernel" if wl["depth"] == 8 else "nlmeans_v3w_kernel") +
                   " (all tiles of Y, U, V of one frame in one launch)",
         "kernel_ms_per_frame": round(kern_ms, 4), "launch_ms_avg": round(launch_ms, 4), "launches_in_flight": round(in_flight, 2),
         "launches_timed": ks["kernel_calls"], "algorithmic_bytes_per_frame": alg, "peak_source": peak_src,
         "note": "NLMeans is instruction-issue bound on B200, not HBM bound (DESIGN.md 4.1): frac is the honest HBM fraction, issue_frac the "
                 "fraction of the instruction-issue roofline (148 SMs x 4 warp-instructions per clock)"}
    if cap and cap.get("warp_instructions") and clocks_mhz:
        floor_ms = cap["warp_instructions"] / (148 * 4 * clocks_mhz * 1e6) * 1e3
        r["issue_frac"] = round(floor_ms / kern_ms, 4)
        r["issue_floor_ms"] = round(floor_ms, 4)
        r["warp_instructions_per_launch"] = int(cap["warp_instructions"])
    return r


def reference_stream(names, settings, fmt, W, H, flags, host, chunk, budget_s, min_chunks=2, max_chunks=64, warm_chunks=0):
    """the unmodified reference filter(s) (oracle/_ref/libhbref.so) on the host cores: ONE continuous stream fed in
    chunks (a chunk = one full taskset cycle of the multithreaded filters) until the time budget is used; the serial
    EOF flush happens once, after the clock"""
    if not REF_SO.exists():
        raise SystemExit(f"{REF_SO} missing: {REF_HOWTO}")
    ref = C.CDLL(str(REF_SO))
    bind_bench(ref)
    b = open_chain(ref, names, settings, fmt, W, H, flags)
    st = BenchStats()
    for _ in range(warm_chunks):
        if ref.hb_bench_stream(b, host.ctypes.data, host.shape[0], chunk, 0, C.byref(st)) != 0:
            raise RuntimeError("reference stream failed")
    secs, frames, times = 0.0, 0, []
    for c in range(max_chunks):
        if ref.hb_bench_stream(b, host.ctypes.data, host.shape[0], chunk, 0, C.byref(st)) != 0:
            raise RuntimeError("reference stream failed")
        secs += st.seconds
        frames += chunk
        times.append(round(st.seconds, 3))
        if c + 1 >= min_chunks and secs >= budget_s:
            break
    # no EOF flush: the reference flushes a partly filled taskset cycle SERIALLY (minutes at 4K / 8K) and the flush is not part
    # of the sample; the filters are closed with what they buffer, as a cancelled libhb job does
    if hasattr(ref, "hb_bench_abort"):
        ref.hb_bench_abort.argtypes = [C.c_void_p]
        ref.hb_bench_abort(b)
    else:
        ref.hb_bench_finish(b, None)
    return dict(fps=frames / secs, seconds=secs, frames=frames, chunks=len(times), chunk=chunk, chunk_seconds=times,
                ncpu=ref.hb_get_cpu_count())


def ref_threads(ncpu):
    return ncpu // 2 if ncpu >= 32 else (ncpu // 4) * 3 if ncpu >= 16 else ncpu     # nlmeans.c:362-373


def cpu_baseline_nlmeans(wl, budget_s, host=None):
    W, H, depth = wl["width"], wl["height"], wl["depth"]
    fmt = fmt_of(depth)
    if host is None:
        host = np.stack([synth.progressive_frame(fmt, W, H, t) for t in range(4)])
    ncpu = os.cpu_count() or 1
    threads = ref_threads(ncpu)
    r = reference_stream(["hb_filter_nlmeans"], [wl["settings"]], fmt, W, H, synth.PIC_FLAG_PROGRESSIVE_FRAME, host,
                         chunk=threads, budget_s=budget_s, min_chunks=3, warm_chunks=0)
    return r, {"value": round(r["fps"], 4), "unit": "frames/s", "cores": threads, "kind": "reference",
               "sample": f"{r['frames']} frames of {wl['desc']}: one continuous stream, {r['chunks']} taskset cycles of {threads} frames "
                         f"(the filter's own thread heuristic), no EOF flush, {r['seconds']:.1f} s",
               "host_logical_cpus": r["ncpu"],
               "what": "HandBrake libhb nlmeans.c + nlmeans_x86.c (SSE2) compiled unmodified, gcc -O3 -msse2"}


def eedi2_device_arm(ours, ex, host):
    """kernel-only arm of config 3's dominant filter: decomb EEDI2 bob on frames resident in HBM (both fields of every
    frame), algorithmic bytes 8 F per input frame (SURVEY.md 8d)"""
    torch, core, ck = ours.torch, ours.core, ours.ck
    W, H, depth = ex["width"], ex["height"], ex["depth"]
    fmt = fmt_of(depth); bps = 2 if depth > 8 else 1
    fb = synth.frame_bytes(fmt, W, H)
    mode = 31
    cfg = DecombConfig(W, H, depth, 1, 1, ours.gpu, 8, 8, mode, 10, 20, 20, 4, 2, 50, 24, 1)
    h = C.c_void_p(); ck(core.hbcu_decomb_create(C.byref(h), C.byref(cfg)))
    dims = synth.plane_dims(W, H)
    dev = [torch.from_numpy(host[i % host.shape[0]]).cuda() for i in range(8)]
    pp = [plane_ptrs(t, dims, bps) for t in dev]
    core.hbcu_decomb_upload_device.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    core.hbcu_decomb_filter_device.argtypes = [C.c_void_p] + [C.c_int64] * 4 + [C.c_int] * 3 + [C.c_void_p, C.c_void_p]

    def run(count, base):
        tk = base * 2
        for i in range(count):
            idx = base + i
            ck(core.hbcu_decomb_upload_device(h, idx, pp[idx % 8][0], pp[idx % 8][1]))
            if idx >= 2:
                for f in range(2):
                    ck(core.hbcu_decomb_filter_device(h, tk, idx - 2, idx - 1, idx, mode, f, 1, None, None)); tk += 1
    run(16, 0)
    n = 2200
    ck(core.hbcu_decomb_sync(h)); ck(core.hbcu_decomb_mark(h, 0))
    run(n, 16)
    ck(core.hbcu_decomb_mark(h, 1))
    ms = C.c_float(); ck(core.hbcu_decomb_elapsed_ms(h, C.byref(ms)))
    core.hbcu_decomb_destroy(h)
    del dev
    torch.cuda.empty_cache()
    peak, peak_src = measured_peaks()
    fps = n / (ms.value / 1e3)
    ach = 8 * fb * fps / 1e9
    cap = REPO / "profiles" / "r02_eedi2_dram.json"
    traffic = json.loads(cap.read_text()) if cap.exists() else None
    return {"value": round(fps, 2), "value_unit": "input frames/s (two EEDI2 fields each), every frame combed", "value_seconds": round(ms.value / 1e3, 3),
            "roofline": {"bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                         "traffic": traffic.get("dram_bytes_per_frame") if traffic else None,
                         "traffic_source": "profiles/r02_eedi2_dram.json" if traffic else None,
                         "algorithmic_bytes_per_frame": 8 * fb, "kernel": "decomb EEDI2 bob: stage kernels of both fields, one CUDA graph per field",
                         "peak_source": peak_src}}


def run_extra(ours, ex, budget_cpu_s, with_cpu=True):
    """one entry of `extra`: e2e through the filter objects (device-resident chain between upload and download
    adapters), the reference on the host cores (bounded sample), roofline"""
    W, H, depth = ex["width"], ex["height"], ex["depth"]
    fmt = fmt_of(depth)
    fb = synth.frame_bytes(fmt, W, H)
    nu = ex.get("n_unique", 5 if ex["interlaced"] else 4)
    if ex["interlaced"]:
        host = np.stack([synth.interlaced_frame(fmt, W, H, t, static=(t % 5 == 4)) for t in range(nu)])
        flags = synth.PIC_FLAG_TOP_FIELD_FIRST
    else:
        host = np.stack([synth.progressive_frame(fmt, W, H, t) for t in range(nu)])
        flags = synth.PIC_FLAG_PROGRESSIVE_FRAME
    cuda = [f"hb_filter_{x}_cuda" for x in ex["filters"]]
    if len(cuda) > 1:
        names, sets = ["hb_filter_hbcu_upload"] + cuda + ["hb_filter_hbcu_download"], [None] + ex["settings"] + [None]
    else:
        names, sets = cuda, ex["settings"]
    ring = 24 if fb > 60e6 else 48
    # a first pass of the clip's own length measures the rate (and warms pools / graphs); the timed pass then lasts >= ~2 s
    first = ours.stream_arm(names, sets, fmt, W, H, flags, host, min(ex["frames"], 32), ex["frames"], ring=ring)
    rate = ex["frames"] / first["seconds"]
    n = int(min(max(ex["frames"], rate * 2.2), 12000))
    r = ours.stream_arm(names, sets, fmt, W, H, flags, host, min(ex["frames"], 32), n, ring=ring)
    e2e = n / r["seconds"]
    peak, peak_src = measured_peaks()
    out = {"workload": ex["name"], "config": ex["config"], "desc": ex["desc"], "unit": "frames/s", "frames_timed": n,
           "clip_frames": ex["frames"], "first_pass_fps": round(rate, 2),
           "e2e": {"value": round(e2e, 2), "unit": "frames/s", "seconds": round(r["seconds"], 3), "h2d_bytes": r["bytes_in"],
                   "d2h_bytes": r["bytes_out"], "frames_out": r["frames_out"], "checksum": r["checksum"], "ring_misses": r["ring_misses"],
                   "path": " -> ".join(names)}}
    if ex.get("nlm_workload"):
        wl = WORKLOADS[ex["nlm_workload"]]
        B = max(16, min(512, int(rate * 0.25)))
        K = max(3, int(2.2 * rate * 1.2 / B) + 1)
        ms, ks = ours.nlmeans_device_arm(wl, host, B, K, 2)
        out["value"] = round(K * B / (ms / 1e3), 2)
        out["value_seconds"] = round(ms / 1e3, 3)
        out["roofline"] = nlm_roofline(wl, ex["nlm_workload"], ms, ks, K * B)
    elif ex["name"].startswith("cfg3"):
        out.update(eedi2_device_arm(ours, ex, host))
    else:
        ach = ex["alg_f"] * fb * e2e / 1e9
        out["value"] = None
        out["roofline"] = {"bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                           "traffic": None, "algorithmic_bytes_per_frame": int(ex["alg_f"] * fb), "peak_source": peak_src,
                           "basis": "end-to-end rate (host frames in and out; no kernel-only arm for a chain): " + ex.get("alg_note", "")}
    if with_cpu:
        refn = [f"hb_filter_{x}" + ("_mt" if x == "lapsharp" else "") for x in ex["filters"]]
        ncpu = os.cpu_count() or 1
        chunk = ref_threads(ncpu) if ex["filters"] == ["nlmeans"] else (4 if fb > 60e6 else 8)
        c = reference_stream(refn, ex["settings"], fmt, W, H, flags, host, chunk=chunk, budget_s=budget_cpu_s, min_chunks=1, max_chunks=40)
        out["cpu_baseline"] = {"value": round(c["fps"], 4), "unit": "frames/s", "kind": "reference", "cores": c["ncpu"],
                               "sample": f"{c['frames']} frames in {c['chunks']} chunks of {c['chunk']}, one continuous stream, {c['seconds']:.1f} s",
                               "path": " -> ".join(refn)}
    return out


def gather_arm(ours, dist, wl, host, rank, world, B, K, barrier, max_over_ranks):
    torch, core, ck = ours.torch, ours.core, ours.ck
    W, H, depth, nf = wl["width"], wl["height"], wl["depth"], wl["nframes"]
    bps = 2 if depth > 8 else 1
    dims = synth.plane_dims(W, H)
    fb = host.shape[1]
    nin = B + nf - 1
    cfg = nlm_config(ours.flt, wl, ours.gpu, ring=nin + 4, out_slots=4)
    h = C.c_void_p()
    ck(core.hbcu_nlmeans_create(C.byref(h), C.byref(cfg)))
    dev = [torch.from_numpy(host[i % host.shape[0]]).cuda() for i in range(nin)]
    ptrs = [plane_ptrs(t, dims, bps) for t in dev]
    core.hbcu_nlmeans_filter_into.argtypes = [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p]
    core.hbcu_nlmeans_stream_wait.argtypes = [C.c_void_p, C.c_void_p]
    block = torch.empty((B, fb), dtype=torch.uint8, device="cuda")            # this rank's finished block
    out_ptrs = [plane_ptrs(block[i], dims, bps) for i in range(B)]
    if rank == 0:
        recv = [torch.empty((B, fb), dtype=torch.uint8, device="cuda") for _ in range(world - 1)]
        host_out = torch.empty((world, B, fb), dtype=torch.uint8).pin_memory()
    idx = [0]

    def step_gather():
        base = idx[0]
        for i in range(nin):
            ck(core.hbcu_nlmeans_upload_device(h, C.c_int64(base + i), ptrs[i][0], ptrs[i][1]))
        for i in range(B):
            ck(core.hbcu_nlmeans_filter_into(h, base + i, nf, out_ptrs[i][0], out_ptrs[i][1]))
        idx[0] = base + nin
        ck(core.hbcu_nlmeans_stream_wait(h, C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        if rank == 0:
            host_out[0].copy_(block, non_blocking=True)
            for src in range(1, world):          # stream order = frame order: block of rank 1, then 2, ...
                dist.recv(recv[src - 1], src=src)
                host_out[src].copy_(recv[src - 1], non_blocking=True)
        else:
            dist.send(block, dst=0)

    for _ in range(2):
        step_gather()
    barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        step_gather()
    barrier()
    g_s = max_over_ranks(time.perf_counter() - t0)
    core.hbcu_nlmeans_destroy(h)
    return {"value": round(world * K * B / g_s, 2), "unit": "frames/s", "seconds": round(g_s, 3),
            "via": "ncclSend/ncclRecv (torch.distributed p2p over NVLink) of finished frames to rank 0, D2H on rank 0 only",
            "nvlink_bytes_per_step": int((world - 1) * B * fb), "d2h_bytes_per_step_rank0": int(world * B * fb)}


def run_ours(args, wl, rank, world, local_rank):
    gpu = pick_gpu(local_rank, world)
    numa_cpus = bind_to_gpu_numa_node(gpu) if world > 1 else None
    ours = Ours(gpu)
    torch = ours.torch
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", gpu))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    W, H, depth = wl["width"], wl["height"], wl["depth"]
    fmt = fmt_of(depth)
    B, K, Wm = args.batch, args.steps, args.warmup
    fb = synth.frame_bytes(fmt, W, H)
    n_unique = 4
    # every rank gets its own block of the clip (frame-sharded job): seeds differ per rank
    host = np.stack([synth.progressive_frame(fmt, W, H, rank * 1000 + t) for t in range(n_unique)])

    # ---------------- value: inputs resident in HBM ----------------
    clk = ClockSampler(gpu)
    dev_ms_local, ks = ours.nlmeans_device_arm(wl, host, B, K, Wm, barrier=barrier, clock=clk,
                                               dump_dir=args.dump_outputs if rank == 0 else None)
    dev_ms = max_over_ranks(dev_ms_local)
    value = world * K * B / (dev_ms / 1e3)

    # ---------------- e2e: host hb_buffer_t frames through the filter object ----------------
    settings = wl["settings"] + f":threads={args.inflight}"
    r = ours.stream_arm(["hb_filter_nlmeans_cuda"], [settings], fmt, W, H, synth.PIC_FLAG_PROGRESSIVE_FRAME, host,
                        Wm * B, K * B, ring=args.ring, barrier=barrier)
    clocks = clk.stop()
    e2e_s = max_over_ranks(r["seconds"])
    e2e = world * K * B / e2e_s
    pinned_numa = numa_of_pinned()

    # ---------------- copy_only: the same pipeline with every plane bypassed (the box's transfer ceiling at this N) ----------------
    copy_only = None
    if not args.no_copy_only:
        cw = dict(wl, settings="y-strength=0")
        nco = max(B, int(K * B * 0.4))
        rc = ours.stream_arm(["hb_filter_nlmeans_cuda"], [cw["settings"] + f":threads={args.inflight}"], fmt, W, H,
                             synth.PIC_FLAG_PROGRESSIVE_FRAME, host, min(Wm * B, 256), nco, ring=args.ring, barrier=barrier)
        co_s = max_over_ranks(rc["seconds"])
        co = world * nco / co_s
        copy_only = {"value": round(co, 2), "unit": "frames/s", "seconds": round(co_s, 3), "frames_per_gpu": nco,
                     "gb_s_per_gpu_per_direction": round(co / world * fb / 1e9, 2),
                     "e2e_over_copy_only": round(e2e / co, 4),
                     "what": "hb_filter_nlmeans_cuda with strength 0 on every plane: H2D, a device copy, D2H -- the transfer pipeline alone"}

    # ---------------- ordered gather to the muxer rank over NCCL p2p (north-star; only for N > 1) ----------------
    gather = None
    if world > 1 and not args.no_gather:
        gather = gather_arm(ours, dist, wl, host, rank, world, min(B, 64), max(2, min(K, 6)), barrier, max_over_ranks)

    # ---------------- the plugin's own multi-device path: ONE process, ONE ordered stream dealt to all N GPUs in C ----------------
    # (what a libhb job -- one process, one thread per filter, work.c:2255-2270 -- does with `devices=`; the ranks above
    # each filter a private stream.)  A child process of rank 0 drives every GPU of the job while all ranks wait at the
    # barrier; a child, so that a fault in this side arm can neither hang nor take down the headline line.
    plugin_multi = None
    if world > 1 and not args.no_plugin_multi:
        barrier()
        # the other ranks must wait on the CPU: an NCCL barrier is a kernel spinning on their GPUs, which the child is about to use
        # (measured: 4909 frames/s on 2 GPUs with the ranks parked in dist.barrier(), 7776 with idle GPUs)
        store = dist.distributed_c10d._get_default_store()
        if rank == 0:
            devs = [pick_gpu(r_, world) for r_ in range(world)]
            nfr = world * max(B // 2, int(K * B * 0.25))
            env = {k: v for k, v in os.environ.items() if k not in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT",
                                                                      "TORCHELASTIC_RUN_ID", "GROUP_RANK", "ROLE_RANK", "HBCU_DEVICE")}
            cmd = [sys.executable, str(Path(__file__).resolve()), "--plugin-multi-child", ",".join(map(str, devs)), "--workload", args.workload,
                   "--plugin-frames", str(nfr), "--plugin-warm", str(min(Wm * B, 128 * world)), "--block", str(args.block), "--inflight", str(args.inflight)]
            try:
                cp = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env)
                line = [l for l in cp.stdout.splitlines() if l.startswith("{")]
                plugin_multi = json.loads(line[-1]) if line else {"error": (cp.stderr or "no output")[-400:], "devices": devs}
            except Exception as e:
                plugin_multi = {"error": f"{type(e).__name__}: {e}", "devices": devs}
            store.set("hbcu_plugin_multi_done", "1")
        else:
            import datetime
            try:
                store.wait(["hbcu_plugin_multi_done"], datetime.timedelta(seconds=420))
            except Exception:
                pass
        barrier()

    out = {
        "metric": "4K NLMeans frames/sec" if W == 3840 else "NLMeans frames/sec",
        "value": round(value, 2), "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": round(dev_ms / K, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8" if depth == 8 else "u16", "data": "synthetic",
        "config": {"workload": args.workload, "desc": wl["desc"], "frames_per_step_per_gpu": B,
                   "sharding": f"frame blocks x{world}, {wl['nframes'] - 1}-frame temporal halo per block, no data-path collective",
                   "gpu_of_rank0": gpu, "cpu_affinity": numa_cpus,
                   "l2": f"inputs cycle through {ks['input_mb']:.0f} MB of distinct device frames > 126 MB L2",
                   "timed_seconds": {"value": round(dev_ms / 1e3, 3), "e2e": round(e2e_s, 3)}},
        "e2e": {"value": round(e2e, 2), "unit": "frames/s", "h2d_bytes_per_step": int(world * r["bytes_in"] // K),
                "d2h_bytes_per_step": int(world * r["bytes_out"] // K), "seconds": round(e2e_s, 4), "checksum": r["checksum"],
                "input_ring": args.ring, "ring_misses": r["ring_misses"], "pinned_numa": pinned_numa},
        "gpu_launches": ks["launches"],
        "clocks": clocks,
        "roofline": nlm_roofline(wl, args.workload, dev_ms_local, ks, K * B, clocks.get("sm_mhz")),
    }
    if copy_only is not None:
        out["copy_only"] = copy_only
    if gather is not None:
        out["gather"] = gather
    if plugin_multi is not None:
        out["plugin_multi_device"] = plugin_multi
    if world == 1 and not args.no_cpu_baseline:
        if REF_SO.exists():
            _, out["cpu_baseline"] = cpu_baseline_nlmeans(wl, budget_s=12.0)
        else:
            out["cpu_baseline"] = {"value": None, "note": f"not measured: {REF_SO.relative_to(REPO)} is not built ({REF_HOWTO})"}
    if world == 1 and not args.no_extra:
        extra = []
        for ex in EXTRAS:
            if args.only_extra and args.only_extra not in ex["name"]:
                continue
            try:
                extra.append(run_extra(ours, ex, budget_cpu_s=8.0, with_cpu=not args.no_cpu_baseline and REF_SO.exists()))
            except Exception as e:  # an extra must never take the headline line down with it
                extra.append({"workload": ex["name"], "error": f"{type(e).__name__}: {e}"})
        out["extra"] = extra
    if world > 1:
        dist.destroy_process_group()
    return out


def run_reference(args, wl, rank, world):
    if rank != 0:
        return None
    W, H, depth = wl["width"], wl["height"], wl["depth"]
    fmt = fmt_of(depth)
    host = np.stack([synth.progressive_frame(fmt, W, H, t) for t in range(4)])
    ncpu = os.cpu_count() or 1
    threads = ref_threads(ncpu)
    # one step = one full taskset cycle (`threads` frames in parallel) of ONE continuous stream: no step pays the
    # serial EOF flush or thread creation (they happen once, outside the clock)
    r = reference_stream(["hb_filter_nlmeans"], [wl["settings"]], fmt, W, H, synth.PIC_FLAG_PROGRESSIVE_FRAME, host,
                         chunk=threads, budget_s=1e9, min_chunks=args.steps, max_chunks=args.steps, warm_chunks=args.warmup)
    sample = f"{args.steps} steps of {threads} frames (one parallel taskset cycle each) of one continuous stream of {wl['desc']}"
    return {
        "impl": "reference",
        "metric": "4K NLMeans frames/sec" if W == 3840 else "NLMeans frames/sec",
        "value": round(r["fps"], 4), "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(1e3 * r["seconds"] / args.steps, 2), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8" if depth == 8 else "u16", "data": "synthetic",
        "config": {"workload": args.workload, "desc": wl["desc"], "frames_per_step": threads},
        "cpu_baseline": {"value": round(r["fps"], 4), "unit": "frames/s", "cores": threads, "kind": "reference", "sample": sample,
                         "host_logical_cpus": r["ncpu"],
                         "what": "HandBrake libhb nlmeans.c + nlmeans_x86.c (SSE2) compiled unmodified, gcc -O3 -msse2, its own thread heuristic"},
        "e2e": {"value": round(r["fps"], 4), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }


def plugin_multi_child(args, wl):
    """one process, one ordered stream through hb_filter_nlmeans_cuda.work() with devices=<list> (see run_ours)"""
    devs = [int(x) for x in args.plugin_multi_child.split(",")]
    # one process feeds GPUs on both sockets: undo the per-rank NUMA binding inherited from rank 0 and interleave this
    # process's pages (the pinned frame pool among them) over all nodes
    policy = "default"
    try:
        os.sched_setaffinity(0, range(os.cpu_count() or 1))
        nodes = sorted(int(m.group(1)) for m in (re.match(r"node(\d+)$", n) for n in os.listdir("/sys/devices/system/node")) if m)
        if len(nodes) > 1 and os.environ.get("HBCU_BENCH_NO_INTERLEAVE", "0") != "1":
            libc = C.CDLL(None, use_errno=True)
            mask = C.c_ulong(sum(1 << n for n in nodes))
            if libc.syscall(238, 3, C.byref(mask), C.c_ulong(max(nodes) + 2)) == 0:          # set_mempolicy(MPOL_INTERLEAVE)
                policy = f"interleave over nodes {nodes}"
            else:
                policy = f"set_mempolicy failed (errno {C.get_errno()})"
    except Exception as e:
        policy = f"default ({type(e).__name__})"
    ours = Ours(devs[0])
    os.environ.pop("HBCU_DEVICE", None)
    W, H, depth = wl["width"], wl["height"], wl["depth"]
    fmt = fmt_of(depth)
    host = np.stack([synth.progressive_frame(fmt, W, H, t) for t in range(4)])
    settings = wl["settings"] + f":threads={args.inflight}:devices={args.plugin_multi_child}:block={args.block}"
    rm = ours.stream_arm(["hb_filter_nlmeans_cuda"], [settings], fmt, W, H, synth.PIC_FLAG_PROGRESSIVE_FRAME, host,
                         args.plugin_warm, args.plugin_frames, ring=min(256, 48 + 16 * len(devs)))
    fb = synth.frame_bytes(fmt, W, H)
    print(json.dumps({"value": round(args.plugin_frames / rm["seconds"], 2), "unit": "frames/s", "seconds": round(rm["seconds"], 3),
                      "frames": args.plugin_frames, "devices": devs, "block": args.block, "ring_misses": rm["ring_misses"], "checksum": rm["checksum"],
                      "gb_s_per_direction_total": round(args.plugin_frames / rm["seconds"] * fb / 1e9, 1), "pinned_numa": numa_of_pinned(),
                      "mempolicy": policy,
                      "what": "one process, one ordered stream of host hb_buffer_t frames through hb_filter_nlmeans_cuda.work() with "
                              "devices=<all GPUs>: block-cyclic dealing in C (nlmeans_cuda.c), one submission thread per device, look-ahead "
                              "halo by NVLink peer copy (hbcu_nlmeans_upload_peer), outputs harvested in stream order; H2D + kernels + D2H "
                              "inside the clock"}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="4k_nlmeans_strong", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=768, help="frames per step per GPU")
    ap.add_argument("--ring", type=int, default=48, help="pinned input payloads the e2e stream cycles through")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true")
    ap.add_argument("--only-extra", default="", help="substring of the one extra entry to run")
    ap.add_argument("--no-copy-only", action="store_true")
    ap.add_argument("--no-gather", action="store_true")
    ap.add_argument("--no-plugin-multi", action="store_true")
    ap.add_argument("--plugin-multi-child", default="", help=argparse.SUPPRESS)
    ap.add_argument("--plugin-frames", type=int, default=2048, help=argparse.SUPPRESS)
    ap.add_argument("--plugin-warm", type=int, default=256, help=argparse.SUPPRESS)
    ap.add_argument("--block", type=int, default=8, help="frames per device turn of the plugin's multi-device dealing")
    ap.add_argument("--inflight", type=int, default=6, help="frames in flight in the e2e arm (the filter's `threads` setting)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the Y/U/V output planes of the last step's final frames (the frames the "
                         "kernel-only arm still holds) to DIR/{y,u,v}.npy as float32; a fixed sample of positions when larger than 64 MB")
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3                     # timing rule: at least three warm-up steps
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = WORKLOADS[args.workload]
    if args.plugin_multi_child:
        plugin_multi_child(args, wl)
        return
    if args.impl == "reference":
        out = run_reference(args, wl, rank, world)
    else:
        out = run_ours(args, wl, rank, world, local_rank)
    if rank == 0 and out is not None:
        print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
