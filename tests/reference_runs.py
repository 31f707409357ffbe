"""The reference's filters as the tests see them: stored runs of the compiled reference (oracle/_ref/libhbref.so).

The reference is HandBrake's own libhb sources compiled unmodified; a checkout of this project does not carry them, so
what the reference computed for each call a test makes is stored in tests/golden/reference_runs.json.gz: per output
frame a digest of its bytes, and in full the per-frame metadata (timestamps, flags, comb verdicts, frame rate).  A call
is looked up by a digest of everything that goes into it (filter names, settings, input frames, flags, tags, format,
size, CPU count).  A digest here is the first 16 hex digits (64 bits) of a SHA-256, which keeps the file small enough to
commit; the file is gzipped JSON, one entry per line.  A call the file does not know fails the test.  The stored runs
are regenerated with the reference built (`make -C oracle ref REF=<HandBrake tree>`) by running the suite with

    HBCU_RECORD_REFERENCE=<output .json.gz> python -m pytest tests

which runs every call on the reference library and writes the stored runs plus everything it ran to that file.

Output frames come back as `RecordedFrames`: a stack of digests that np.array_equal and np.concatenate accept in place
of the frames, which is all the tests do with the reference's pictures.
"""
import ctypes as C
import gzip
import hashlib
import json
from pathlib import Path

import numpy as np

STORE = Path(__file__).resolve().parent / "golden" / "reference_runs.json.gz"
DIGEST_HEX = 16


def short_digest(a):
    """first DIGEST_HEX hex digits of the SHA-256 of an array's bytes"""
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:DIGEST_HEX]


class RecordedFrames:
    """Frames known by their short digests: shape (n, frame_bytes), or (frame_bytes,) for one frame taken out."""

    def __init__(self, digests, frame_bytes, single=False):
        self.digests = list(digests)
        self.frame_bytes = frame_bytes
        self.single = single
        self.shape = (frame_bytes,) if single else (len(self.digests), frame_bytes)
        self.ndim = len(self.shape)

    def __len__(self):
        return self.shape[0]

    def __getitem__(self, i):
        if self.single:
            raise TypeError("a recorded frame is known by its digest only")
        if isinstance(i, slice):
            return RecordedFrames(self.digests[i], self.frame_bytes)
        return RecordedFrames([self.digests[i]], self.frame_bytes, single=True)

    def __iter__(self):
        return (self[i] for i in range(len(self)))

    def __repr__(self):
        return f"RecordedFrames(shape={self.shape})"

    def __array_function__(self, func, types, args, kwargs):
        if func is np.array_equal and not kwargs:
            return _equal(*args)
        if func is np.concatenate and not kwargs and len(args) == 1:
            parts = list(args[0])
            if all(isinstance(p, RecordedFrames) and not p.single for p in parts) and len({p.frame_bytes for p in parts}) == 1:
                return RecordedFrames([d for p in parts for d in p.digests], parts[0].frame_bytes)
        return NotImplemented


def frame_digests(frames):
    """per-frame short digests of real (n, frame_bytes) uint8 frames or of RecordedFrames"""
    if isinstance(frames, RecordedFrames):
        return [frames.digests[0]] if frames.single else list(frames.digests)
    a = np.asarray(frames)
    if a.dtype != np.uint8:
        raise TypeError(f"frames are uint8, not {a.dtype}")
    return [short_digest(a)] if a.ndim == 1 else [short_digest(f) for f in a]


def _equal(a, b):
    if tuple(a.shape) != tuple(b.shape):
        return False
    return frame_digests(a) == frame_digests(b)


def differing_frames(a, b):
    """indices of the frames in which two equally long stacks (real or recorded) differ"""
    return [i for i, (x, y) in enumerate(zip(frame_digests(a), frame_digests(b))) if x != y]


class ReferenceResult:
    """hblib.FilterResult of a stored reference run"""

    def __init__(self, rec):
        self.frames = RecordedFrames(rec["frames"], rec["frame_bytes"])
        self.combed = np.array(rec["combed"], np.uint8)
        self.flags = np.array(rec["flags"], np.uint16)
        self.start = np.array(rec["start"], np.int64)
        self.stop = np.array(rec["stop"], np.int64)
        self.duration = np.array(rec["duration"], np.float64)
        self.saw_eof = bool(rec["saw_eof"])
        self.init_failed = rec["init_failed"]
        self.vrate = tuple(rec["vrate"])
        self.n_dropped = rec["n_dropped"]


def _key(parts):
    return hashlib.sha256(json.dumps(parts).encode()).hexdigest()[:24]


def _opt_digest(a, dtype):
    return None if a is None else short_digest(np.ascontiguousarray(a, dtype=dtype))


class ReferenceRuns:
    """The reference's filter library as the tests use it (run, buffers_alive, set_cpu_count), plus its settings
    templates and direct calls of its exported functions.  `lib` is the compiled reference (hblib.FilterLib) while
    recording, None when replaying the stored runs."""

    def __init__(self, store, lib=None):
        self.store = store
        self.lib = lib
        self.cpu_count = 0
        self.alive = 0

    @classmethod
    def load(cls, lib=None, path=STORE):
        store = json.loads(gzip.decompress(path.read_bytes())) if path.exists() else {}
        for section in ("runs", "templates", "calls"):
            store.setdefault(section, {})
        return cls(store, lib)

    def save(self, path):
        """one entry per line, so that a regenerated file diffs entry by entry"""
        lines = []
        for section in ("runs", "templates", "calls"):
            entries = [f"  {json.dumps(k)}: {json.dumps(v, separators=(',', ':'))}" for k, v in sorted(self.store[section].items())]
            lines.append(f" {json.dumps(section)}: {{\n" + ",\n".join(entries) + "\n }")
        Path(path).write_bytes(gzip.compress(("{\n" + ",\n".join(lines) + "\n}\n").encode(), mtime=0))

    def _lookup(self, section, key, what):
        try:
            return self.store[section][key]
        except KeyError:
            raise LookupError(f"no stored reference result for {what}: regenerate {STORE.name} (see {Path(__file__).name})") from None

    def set_cpu_count(self, n):
        self.cpu_count = int(n)
        if self.lib is not None:
            self.lib.set_cpu_count(n)

    def buffers_alive(self):
        """hb_buffer_t objects the reference left alive after the last run"""
        return self.alive

    def run(self, filters, settings, frames, pix_fmt, width, height, flags=None, combed=None, max_out=None, out_scale=1,
            columns=None):
        """hblib.FilterLib.run; `columns` (a slice of the frame bytes) keeps only those bytes of every output frame"""
        if isinstance(filters, str):
            filters, settings = [filters], [settings]
        frames = np.ascontiguousarray(frames, dtype=np.uint8)
        cols = None if columns is None else [columns.start, columns.stop]
        key = _key([list(filters), list(settings), pix_fmt, width, height, list(frames.shape), short_digest(frames),
                    _opt_digest(flags, np.uint16), _opt_digest(combed, np.uint8), max_out, out_scale, self.cpu_count, cols])
        what = f"{filters} {settings} on {frames.shape[0]} frames {width}x{height}"
        if self.lib is not None:
            try:
                r = self.lib.run(filters, settings, frames, pix_fmt, width, height, flags=flags, combed=combed,
                                 max_out=max_out, out_scale=out_scale)
                out = r.frames if columns is None else r.frames[:, columns]
                rec = dict(frames=frame_digests(out), frame_bytes=int(out.shape[1]),
                           combed=r.combed.tolist(), flags=r.flags.tolist(), start=r.start.tolist(), stop=r.stop.tolist(),
                           duration=r.duration.tolist(), saw_eof=int(r.saw_eof), init_failed=int(r.init_failed),
                           vrate=list(r.vrate), n_dropped=int(r.n_dropped), buffers_alive=self.lib.buffers_alive())
            except RuntimeError as e:
                rec = dict(error=str(e))
            self.store["runs"][key] = rec
        rec = self._lookup("runs", key, what)
        if "error" in rec:
            raise RuntimeError(rec["error"])
        self.alive = rec["buffers_alive"]
        return ReferenceResult(rec)

    def settings_template(self, name):
        """settings_template string of the reference's filter object `name`"""
        if self.lib is not None:
            class Head(C.Structure):       # head of hb_filter_object_t up to settings_template (handbrake/common.h)
                _fields_ = [("pad", C.c_byte * 96), ("settings_template", C.c_char_p)]
            self.store["templates"][name] = Head.in_dll(self.lib.lib, name).settings_template.decode()
        return self._lookup("templates", name, name).encode()

    def call(self, symbol, *args):
        """Calls the reference's exported C function `symbol` on copies of the numpy arrays among `args` (an array
        passed twice is one buffer, passed twice) and ints; returns the short digests of those arrays afterwards, in
        order of first appearance."""
        arrays = []
        for a in args:
            if isinstance(a, np.ndarray) and not any(a is b for b in arrays):
                arrays.append(a)
        idx = [next(i for i, b in enumerate(arrays) if b is a) if isinstance(a, np.ndarray) else None for a in args]
        key = _key([symbol] + [[i, arrays[i].dtype.str, list(arrays[i].shape), short_digest(arrays[i])] if i is not None else int(a)
                               for a, i in zip(args, idx)])
        if self.lib is not None:
            copies = [np.ascontiguousarray(a).copy() for a in arrays]
            getattr(self.lib.lib, symbol)(*[C.c_void_p(copies[i].ctypes.data) if i is not None else C.c_int(int(a)) for a, i in zip(args, idx)])
            self.store["calls"][key] = [short_digest(c) for c in copies]
        return self._lookup("calls", key, symbol)
