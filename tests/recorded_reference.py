"""The original project's CPU models as recorded answers: a stand-in for CpuChecker("reference").

The tests that pin the port oracle to the original project's own sources compare, call by call, what both return for
the same inputs.  Those sources are not part of this repository, so their answers are kept in
tests/golden/reference_calls.npz: every call is looked up by a digest of its name and arguments, and returns what the
reference build returned for exactly those arguments.  A call that was never recorded (a test's inputs changed) fails
loudly; re-record with `python tests/golden/make_golden.py --calls` where the original sources are available.
"""
import ctypes as C
import hashlib
import io
import lzma
import os

import numpy as np

from oracle import cpu_checker as cc

CALLS = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_calls.npz")


def _feed(h, a):
    if isinstance(a, (list, tuple)):
        h.update(b"[%d" % len(a))
        for x in a:
            _feed(h, x)
        h.update(b"]")
    elif isinstance(a, (np.ndarray, np.void)):
        a = np.ascontiguousarray(a)
        h.update(("A%s%s" % (a.dtype.descr, a.shape)).encode())
        h.update(a.tobytes())
    elif isinstance(a, C.Structure):
        h.update(b"S" + type(a).__name__.encode() + bytes(a))
    else:
        h.update(("V" + repr(a)).encode())


def digest(owner, name, args, kwargs):
    h = hashlib.sha1((owner + "." + name).encode())
    _feed(h, list(args) + sorted(kwargs.items()))
    return h.hexdigest()


def _encode(value):
    """-> [(tag, array)]: a result as arrays that decode back to the same Python types."""
    if isinstance(value, tuple):
        return [(t + str(i), a) for i, v in enumerate(value) for t, a in _encode(v)]
    if isinstance(value, cc.BeamParams):
        return [("s", np.frombuffer(bytes(value), np.uint8))]
    if isinstance(value, (bool, np.bool_)):
        return [("b", np.array(value))]
    if isinstance(value, (int, np.integer)):
        return [("i", np.array(value, np.int64))]
    if isinstance(value, (float, np.floating)):
        return [("f", np.array(value, np.float64))]
    return [("a", np.asarray(value))]


def _decode(tag, a):
    return {"s": lambda: cc.BeamParams.from_buffer_copy(a.tobytes()), "b": lambda: bool(a), "i": lambda: int(a),
            "f": lambda: float(a), "a": lambda: a}[tag]()


class _Recorded:
    """Methods named in METHODS answer from the recording (replay) or from `live`, recording as they go."""
    METHODS = ()

    def __init__(self, store, key, live=None):
        self._store, self._key, self._live = store, key, live

    def _call(self, name, args, kwargs):
        d = digest(self._key, name, args, kwargs)
        if self._live is not None:
            out = getattr(self._live, name)(*args, **kwargs)
            if name != "create":
                self._store.record(d, out)
            return d, out
        return d, (None if name == "create" else self._store.replay(d, name))

    def __getattr__(self, name):
        if name not in self.METHODS:
            raise AttributeError(name)
        return lambda *args, **kwargs: self._call(name, args, kwargs)[1]


class RecordedMap(_Recorded):
    METHODS = ("measure", "beam_status", "beam_params", "radius_search")

    def close(self):
        if self._live is not None:
            self._live.close()


class RecordedReference(_Recorded):
    METHODS = ("dda_walk", "kd_walk", "filter_clip", "global_localization_points", "motion_predict", "pf_resample_1d",
               "pf_resample_6dof", "pf_estimate")
    kind = "reference"

    def create(self, *args, **kwargs):
        d, live_map = self._call("create", args, kwargs)
        return RecordedMap(self._store, d, live_map)


class CallStore:
    def __init__(self, path=CALLS):
        self.path = path
        self.entries = {}

    def load(self):
        with np.load(self.path) as z:
            index, blob = z["index"], lzma.decompress(z["blob"].tobytes())
        for d, tag, off, n in index:
            part = np.load(io.BytesIO(blob[off:off + n]))
            self.entries.setdefault(d.decode(), []).append((tag.decode(), part))
        return self

    def record(self, d, out):
        self.entries[d] = _encode(out)

    def replay(self, d, name):
        if d not in self.entries:
            raise KeyError("no recorded reference answer for this %s call: its inputs differ from the recorded ones "
                           "(re-record with tests/golden/make_golden.py --calls)" % name)
        parts = self.entries[d]
        if len(parts) == 1 and len(parts[0][0]) == 1:
            return _decode(*parts[0])
        return tuple(_decode(tag[0], a) for tag, a in sorted(parts, key=lambda p: int(p[0][1:])))

    def save(self):
        """One index and one xz-compressed blob of .npy images: a member per answer would cost more than the answers."""
        index, chunks, off = [], [], 0
        for d, parts in sorted(self.entries.items()):
            for tag, a in parts:
                f = io.BytesIO()
                np.save(f, a)
                chunks.append(f.getvalue())
                index.append((d, tag, off, len(chunks[-1])))
                off += len(chunks[-1])
        index = np.array(index, dtype=[("digest", "S40"), ("tag", "S4"), ("off", "<i8"), ("len", "<i8")])
        blob = lzma.compress(b"".join(chunks), preset=9 | lzma.PRESET_EXTREME)
        np.savez_compressed(self.path, index=index, blob=np.frombuffer(blob, np.uint8))


def replaying():
    return RecordedReference(CallStore().load(), "reference")


def recording(live):
    store = CallStore()
    return RecordedReference(store, "reference", live), store
