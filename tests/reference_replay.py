"""What the unmodified reference (oracle/_ref/libocvref.so) returned to the CPU tests, kept in the repository.

The CPU tests compare the plain-C port, the product's host tables and the emulated kernels with the reference.  The reference library
can only be built where the reference's sources are, so the `ref` fixture records every call a test makes (`pytest --record-reference`)
into tests/golden/reference_calls.npz, and replays it where the library is absent.

The port (or a function the test names with with_twin) computes the same calls, so a recording stays small.  Every call keeps one 64-bit
check: a digest of the call's name, its inputs and the port's result, recorded when the port's result was the reference's bytes.  Where
the two differ (float paths the tests hold to a tolerance) the recording also keeps the difference of their bit patterns, and the replay
rebuilds the reference's exact bytes from the port's result.  Calls the port cannot answer keep the reference's whole result.  So the
replay answers a call only if the test asked the same question and the port still computes what it did when recorded; otherwise the
test fails, it never compares against a wrong answer.
"""
import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_calls.npz")

LAB_CODES = (32, 33, 34, 35, 44, 45, 56, 57, 74, 75, 78, 79)     # the port answers these through cvtColorLab


class ReplayMismatch(AssertionError):
    pass


def _digest_update(h, x):
    if isinstance(x, np.ndarray):
        h.update(b"A%s%r" % (x.dtype.str.encode(), x.shape))
        h.update(np.ascontiguousarray(x).tobytes())
    elif isinstance(x, (list, tuple)):
        h.update(b"L%d" % len(x))
        for v in x:
            _digest_update(h, v)
    elif isinstance(x, dict):
        _digest_update(h, sorted(x.items()))
    else:
        h.update(repr(x).encode())


def digest(x):
    h = hashlib.blake2b(digest_size=8)
    _digest_update(h, x)
    return int.from_bytes(h.digest(), "little")


def _flatten(x):
    """(leaves, tree): arrays and scalars as leaves, tuples / lists as structure"""
    if isinstance(x, (list, tuple)):
        leaves, trees = [], []
        for v in x:
            lv, t = _flatten(v)
            leaves += lv
            trees.append(t)
        return leaves, ["t" if isinstance(x, tuple) else "l", trees]
    if x is None:
        return [], "n"
    return [x], "a" if isinstance(x, np.ndarray) else "s"


def _unflatten(tree, leaves):
    it = iter(leaves)

    def go(t):
        if t == "n":
            return None
        if t == "a":
            return next(it)
        if t == "s":
            return next(it).item()
        items = [go(c) for c in t[1]]
        return tuple(items) if t[0] == "t" else items
    return go(tree)


def _bits(a):
    """the array's bit pattern as signed integers wide enough to hold the difference of two patterns"""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        return a.view({2: np.int16, 4: np.int32, 8: np.int64}[a.dtype.itemsize]).astype(np.int64)
    return a.astype(np.int64)


def _from_bits(b, like):
    if like.dtype.kind == "f":
        it = {2: np.int16, 4: np.int32, 8: np.int64}[like.dtype.itemsize]
        return b.astype(it).view(like.dtype).reshape(like.shape)
    return b.astype(like.dtype).reshape(like.shape)


def _port_answer(port, name, args, kwargs):
    """the port's answer to the same call, or None when the port has no such entry"""
    if name == "cvtColor" and len(args) >= 2 and int(args[1]) in LAB_CODES and args[0].dtype == np.uint8:
        name, args = "cvtColorLab", args[:2]
    try:
        return getattr(port, name)(*args, **kwargs)
    except (AttributeError, RuntimeError, KeyError, TypeError, ValueError):
        return None


def with_twin(ref, **twins):
    """Answer the named reference calls with the given functions (the code under test, say) when recording and replaying, instead of
    with the port: the recording then needs only digests.  The real reference is returned unchanged."""
    if isinstance(ref, (Recorder, Replay)):
        ref._twins.update(twins)
    return ref


class _Stand:
    def __init__(self, port, test_id):
        self._port, self._test, self._twins = port, test_id, {}

    def _twin(self, name, args, kwargs):
        if name in self._twins:
            return self._twins[name](*args, **kwargs)
        return _port_answer(self._port, name, args, kwargs)


def _check(name, args, kwargs, twin_digests):
    return digest([name, digest([args, kwargs]), twin_digests])


class Recorder(_Stand):
    """wraps the real reference: answers every call from it and notes what the replay needs"""

    def __init__(self, real, port, store, test_id):
        super().__init__(port, test_id)
        self._real, self._calls = real, store.setdefault(test_id, [])
        self._calls.clear()
        self.kind = real.kind

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        fn = getattr(self._real, name)

        def call(*args, **kwargs):
            out = fn(*args, **kwargs)
            leaves, tree = _flatten(out)
            twin = self._twin(name, args, kwargs)
            tl = None
            if twin is not None:
                tl, ttree = _flatten(twin)
                if ttree != tree or any(np.shape(a) != np.shape(b) or np.asarray(a).dtype != np.asarray(b).dtype for a, b in zip(tl, leaves)):
                    tl = None
            rec = {"tree": tree if tl is None else None, "payload": []}
            twin_digests = []
            for i, leaf in enumerate(leaves):
                leaf = np.asarray(leaf)
                if tl is None:
                    rec["payload"].append((i, "full", leaf.copy()))
                    continue
                t = np.asarray(tl[i])
                twin_digests.append(digest(t))
                if twin_digests[-1] != digest(leaf):
                    rec["payload"].append((i, "delta", (_bits(leaf) - _bits(t)).reshape(-1)))
            rec["check"] = _check(name, args, kwargs, twin_digests)
            self._calls.append(rec)
            return out
        return call


def _narrow(a):
    """most differences are a few units in the last place, and many float results hold small integers: the narrowest integer type that
    holds the values exactly (a negative zero keeps its float type)"""
    if a.size and (a.dtype.kind in "iub" or (a.dtype.kind == "f" and np.isfinite(a).all() and np.array_equal(a, np.round(a))
                                             and not np.signbit(a[a == 0]).any())):
        lo, hi = int(a.min()), int(a.max())
        for t in (np.int8, np.uint8, np.int16, np.uint16, np.int32, np.int64):
            if np.iinfo(t).min <= lo and hi <= np.iinfo(t).max:
                return a.astype(t)
    return a


def save(store, path=GOLDEN):
    """one compressed archive: a 64-bit check per call, a small JSON index of the calls that keep arrays, and those arrays"""
    tests, checks, kept, payload, seen = [], [], {}, {}, {}
    for test_id, calls in sorted(store.items()):
        tests.append([test_id, len(checks), len(calls)])
        for n, rec in enumerate(calls):
            checks.append(rec["check"])
            if rec["payload"]:
                outs = []
                for i, kind, a in rec["payload"]:
                    dtype = a.dtype.str
                    a = _narrow(a)
                    key = seen.setdefault((digest(a), a.dtype.str), "p%d" % len(seen))
                    payload[key] = a
                    outs.append([i, kind, key, dtype])
                kept["%s#%d" % (test_id, n)] = {"tree": rec["tree"], "outs": outs}
    meta = json.dumps({"tests": tests, "kept": kept}, separators=(",", ":")).encode()
    np.savez_compressed(path, meta=np.frombuffer(meta, np.uint8), checks=np.array(checks, np.uint64), **payload)


class Replay(_Stand):
    """stands in for the reference in one test: the recorded answers, checked against the port (or the test's twin) as described above"""
    kind = "ref"

    def __init__(self, archive, test, port, test_id):
        super().__init__(port, test_id)
        self._z, self._checks, (self._first, self._count), self._kept = archive["z"], archive["checks"], test, archive["kept"]
        self._n = 0

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)

        def call(*args, **kwargs):
            where = "%s, reference call %d (%s)" % (self._test, self._n, name)
            if self._n >= self._count:
                raise ReplayMismatch(where + ": not in the recording; record again with --record-reference")
            kept = self._kept.get("%s#%d" % (self._test, self._n), {"tree": None, "outs": []})
            want = int(self._checks[self._first + self._n])
            self._n += 1
            full = {i: (key, dtype) for i, kind, key, dtype in kept["outs"] if kind == "full"}
            delta = {i: (key, dtype) for i, kind, key, dtype in kept["outs"] if kind == "delta"}
            if kept["tree"] is not None:          # the port has no such entry: the whole result was kept
                leaves = [self._z[key].astype(dtype) for key, dtype in (full[i] for i in range(len(full)))]
                tree = kept["tree"]
                twin_digests = []
            else:
                twin = self._twin(name, args, kwargs)
                if twin is None:
                    raise ReplayMismatch(where + ": the port no longer answers this call")
                leaves, tree = _flatten(twin)
                leaves = [np.asarray(t) for t in leaves]
                twin_digests = [digest(t) for t in leaves]
            if _check(name, args, kwargs, twin_digests) != want:
                raise ReplayMismatch(where + ": the inputs, or what the port computes from them, differ from the recording: the port's result "
                                     "is not the reference's (or the test changed its inputs: record again with --record-reference)")
            for i, (key, dtype) in delta.items():
                leaves[i] = _from_bits(_bits(leaves[i]).reshape(-1) + self._z[key].astype(np.int64), leaves[i])
            return _unflatten(tree, leaves)
        return call


_ARCHIVE = None


def recording():
    """{"z": archive, "checks": ..., "kept": ..., "tests": {test id: (first call, number of calls)}} of tests/golden/reference_calls.npz
    (tests empty when there is none)"""
    global _ARCHIVE
    if _ARCHIVE is None:
        _ARCHIVE = {"z": None, "kept": {}, "tests": {}}
        if os.path.exists(GOLDEN):
            z = np.load(GOLDEN)
            meta = json.loads(z["meta"].tobytes().decode())
            _ARCHIVE = {"z": z, "checks": z["checks"], "kept": meta["kept"], "tests": {t: (first, n) for t, first, n in meta["tests"]}}
    return _ARCHIVE
