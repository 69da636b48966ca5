"""Stored results of the compiled reference (oracle/_ref) for machines where it cannot be built.

Tests reach the reference through the `refo` and `checker` fixtures (tests/conftest.py).  Where oracle/_ref is built they call
it directly.  Where it is not, they get a stand-in (Replay) that runs each call on the port (oracle/port) and folds everything
the call left behind -- the return value and every array its pointer arguments point into -- into one digest per test.  At the
end of the test that digest must equal the one recorded from the reference on the same inputs (tests/golden/oracle_calls.json),
so the port stands in for the reference only where it computed exactly what the reference computed.  A test with nothing
recorded is checked against the port through `checker`, and skips where it asks `refo`.  Calls the port does not
implement (the reference's own codec / scaler drivers, its table selection), or computes differently (the float transforms,
formats it does not take), are replayed from the reference's recorded effect on the caller's arrays (tests/golden/oracle_effects.bin).
A test skips without oracle/_ref where such an effect cannot stand for the reference: where the call was handed a pointer
outside the caller's arrays (a table of callbacks it may call: the code under test would not run), or returned a context the
test may hand on.  It also skips where its effects do not fit EFFECTS_BUDGET, which takes the smallest first.  Each test's
entry keeps the digest after calls 1, 2, 4, 8, ... so a mismatch names the calls it lies between, and the number of pointer
arguments whose memory was not found ("unresolved": neither digested nor replayed).

Recording needs oracle/_ref built from the reference tree, and is redone whenever a test changes what it asks the reference:

    ORACLE_GOLDEN_RECORD=<dir> python -m pytest tests [-m "not gpu"]      # one file per test under <dir>
    python tests/oracle_golden.py merge <dir>                               # rebuild tests/golden/ from them
"""
import ctypes as C
import functools
import hashlib
import json
import lzma
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle import loader  # noqa: E402

CALLS = os.path.join(HERE, "golden", "oracle_calls.json")
EFFECTS = os.path.join(HERE, "golden", "oracle_effects.bin")
RECORD_ENV = "ORACLE_GOLDEN_RECORD"
EFFECTS_BUDGET = 224 << 10     # compressed bytes of stored effects in all: what the repository carries for this purpose
_PTR_TYPES = (C.c_void_p, C.c_char_p, C._Pointer, C._CFuncPtr)


def _is_ptr_type(t):
    return isinstance(t, type) and issubclass(t, _PTR_TYPES)


def _root(a):
    while isinstance(a.base, np.ndarray):
        a = a.base
    return a


def _defined_here(v):
    m = sys.modules.get(type(v).__module__)
    return os.path.dirname(os.path.abspath(getattr(m, "__file__", None) or "/")) == HERE


def _collect(v, out, depth):
    if isinstance(v, np.ndarray):
        r = _root(v)
        out.setdefault(id(r), r)
    elif depth and hasattr(v, "__dict__") and not isinstance(v, type) and _defined_here(v):     # a test helper's arrays
        for x in list(vars(v).values())[:512]:
            _collect(x, out, depth - 1)
    elif depth and isinstance(v, (list, tuple)):
        for x in v[:512]:
            _collect(x, out, depth - 1)
    elif depth and isinstance(v, dict):
        for x in list(v.values())[:512]:
            _collect(x, out, depth - 1)


def _arrays_near(frame, depth=10):
    """Every numpy array (as its owning base) bound in the caller's frames: the memory a pointer argument can point into."""
    found = {}
    while frame is not None and depth:
        for v in list(frame.f_locals.values()):
            _collect(v, found, 3)
        frame, depth = frame.f_back, depth - 1
    spans = []
    for r in found.values():
        lo, hi = np.lib.array_utils.byte_bounds(r)
        if hi > lo:
            spans.append((lo, hi, r))
    return spans


class _Call:
    """One call's arguments, split into scalars (digested as they are) and pointers (resolved to caller arrays)."""

    def __init__(self, owner, name, args, frame):
        self.owner, self.name = owner, name
        self.spans = _arrays_near(frame)
        self.roots = []            # arrays the pointers point into, in argument order
        self.struct_ptrs = []      # pointer-valued fields of structures / pointer arrays passed in: (container, index)
        self.items = []
        self.uncovered = 0
        for t, v in zip(loader.API[name][1], args):
            self._arg(t, v)
        self.words_before = [self._word(k) for k in range(len(self.struct_ptrs))]

    def _word(self, k):
        words, i = self.struct_ptrs[k]
        return C.cast(words, C.POINTER(C.c_void_p))[i]

    def set_word(self, k, p):
        words, i = self.struct_ptrs[k]
        C.cast(words, C.POINTER(C.c_void_p))[i] = p

    def _root_of(self, p):
        for lo, hi, r in self.spans:
            if lo <= p < hi:
                for k, (x, _) in enumerate(self.roots):
                    if x is r:
                        return k, p - lo
                self.roots.append((r, lo))
                return len(self.roots) - 1, p - lo
        return None

    def _ptr(self, p):
        if not p:
            self.items.append("null")
            return
        if p in self.owner.log["handles"]:
            self.items.append("handle %d" % self.owner.log["handles"][p])
            return
        hit = self._root_of(p)
        if hit is None:
            self.uncovered += 1
            self.items.append("foreign")
        else:
            self.items.append("array %d+%d" % hit)

    def _arg(self, t, v):
        if hasattr(v, "_as_parameter_"):
            v = v._as_parameter_
        if t is not C.c_void_p:
            self.items.append(repr(v))
        elif v is None or isinstance(v, int):
            self._ptr(v)
        elif isinstance(v, C.c_void_p):
            if isinstance(getattr(v, "_arr", None), np.ndarray):      # ndarray.ctypes.data_as keeps its array there
                r = _root(v._arr)
                if not any(x is r for _, _, x in self.spans):
                    lo, hi = np.lib.array_utils.byte_bounds(r)
                    self.spans.append((lo, hi, r))
            self._ptr(v.value)
        elif type(v).__name__ == "CArgObject":           # C.byref(obj)
            self._obj(v._obj)
        else:
            self._obj(v)

    def _obj(self, o):
        if isinstance(o, C.Array) and _is_ptr_type(o._type_):
            self.items.append("pointers[%d]" % len(o))
            for i in range(len(o)):
                self.struct_ptrs.append((o, i))
                self._ptr(self._word(len(self.struct_ptrs) - 1))
        elif isinstance(o, C.Structure):
            self.items.append(type(o).__name__)
            self._struct(o)
        elif isinstance(o, (C.Array, C._SimpleCData)):
            self.items.append(("data", o))                  # digested after the call: it may be an output
        else:
            raise TypeError("oracle stand-in: cannot follow a %s argument of %s" % (type(o).__name__, self.name))

    def _struct(self, s):
        for f in s._fields_:
            name, t = f[0], f[1]
            if _is_ptr_type(t) or (issubclass(t, C.Array) and _is_ptr_type(t._type_)):
                n = t._length_ if issubclass(t, C.Array) else 1
                words = (C.c_void_p * n).from_buffer(s, getattr(type(s), name).offset)
                for i in range(n):
                    self.struct_ptrs.append((words, i))
                    self._ptr(words[i])
            elif issubclass(t, C.Structure):
                self._struct(getattr(s, name))
            else:
                self.items.append(("data", (C.c_ubyte * C.sizeof(t)).from_buffer(s, getattr(type(s), name).offset)))

    def snapshot(self):
        """The bytes of every array and ctypes object the call can write."""
        return [r.tobytes() for r, _ in self.roots], [bytes(it[1]) for it in self.items if isinstance(it, tuple)]

    def restore(self, state):
        for (r, _), b in zip(self.roots, state[0]):
            r[...] = np.frombuffer(b, r.dtype).reshape(r.shape)
        for it, b in zip([it for it in self.items if isinstance(it, tuple)], state[1]):
            C.memmove(C.addressof(it[1]), b, len(b))

    def pointer_words(self):
        """The pointer-valued words handed in, as they are after the call (a selection call writes function pointers there):
        NULL, equal to what word k held before the call, or an address of the callee's own."""
        out = []
        for k in range(len(self.struct_ptrs)):
            p = self._word(k)
            out.append(None if not p else "word %d" % self.words_before.index(p) if p in self.words_before else "foreign")
        return out

    def digest(self, result):
        h = hashlib.blake2b(digest_size=16)
        h.update(self.name.encode())
        for it in self.items:
            if isinstance(it, tuple):
                h.update(bytes(it[1]))
            else:
                h.update(it.encode())
            h.update(b"|")
        rt = loader.API[self.name][0]
        h.update(repr(("handle" if result else None) if rt is C.c_void_p else result).encode())
        for r, _ in self.roots:
            h.update(str(r.nbytes).encode())
            h.update(r if r.flags.c_contiguous else r.tobytes())
        h.update(repr(self.pointer_words()).encode())
        return h.digest()


class _Oracle:
    """The fixture object: the oracle's attribute names, each call folded into the current test's log."""

    def __init__(self, inner, prefix):
        self._inner, self.prefix = inner, prefix
        self.log = None

    def has(self, name):
        return name in loader.API

    def __getattr__(self, name):
        if name == "lib":                       # the reference library itself, driven directly by the test
            return self._lib()
        if name.startswith("_") or name not in loader.API:
            raise AttributeError(name)

        def call(*args):
            if self.log is None:
                raise RuntimeError("oracle stand-in called outside a test")
            return self._call(name, args, sys._getframe(1))
        call.__name__ = name
        return call

    def _lib(self):
        return self._inner.lib

    def _new_handle(self, p):
        if p:
            self.log["handles"][p] = self.log["nhandles"]
            self.log["nhandles"] += 1


def _xor(a, b):
    return np.bitwise_xor(np.frombuffer(a, np.uint8), np.frombuffer(b, np.uint8)).tobytes()


class Record(_Oracle):
    """Runs the compiled reference and logs each call's digest.  The same call is also made on the port, from the same inputs:
    where the port leaves anything different, or has no such function, the reference's effect is logged for Replay."""

    def __init__(self, ref, port):
        super().__init__(ref, ref.prefix)
        self.port = port

    def _call(self, name, args, frame):
        c = _Call(self, name, args, frame)
        before = c.snapshot()
        res = getattr(self._inner, name)(*args)
        digest = c.digest(res)
        after = c.snapshot()
        same, base = False, before
        if self.port.has(name):
            c.restore(before)
            same = c.digest(getattr(self.port, name)(*args)) == digest
            base = c.snapshot()
            c.restore(after)
        if loader.API[name][0] is C.c_void_p:
            self._new_handle(res)
        _count(self.log, digest)
        self.log["uncovered"] += c.uncovered
        if not same and c.uncovered:
            self.log["unstorable"] = "the reference's %s was handed pointers outside the caller's arrays (callbacks it may call)" % name
        elif not same and loader.API[name][0] is C.c_void_p:
            self.log["unstorable"] = "the reference's %s returns a context the test may hand on" % name
        if not same:
            # the effect on each array is stored as the XOR of the reference's bytes after the call with the port's after the
            # same call (or, where the port has no such function, with the bytes before the call)
            self.log["effects"].append({"call": self.log["calls"] - 1, "result": bool(res) if loader.API[name][0] is C.c_void_p else res,
                                        "on_port": base is not before,
                                        "roots": {k: _xor(b, a) for k, (b, a) in enumerate(zip(base[0], after[0])) if a != b},
                                        "words": c.pointer_words(), "data": after[1]})
        return res


class Replay(_Oracle):
    """Runs the port where it computes what the reference computed; replays the reference's recorded effect elsewhere."""

    def __init__(self, port, effects):
        super().__init__(port, "golden:" + port.prefix)
        self.effects = effects

    def _lib(self):
        import pytest
        self.log["skipped"] = True
        pytest.skip("drives the reference library itself: it needs oracle/_ref built")

    def _call(self, name, args, frame):
        want = load_calls().get(self.log["test"])
        if want is None and not self.log["strict"] and self._inner.has(name):
            return getattr(self._inner, name)(*args)        # nothing recorded: the port is the checker
        if want is None or want.get("effects") == "not stored":
            import pytest
            self.log["skipped"] = True
            pytest.skip("no recorded reference results for this test: it needs oracle/_ref built" if want is None else
                        "%s: it needs oracle/_ref built" % want["why"])
        c = _Call(self, name, args, frame)
        k = self.log["calls"]
        eff = self.effects.get((self.log["test"], k))
        if eff is None and self._inner.has(name):
            res = getattr(self._inner, name)(*args)
        else:
            if eff is None:
                raise AssertionError("%s: no recorded effect of the reference's %s (call %d); record the golden data again"
                                     % (self.log["test"], name, k))
            if eff["on_port"]:
                getattr(self._inner, name)(*args)
            res = eff["result"]
            roots = c.snapshot()[0]
            c.restore(([_xor(roots[j], eff["roots"][j]) if j in eff["roots"] else b for j, b in enumerate(roots)], eff["data"]))
            for j, w in enumerate(eff["words"]):
                # a function of the reference's own: any non-NULL address stands for it
                c.set_word(j, None if w is None else c.words_before[int(w.split()[1])] if w.startswith("word ") else 1)
        if loader.API[name][0] is C.c_void_p:
            self._new_handle(res)
        _count(self.log, c.digest(res))
        return res


def new_log(test):
    return {"test": test, "digest": hashlib.blake2b(digest_size=16), "calls": 0, "checkpoints": [], "uncovered": 0, "effects": [],
            "handles": {}, "nhandles": 0, "unstorable": None, "skipped": False, "strict": False}


def _count(log, digest):
    log["digest"].update(digest)
    log["calls"] += 1
    if log["calls"] & (log["calls"] - 1) == 0:
        log["checkpoints"].append(log["digest"].hexdigest()[:8])


def mismatch(log, want):
    """None when the test's calls match the recorded ones, else where they first differ."""
    if (log["calls"], log["digest"].hexdigest()) == (want["calls"], want["digest"]):
        return None
    for i, (a, b) in enumerate(zip(log["checkpoints"], want["checkpoints"])):
        if a != b:
            return "the stand-in's calls first differ from the reference's within calls %d..%d" % ((1 << i >> 1) + 1, 1 << i)
    return "the stand-in made %d calls, the reference %d; they first differ after call %d" % (
        log["calls"], want["calls"], 1 << (min(len(log["checkpoints"]), len(want["checkpoints"])) - 1))


@functools.lru_cache(None)
def load_calls():
    if not os.path.exists(CALLS):
        return {}
    return json.load(open(CALLS))


def load_effects():
    """{(test, call index): effect} from the packed effects file."""
    out = {}
    if not os.path.exists(EFFECTS):
        return out
    blob = lzma.decompress(open(EFFECTS, "rb").read())
    n = int.from_bytes(blob[:8], "little")
    index = json.loads(blob[8:8 + n])
    base = 8 + n
    for e in index:
        def take(span):
            return blob[base + span[0]:base + span[0] + span[1]]
        out[(e["test"], e["call"])] = {"result": e["result"], "on_port": e["on_port"], "words": e["words"],
                                       "roots": {int(k): take(v) for k, v in e["roots"].items()},
                                       "data": [take(v) for v in e["data"]]}
    return out


def write_record(directory, log):
    """One JSON file per test (the recording run may be spread over worker processes)."""
    os.makedirs(directory, exist_ok=True)
    name = hashlib.sha1(log["test"].encode()).hexdigest()[:16] + ".json"
    effects = [{"call": e["call"], "result": e["result"], "on_port": e["on_port"], "words": e["words"],
                "roots": {k: v.hex() for k, v in e["roots"].items()}, "data": [d.hex() for d in e["data"]]} for e in log["effects"]]
    size = len(lzma.compress(b"".join(v for e in log["effects"] for v in e["roots"].values()))) if effects else 0
    why = log["unstorable"] or ("the reference's output for this test is too large to store" if size > EFFECTS_BUDGET else None)
    with open(os.path.join(directory, name), "w") as f:
        json.dump({"test": log["test"], "calls": log["calls"], "digest": log["digest"].hexdigest(), "checkpoints": log["checkpoints"],
                   "uncovered": log["uncovered"], "size": size, "why": why, "effects": None if why else effects}, f)


def merge(directory):
    """Rebuilds tests/golden/oracle_calls.json and oracle_effects.bin from a recording of the whole suite."""
    recorded = [json.load(open(os.path.join(directory, n))) for n in sorted(os.listdir(directory)) if n.endswith(".json")]
    calls, effects, used = {}, {}, 0
    for r in sorted(recorded, key=lambda r: (r["why"] is not None, r["size"], r["test"])):
        calls[r["test"]] = e = {"calls": r["calls"], "digest": r["digest"], "checkpoints": r["checkpoints"]}
        if r["uncovered"]:
            e["unresolved"] = r["uncovered"]
        why = r["why"] or ("the reference's output for this test does not fit the stored effects" if used + r["size"] > EFFECTS_BUDGET else None)
        if why:
            e["effects"], e["why"] = "not stored", why
            continue
        used += r["size"]
        for x in r["effects"]:
            effects[(r["test"], x["call"])] = {"result": x["result"], "on_port": x["on_port"], "words": x["words"],
                                               "roots": {int(k): bytes.fromhex(v) for k, v in x["roots"].items()},
                                               "data": [bytes.fromhex(d) for d in x["data"]]}
    with open(CALLS, "w") as f:
        json.dump(dict(sorted(calls.items())), f, indent=0, sort_keys=True)
        f.write("\n")
    index, payload = [], bytearray()

    def put(b):
        payload.extend(b)
        return [len(payload) - len(b), len(b)]
    for (test, call), e in sorted(effects.items()):
        index.append({"test": test, "call": call, "result": e["result"], "on_port": e["on_port"], "words": e["words"],
                      "roots": {str(k): put(v) for k, v in sorted(e["roots"].items())}, "data": [put(d) for d in e["data"]]})
    head = json.dumps(index, separators=(",", ":")).encode()
    with open(EFFECTS, "wb") as f:
        f.write(lzma.compress(len(head).to_bytes(8, "little") + head + bytes(payload), preset=9 | lzma.PRESET_EXTREME))
    return len(recorded)


if __name__ == "__main__":
    if len(sys.argv) == 3 and sys.argv[1] == "merge":
        print("merged %d tests" % merge(sys.argv[2]))
    else:
        raise SystemExit(__doc__)
