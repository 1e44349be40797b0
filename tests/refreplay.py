"""Record / replay of the reference's Python stack for tests/test_refpin_vector.py.

The reference package (`metaworld`, running on the gymnasium / mujoco stand-ins of oracle/refshim) is not part of this
repository.  tests/golden/make_refstack_goldens.py runs each test of that module once against the live reference with a
recording session, which logs every value the reference hands back; the suite runs the same test bodies against a
replaying session, which hands those values back in the same order from tests/golden/refstack/<test>.npz.

Values are stored as plain data (numpy arrays and scalars, Python scalars, strings, bytes, tuples, lists, dicts).  Any
other object (a module, an env, a space, a class, a bound method) becomes a `Proxy`; its attribute reads and writes,
calls, item reads and repr are logged in turn, and so are the exceptions they raise.  Replay checks that the test asks
for the same thing at every position of the log, so a test that drifts from its recording fails instead of comparing
against the wrong value."""
from __future__ import annotations

import base64
import builtins
import hashlib
import io
import json
import os
import pickle

import numpy as np

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "refstack")
_LEAF = (type(None), bool, int, float, str)


class Proxy:
    """Stand-in for one reference object (the live object while recording, nothing but an id while replaying)."""

    __slots__ = ("_session", "_id", "_real")

    def __init__(self, session, oid, real):
        object.__setattr__(self, "_session", session)
        object.__setattr__(self, "_id", oid)
        object.__setattr__(self, "_real", real)

    def __getattr__(self, name):
        return self._session.op(self, "getattr", name, lambda r: getattr(r, name))

    def __setattr__(self, name, value):
        self._session.op(self, "setattr", name, lambda r: setattr(r, name, _unwrap(value)))

    def __call__(self, *args, **kwargs):
        return self._session.op(self, "call", _fingerprint((args, kwargs)), lambda r: r(*_unwrap(args), **_unwrap(kwargs)))

    def __getitem__(self, key):
        return self._session.op(self, "getitem", key, lambda r: r[_unwrap(key)])

    def __repr__(self):
        return self._session.op(self, "repr", None, repr)


def unpickle(data):
    """pickle.loads for bytes the reference pickled: its classes (not importable here) come back as dotted names."""
    class _Unpickler(pickle.Unpickler):
        def find_class(self, module, name):
            try:
                return super().find_class(module, name)
            except ImportError:
                return f"{module}.{name}"
    return _Unpickler(io.BytesIO(data)).load()


def _fingerprint(x):
    """Call arguments as a string: replay checks that the test passes the reference what it passed when recorded."""
    if isinstance(x, Proxy):
        return f"<proxy {x._id}>"
    if isinstance(x, np.ndarray) and x.dtype != object:
        return f"array({x.dtype.str}, {x.shape}, {hashlib.sha1(np.ascontiguousarray(x).tobytes()).hexdigest()[:16]})"
    if isinstance(x, (tuple, list, np.ndarray)):
        return "[" + ", ".join(_fingerprint(v) for v in x) + "]"
    if isinstance(x, dict):
        return "{" + ", ".join(f"{_fingerprint(k)}: {_fingerprint(v)}" for k, v in x.items()) + "}"
    return repr(x)


def _unwrap(x):
    if isinstance(x, Proxy):
        return x._real
    if type(x) in (tuple, list):
        return type(x)(_unwrap(v) for v in x)
    if type(x) is dict:
        return {k: _unwrap(v) for k, v in x.items()}
    return x


class Session:
    """One test's log.  `Session(None)` records (the objects come from `root(obj)`); `Session.load(name)` replays."""

    def __init__(self, log=None, arrays=None):
        self.recording = log is None
        self.log = [] if log is None else log
        self.arrays = [] if arrays is None else arrays
        self.pos = 0
        self.n_obj = 0

    @classmethod
    def load(cls, name):
        with np.load(os.path.join(GOLD, name + ".npz"), allow_pickle=False) as z:
            log, index = json.loads(str(z["log"])), json.loads(str(z["index"]))
            blobs = {k: z[k] for k in z.files}
        arrays = [blobs[dt][off: off + int(np.prod(shape, dtype=np.int64))].reshape(shape) for dt, off, shape in index]
        return cls(log, arrays)

    def save(self, name):
        """The arrays go into one flat blob per dtype (thousands of small npz members would cost more than the data);
        an array equal to an earlier one (a goal vector asked for every step, say) is stored once."""
        blobs, index, seen = {}, [], {}
        for a in self.arrays:
            parts = blobs.setdefault(a.dtype.str, [])
            key = (a.dtype.str, a.shape, a.tobytes())
            if key not in seen:
                seen[key] = sum(p.size for p in parts)
                parts.append(a.ravel())
            index.append([a.dtype.str, seen[key], list(a.shape)])
        os.makedirs(GOLD, exist_ok=True)
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), log=np.array(json.dumps(self.log)), index=np.array(json.dumps(index)),
                            **{dt: np.concatenate(parts) for dt, parts in blobs.items()})

    def root(self, real=None):
        """The proxy every test starts from (its attributes are the reference modules)."""
        return self._proxy(real)

    def _proxy(self, real):
        self.n_obj += 1
        return Proxy(self, self.n_obj, real)

    def op(self, proxy, op, key, fn):
        where = [proxy._id, op, key if isinstance(key, _LEAF) else repr(key)]
        if self.recording:
            try:
                value = fn(proxy._real)
            except Exception as e:
                base = next(c.__name__ for c in type(e).__mro__ if getattr(builtins, c.__name__, None) is c)
                self.log.append(where + [{"$raise": base, "msg": str(e)}])
                raise
            enc, out = self._encode(value)
            self.log.append(where + [enc])
            return out
        if self.pos >= len(self.log) or self.log[self.pos][:3] != where:
            got = self.log[self.pos][:3] if self.pos < len(self.log) else "end of log"
            raise AssertionError(f"replay diverged from the recording at entry {self.pos}: test asks {where}, log has {got}")
        enc = self.log[self.pos][3]
        self.pos += 1
        if isinstance(enc, dict) and "$raise" in enc:
            raise getattr(builtins, enc["$raise"])(enc["msg"])
        return self._decode(enc)

    # value <-> (JSON tree, arrays); while recording, objects inside a value are handed to the test as proxies
    def _encode(self, v):
        if isinstance(v, _LEAF):
            return v, v
        if isinstance(v, bytes):
            return {"$b": base64.b64encode(v).decode()}, v
        if isinstance(v, np.dtype):
            return {"$dt": v.str}, v
        if isinstance(v, (np.ndarray, np.generic)) and np.asarray(v).dtype != object:
            self.arrays.append(np.array(v))          # a copy: the reference may reuse its buffers
            return {"$a" if isinstance(v, np.ndarray) else "$s": len(self.arrays) - 1}, v
        if isinstance(v, np.ndarray):
            pairs = [self._encode(x) for x in v.ravel()]
            out = np.empty(v.shape, dtype=object)
            out.ravel()[:] = [p[1] for p in pairs] if len(pairs) else []
            return {"$o": [p[0] for p in pairs], "shape": list(v.shape)}, out
        if type(v) in (tuple, list):
            pairs = [self._encode(x) for x in v]
            return {"$t" if type(v) is tuple else "$l": [p[0] for p in pairs]}, type(v)(p[1] for p in pairs)
        if isinstance(v, dict):
            items = [(self._encode(k), self._encode(x)) for k, x in v.items()]
            return {"$d": [[k[0], x[0]] for k, x in items]}, {k[1]: x[1] for k, x in items}
        p = self._proxy(v)
        return {"$p": p._id}, p

    def _decode(self, e):
        if not isinstance(e, dict):
            return e
        if "$b" in e:
            return base64.b64decode(e["$b"])
        if "$dt" in e:
            return np.dtype(e["$dt"])
        if "$a" in e:
            return self.arrays[e["$a"]].copy()
        if "$s" in e:
            return self.arrays[e["$s"]][()]
        if "$o" in e:
            out = np.empty(len(e["$o"]), dtype=object)
            out[:] = [self._decode(x) for x in e["$o"]] if e["$o"] else []
            return out.reshape(e["shape"])
        if "$t" in e:
            return tuple(self._decode(x) for x in e["$t"])
        if "$l" in e:
            return [self._decode(x) for x in e["$l"]]
        if "$d" in e:
            return {self._decode(k): self._decode(x) for k, x in e["$d"]}
        self.n_obj += 1
        assert e["$p"] == self.n_obj, (e, self.n_obj)
        return Proxy(self, self.n_obj, None)

    def finish(self):
        assert self.recording or self.pos == len(self.log), f"the test stopped at entry {self.pos} of {len(self.log)}"
