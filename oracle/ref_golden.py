"""ORACLE / REFERENCE SHIM (test infrastructure, not product code).

Recorded answers of the compiled reference (oracle/ref.py), so that the tests pinning the oracle and the product against the
reference's own code run from the repository alone.  The reference's sources are not part of the repository, so oracle/_ref/
can only be built where they are available (oracle/Makefile); everywhere else the tests replay what it answered.

A Recording holds, per test, the sequence of calls made to the reference: the call's name, a hash of its inputs and its output.
  * record mode (LTR_RECORD_REFERENCE=1, oracle/_ref built): every call runs the reference and is appended; the file under
    tests/golden/ is rewritten when the test module finishes.  Run single-process:
        LTR_RECORD_REFERENCE=1 python -m pytest -p no:xdist tests/test_ref_pin.py
  * replay mode (default): every call is answered from the file after checking that its name and inputs are the recorded ones,
    so a replay only ever answers the question that was asked of the reference.
Small float64 arrays (poses, their inverses, extrinsics: the tests feed them to the oracle) are stored as they are, every other
array as shape, dtype and SHA-256 (a Digest): the tests compare bit for bit, so a digest loses nothing, and bits_equal /
values_equal below accept either form.
"""
import contextlib
import gzip
import hashlib
import inspect
import json
import os

import numpy as np

RAW_BYTES = 1024
RECORD = os.environ.get("LTR_RECORD_REFERENCE") == "1"


def _sha(a):
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()[:32]


class Digest:
    """An array of the reference known by its shape, dtype and SHA-256."""

    def __init__(self, shape, dtype, sha):
        self.shape, self.dtype, self.sha = tuple(shape), np.dtype(dtype), sha

    def __len__(self):
        return self.shape[0]

    def matches(self, a):
        a = np.ascontiguousarray(a)
        return a.shape == self.shape and a.dtype == self.dtype and _sha(a) == self.sha

    def __repr__(self):
        return f"Digest(shape={self.shape}, dtype={self.dtype}, sha={self.sha})"


def bits_equal(a, b):
    """Same shape, dtype and bytes; either side may be a Digest."""
    if isinstance(a, Digest) or isinstance(b, Digest):
        d, x = (a, b) if isinstance(a, Digest) else (b, a)
        return d.matches(x) if not isinstance(x, Digest) else (d.shape, d.dtype, d.sha) == (x.shape, x.dtype, x.sha)
    a = np.ascontiguousarray(a); b = np.ascontiguousarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a.view(np.uint8), b.view(np.uint8))


def values_equal(a, b):
    """np.array_equal (same shape, equal values, any dtypes); either side may be a Digest."""
    if isinstance(a, Digest) or isinstance(b, Digest):
        d, x = (a, b) if isinstance(a, Digest) else (b, a)
        x = np.asarray(x)
        if x.shape != d.shape:
            return False
        xc = x.astype(d.dtype)
        return bool(np.array_equal(xc, x)) and d.matches(xc)
    return bool(np.array_equal(a, b))


def _in_hash(x, h):
    """Feeds the inputs of a call into h.  String values of a dict are file-system paths (the node's parameters) and are left out."""
    if isinstance(x, Digest):
        h.update(b"A" + x.sha.encode())
    elif isinstance(x, np.ndarray):
        h.update(b"A" + _sha(x).encode())
    elif isinstance(x, dict):
        h.update(b"{")
        for k in sorted(x):
            if not isinstance(x[k], str):
                h.update(str(k).encode()); _in_hash(x[k], h)
        h.update(b"}")
    elif isinstance(x, (list, tuple)):
        h.update(b"[")
        for v in x:
            _in_hash(v, h)
        h.update(b"]")
    else:
        h.update(repr(x.item() if isinstance(x, np.generic) else x).encode() + b",")


class Recording:
    def __init__(self, path, record=RECORD):
        self.path, self.record = path, record
        self.streams, self.cur = {}, None
        if not record:
            with gzip.open(path, "rt") as f:
                self.streams = json.load(f)

    @contextlib.contextmanager
    def test(self, name):
        """Scope of one test: its calls form one stream.  A replayed test must make every recorded call."""
        if not self.record and name not in self.streams:
            raise KeyError(f"{os.path.basename(self.path)} holds no recording of {name}")
        self.cur, self.pos, self._calls = name, 0, []
        if self.record:
            self.streams.pop(name, None)
        try:
            yield
        finally:
            self.cur = None
        if self.record:
            self.streams[name] = self._calls
        else:
            assert self.pos == len(self.streams[name]), f"{name}: {len(self.streams[name]) - self.pos} recorded calls were not made"

    def _encode(self, v):
        if v is None or isinstance(v, (bool, int, float, str)):
            return v
        if isinstance(v, np.generic):
            return v.item()
        if isinstance(v, np.ndarray):
            if v.dtype == np.float64 and v.nbytes <= RAW_BYTES:
                return {"f": [list(v.shape), v.ravel().tolist()]}
            return {"d": [list(v.shape), v.dtype.str, _sha(v)]}
        if isinstance(v, tuple):
            return {"t": [self._encode(x) for x in v]}
        if isinstance(v, list):
            return [self._encode(x) for x in v]
        if isinstance(v, dict):
            return {"m": [[k, self._encode(x)] for k, x in v.items()]}
        raise TypeError(f"cannot record a {type(v).__name__}")

    def _decode(self, v):
        if isinstance(v, list):
            return [self._decode(x) for x in v]
        if isinstance(v, dict):
            if "f" in v:
                return np.array(v["f"][1], np.float64).reshape(v["f"][0])
            if "d" in v:
                return Digest(*v["d"])
            if "t" in v:
                return tuple(self._decode(x) for x in v["t"])
            return {k: self._decode(x) for k, x in v["m"]}
        return v

    def call(self, what, inputs, fn):
        """fn() when recording (its result is stored), the recorded result otherwise."""
        assert self.cur is not None, "reference call outside a recorded test"
        h = hashlib.sha256(what.encode())
        _in_hash(inputs, h)
        h = h.hexdigest()[:16]
        if self.record:
            out = fn()
            self._calls.append([what, h, self._encode(out)])
            return out
        stream = self.streams[self.cur]
        assert self.pos < len(stream), f"{self.cur}: call {self.pos} ({what}) was not recorded"
        w, rh, out = stream[self.pos]
        assert (w, rh) == (what, h), f"{self.cur}: call {self.pos} is {what} with inputs {h}, the recording has {w} with inputs {rh}"
        self.pos += 1
        return self._decode(out)

    def examples(self, body, decorate):
        """Property tests: decorate(f) applies hypothesis' @settings/@given to f.  Recording runs body over the generated examples and
        stores each example's arguments; replay runs body over the stored examples."""
        if self.record:
            def run(*args):
                self.call("example", (), lambda: list(args))
                body(*args)
            run.__signature__ = inspect.signature(body)
            decorate(run)()
            return
        stream = self.streams[self.cur]
        n = 0
        while self.pos < len(stream) and stream[self.pos][0] == "example":
            body(*self.call("example", (), None))
            n += 1
        assert n > 0, f"{self.cur}: no recorded examples"

    def save(self, all_passed=True):
        """Writes the recording (record mode only), and only after a run in which every test passed."""
        if not self.record:
            return
        if not all_passed:
            raise RuntimeError(f"not writing {self.path}: a test failed while recording")
        with open(self.path, "wb") as raw, gzip.GzipFile(fileobj=raw, mode="wb", mtime=0) as f:
            f.write(json.dumps(self.streams, sort_keys=True, separators=(",", ":")).encode())


class RecordedRef:
    """oracle.ref's interface (free functions and the Removerter node) answered through a Recording."""
    FREE = ("cart2sph", "rad2deg", "reset_rimg_size", "map2rimg", "parse_projected", "transform_global_to_local", "linspace_int", "inverse4x4")

    def __init__(self, path):
        self.rec = Recording(path)

    @property
    def compiled(self):
        """The compiled reference itself (record mode only)."""
        from oracle import ref
        if not ref.available():
            raise RuntimeError("recording needs oracle/_ref/libltremovert_ref.so (make -C oracle ref)")
        return ref

    def __getattr__(self, name):
        if name not in self.FREE:
            raise AttributeError(name)
        return lambda *a, **k: self.rec.call(name, (a, k), lambda: getattr(self.compiled, name)(*a, **k))

    def capture(self, what, inputs, fn):
        """A value computed from the reference's outputs by fn (which may use self.compiled) when recording; the recorded one otherwise."""
        return self.rec.call(what, inputs, fn)

    def Removerter(self, params, **kw):
        return _RecordedRemoverter(self, params, kw)


class _RecordedRemoverter:
    def __init__(self, owner, params, kw):
        self._rec, self._dir = owner.rec, params.get("save_pcd_directory", "")
        self._R = owner.compiled.Removerter(params, **kw) if self._rec.record else None
        self._rec.call("Removerter", (params, kw), lambda: None)

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        return lambda *a, **k: self._rec.call(name, (a, k), lambda: getattr(self._R, name)(*a, **k))

    def saved(self):
        """As oracle.ref: [(path, cloud)]; paths below save_pcd_directory are stored relative to it."""
        d = self._dir

        def run():
            return [("<out>" + p[len(d):] if d and p.startswith(d) else p, a) for p, a in self._R.saved()]
        return [(d + p[5:] if p.startswith("<out>") else p, a) for p, a in self._rec.call("saved", (), run)]
