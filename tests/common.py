"""Shared test helpers: library loading (oracle, reference-from-source, product), PU tables, fixtures.

The reference library (oracle/_ref/libx265ref{8,10}.so) is compiled from /root/reference by
oracle/Makefile.ref; it is test infrastructure and travels to the GPU box as a prebuilt .so.
"""
import ctypes as C
import hashlib
import json
import os
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# LumaPU order of /root/reference/source/common/primitives.h:41-55
LUMA_PU = [(4, 4), (8, 8), (16, 16), (32, 32), (64, 64), (8, 4), (4, 8), (16, 8), (8, 16), (32, 16), (16, 32),
           (64, 32), (32, 64), (16, 12), (12, 16), (16, 4), (4, 16), (32, 24), (24, 32), (32, 8), (8, 32),
           (64, 48), (48, 64), (64, 16), (16, 64)]
LUMA_CU = [4, 8, 16, 32, 64]
CSP_I420 = 1

P = C.c_void_p
I = C.c_int
IP = C.c_ssize_t  # intptr_t


def pixel_dtype(depth):
    return np.uint8 if depth == 8 else np.uint16


def ref_path(depth):
    return os.path.join(ROOT, "oracle", "_ref", "libx265ref%d.so" % depth)


def oracle_path(depth):
    return os.path.join(ROOT, "oracle", "liboracle%d.so" % depth)


_cache = {}


def load_ref(depth):
    key = ("ref", depth)
    if key not in _cache:
        p = ref_path(depth)
        if not os.path.exists(p):
            return None
        L = C.CDLL(p)
        L.x265ref_get.restype = C.c_void_p
        L.x265ref_get.argtypes = [C.c_char_p, I, I, I]
        L.x265ref_dct_matrix.restype = C.c_void_p
        L.x265ref_luma_filter.restype = C.c_void_p
        L.x265ref_chroma_filter.restype = C.c_void_p
        L.x265ref_intra_filter_flags.restype = C.c_void_p
        L.x265ref_lambda.restype = C.c_double
        L.x265ref_lambda2.restype = C.c_double
        L.x265ref_lambda.argtypes = [I]
        _cache[key] = L
    return _cache[key]


def load_oracle(depth):
    key = ("orc", depth)
    if key not in _cache:
        p = oracle_path(depth)
        if not os.path.exists(p):
            import subprocess
            subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")], stdout=subprocess.DEVNULL)
        L = C.CDLL(p)
        L.orc_dct_matrix.restype = C.c_void_p
        L.orc_var.restype = C.c_uint64
        sse = C.c_uint32 if depth == 8 else C.c_uint64
        L.orc_sse_pp.restype = sse
        L.orc_sse_ss.restype = sse
        L.orc_ssd_s.restype = sse
        L.orc_quant.restype = C.c_uint32
        L.orc_nquant.restype = C.c_uint32
        L.orc_copy_cnt.restype = C.c_uint32
        _cache[key] = L
    return _cache[key]


class Digest(str):
    """The first 32 bits of the SHA-256 of an array's dtype, shape and bytes: what tests/golden/ref stores for arrays too
    large to keep whole.  The table checks compare about 20000 output blocks, so longer digests would outweigh the rest of
    the data; a wrong block still passes with probability 2**-32 only."""

    @classmethod
    def of(cls, a):
        a = np.ascontiguousarray(a)
        return cls(hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode() + a.tobytes()).hexdigest()[:8])


def same(a, b):
    """Exact equality of two arrays, either of which may be given by its Digest."""
    if isinstance(a, Digest) or isinstance(b, Digest):
        return (a if isinstance(a, Digest) else Digest.of(a)) == (b if isinstance(b, Digest) else Digest.of(b))
    return np.array_equal(a, b)


class _RefStandIn:
    """Takes the place of the reference library while stored results are replayed: its entry points accept any call and
    compute nothing, except the lambda table, which the tests also feed to the oracle (constants.cpp:33-50)."""

    def __init__(self, depth):
        self.depth = depth

    def x265ref_lambda(self, qp):
        from frame_helpers import lambda_for
        return lambda_for(qp, self.depth)

    def __getattr__(self, name):
        fn = lambda *args: 0           # noqa: E731
        setattr(self, name, fn)
        return fn


def _steps(keys):
    """Keys "<result index>.<suffix>" as index steps and suffixes, which compress to almost nothing."""
    idx = [int(k[:5]) for k in keys]
    return {"step": [b - a for a, b in zip([0] + idx, idx)], "suffix": [k[5:] for k in keys]}


def _keys(part):
    return ["%05d%s" % (i, sfx) for i, sfx in zip(np.cumsum(part["step"], dtype=np.int64), part["suffix"])]


class RefResults:
    """What the reference computed in one test, in the order the test asks for it.

    The tests that pin the oracle to the reference's own code run the same seeded inputs through both and compare.  The
    reference's side is read from tests/golden/ref/<name>.npz, so the tests need neither the reference sources nor
    oracle/_ref; `R` is then a stand-in whose calls compute nothing, and `rec(value)` returns the stored result in place
    of `value`.  With X265_RECORD_GOLDEN=1 and oracle/_ref built (tests/golden/make_golden.py --ref), `R` is the real
    reference library, `rec(value)` keeps `value`, and `done()` writes the file.  Integers and tuples of integers and
    arrays up to 64 elements are stored whole, larger arrays as their Digest (compare those with `same`)."""

    LIMIT = 64

    def __init__(self, name, depth):
        self.path = os.path.join(ROOT, "tests", "golden", "ref", name + ".npz")
        self.recording = os.environ.get("X265_RECORD_GOLDEN") == "1"
        self.n = 0
        if self.recording:
            self.R = load_ref(depth)
            assert self.R is not None, "X265_RECORD_GOLDEN=1 needs oracle/_ref (build() where the reference sources are)"
            self.out, self.small, self.hashes, self.packed = {}, {}, {}, {}
        else:
            self.R = _RefStandIn(depth)
            # integers, tuples, digests and small arrays are kept in one JSON index and one byte array: a zip member
            # each would cost more than the values
            with np.load(self.path) as z:
                self.stored = {k: v for k, v in z.items() if not k.startswith("_")}
                index = json.loads(z["_index"].tobytes())
                data, at = z["_data"].tobytes(), 0
            self.stored.update(zip(_keys(index["small"]), index["small"]["val"]))
            self.stored.update(zip(_keys(index["hash"]), index["hash"]["val"]))
            for k, dt, shape in zip(_keys(index["arr"]), index["arr"]["dtype"], index["arr"]["shape"]):
                a = np.frombuffer(data, dt, int(np.prod(shape)), at).reshape(shape)
                self.stored[k] = a
                at += a.nbytes
            self.by_result = {}
            for k in self.stored:
                self.by_result.setdefault(k.split(".")[0], []).append(k)

    def _put(self, key, v, whole=False):
        if isinstance(v, (int, np.integer)):
            self.small[key + ".i"] = [int(v)]
        elif isinstance(v, tuple):
            self.small[key + ".t"] = [int(x) for x in v]
        elif v.size <= self.LIMIT and v.dtype.names is None:
            self.packed[key + ".a"] = np.array(v)          # a copy: the test may reuse the buffer
        elif v.size <= self.LIMIT or whole:
            self.out[key + ".a"] = np.array(v)
        else:
            self.hashes[key + ".h"] = Digest.of(v)

    def _decode(self, k):
        v = self.stored[k]
        return {"i": lambda: int(v[0]), "t": lambda: tuple(int(x) for x in v), "a": lambda: v, "h": lambda: Digest(str(v))}[k[-1]]()

    def __call__(self, value, whole=False):
        """The reference's result `value`: an int, a tuple of ints, an array, or a dict of those and of lists of arrays.
        `whole` keeps arrays whole whatever their size (results the test feeds on as inputs)."""
        key = "%05d" % self.n
        self.n += 1
        if self.recording:
            items = value.items() if isinstance(value, dict) else [(None, value)]
            for k, v in items:
                sub = key if k is None else "%s.d.%s" % (key, k)
                if isinstance(v, list):
                    for i, x in enumerate(v):
                        self._put("%s.l%d" % (sub, i), x, whole)
                else:
                    self._put(sub, v, whole)
            return value
        return self._replay(key)

    def _replay(self, key):
        # stored keys: <key>.<kind>, <key>.l<i>.<kind>, <key>.d.<field>.<kind>, <key>.d.<field>.l<i>.<kind>
        fields = {}
        for k in self.by_result.get(key, []):
            parts = k[len(key) + 1:].split(".")
            field, rest = (parts[1], parts[2:]) if parts[0] == "d" else (None, parts)
            fields.setdefault(field, {})[int(rest[0][1:]) if len(rest) == 2 else None] = self._decode(k)
        if not fields:
            raise KeyError("%s: no stored result %s (regenerate with tests/golden/make_golden.py --ref)" % (self.path, key))
        vals = {f: items[None] if None in items else [items[i] for i in range(len(items))] for f, items in fields.items()}
        return vals[None] if None in vals else vals

    def done(self):
        """End of the test: write the recorded results, or check that every stored one was asked for."""
        if self.recording:
            os.makedirs(os.path.dirname(self.path), exist_ok=True)
            index = {"small": dict(_steps(self.small), val=list(self.small.values())),
                     "hash": dict(_steps(self.hashes), val=list(self.hashes.values())),
                     "arr": dict(_steps(self.packed), dtype=[a.dtype.str for a in self.packed.values()],
                                 shape=[a.shape for a in self.packed.values()])}
            self.out["_index"] = np.frombuffer(json.dumps(index, separators=(",", ":")).encode(), np.uint8)
            self.out["_data"] = np.frombuffer(b"".join(a.tobytes() for a in self.packed.values()), np.uint8)
            np.savez_compressed(self.path, **self.out)
        else:
            assert self.n == len(self.by_result), "%s: %d results stored, %d asked for" % (self.path, len(self.by_result), self.n)


def ref_fn(L, name, restype, argtypes, i=0, j=0, k=0):
    """Fetch a function pointer from the reference's C table and type it."""
    ptr = L.x265ref_get(name.encode(), i, j, k)
    if not ptr:
        return None
    return C.CFUNCTYPE(restype, *argtypes)(ptr)


def ptr(a, off=0):
    """void* to element `off` of a numpy array."""
    return C.c_void_p(a.ctypes.data + off * a.itemsize)


def fixtures(rng, depth, shape, kind):
    """Harness-style inputs (pixelharness.cpp:31-80): random / all-min / all-max pixels."""
    mx = (1 << depth) - 1
    dt = pixel_dtype(depth)
    if kind == "rand":
        return rng.integers(0, mx + 1, shape).astype(dt)
    if kind == "min":
        return np.zeros(shape, dt)
    if kind == "max":
        return np.full(shape, mx, dt)
    raise ValueError(kind)


def resid_fixture(rng, depth, shape, kind):
    """Residual inputs as in mbdstharness.cpp:61-82."""
    mx = (1 << depth) - 1
    if kind == "rand":
        return (rng.integers(0, mx + 1, shape) - rng.integers(0, mx + 1, shape)).astype(np.int16)
    if kind == "min":
        return np.full(shape, -mx, np.int16)
    if kind == "max":
        return np.full(shape, mx, np.int16)
    raise ValueError(kind)


def make_plane(rng, depth, w, h, margin, kind="rand", smooth=False):
    """A picture plane with replicated margins; returns (buffer, stride, origin_offset)."""
    dt = pixel_dtype(depth)
    mx = (1 << depth) - 1
    stride = (w + 2 * margin + 63) // 64 * 64
    buf = np.zeros((h + 2 * margin, stride), dt)
    if smooth:
        yy, xx = np.mgrid[0:h, 0:w]
        img = 128 + 60 * np.sin(xx / 17.0) + 40 * np.cos(yy / 11.0) + rng.integers(-6, 7, (h, w))
        img = np.clip(img, 0, 255).astype(np.int64) << (depth - 8)
    elif kind == "rand":
        img = rng.integers(0, mx + 1, (h, w))
    else:
        img = np.full((h, w), 0 if kind == "min" else mx)
    buf[margin:margin + h, margin:margin + w] = img
    buf[margin:margin + h, :margin] = buf[margin:margin + h, margin:margin + 1]
    buf[margin:margin + h, margin + w:margin + w + margin] = buf[margin:margin + h, margin + w - 1:margin + w]
    buf[:margin, :] = buf[margin:margin + 1, :]
    buf[margin + h:, :] = buf[margin + h - 1:margin + h, :]
    return buf, stride, margin * stride + margin
