import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def golden(name):
    return dict(np.load(os.path.join(GOLDEN, name)))


def bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def bit_equal(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and bool(np.all(bits(a) == bits(b))) if a.dtype.kind == "f" else a.shape == b.shape and bool(np.all(a == b))


def rel_l2(a, b):
    a = np.asarray(like(a, b), np.float64)
    b = np.asarray(b, np.float64)
    return float(np.sqrt(((a - b) ** 2).sum()) / max(np.sqrt((b ** 2).sum()), 1e-30))


# Outputs of the live oracle for the tests that compare the device with it, recorded so that they also run where oracle/_ref is not built
# (it is built only where the reference sources exist).  An array the test compares bit for bit is kept as a 128-bit digest of its bytes; one it
# compares within a tolerance (named in `keep`) as a fixed, seeded sample of RECORD_PIXELS pixels; arrays of up to RECORD_SMALL elements whole.
# ETXB_RECORD_ORACLE=1 with the oracle built rewrites the entries of the tests that ran.
ORACLE_RECORDS = os.path.join(GOLDEN, "oracle_records.npz")
RECORD_SMALL, RECORD_PIXELS = 16, 128
_records, _recorded = None, {}


class Digest(str):
    @classmethod
    def of(cls, a):
        import hashlib
        a = np.ascontiguousarray(a)
        return cls(hashlib.sha256(f"{a.dtype.str}{a.shape}".encode() + a.tobytes()).hexdigest()[:32])


class PixelSample(np.ndarray):
    """The same RECORD_PIXELS pixels of an (H, W, C) image every time: `pixels_of(a)` takes them from another image of that shape."""

    @staticmethod
    def index(shape):
        n = shape[0] * shape[1]
        return np.sort(np.random.default_rng(0).choice(n, min(RECORD_PIXELS, n), replace=False))

    @classmethod
    def of(cls, a):
        s = np.ascontiguousarray(a.reshape(a.shape[0] * a.shape[1], -1)[cls.index(a.shape)]).view(cls)
        s.image_shape = tuple(a.shape)
        return s

    def pixels_of(self, a):
        assert tuple(a.shape) == self.image_shape, (a.shape, self.image_shape)
        return np.asarray(a).reshape(a.shape[0] * a.shape[1], -1)[self.index(a.shape)]


def like(a, b):
    """`a` reduced to what `b` holds: the pixels of a recorded sample, else `a` itself."""
    return b.pixels_of(a) if isinstance(b, PixelSample) else a


def same_bits(a, b):
    """`a` (device output) is bit for bit `b` (a live oracle output or its recorded digest)."""
    return Digest.of(a) == b if isinstance(b, Digest) else bit_equal(a, b)


def _read_records():
    """{test key: {name: Digest, PixelSample or array}} from ORACLE_RECORDS: `names` (key|name|kind), `digests` (16 bytes each), and the samples
    and small arrays one after another in `values` (float64; `shapes` gives each one's shape, `dtypes` its type)."""
    global _records
    if _records is None:
        _records = {}
        if os.path.exists(ORACLE_RECORDS):
            with np.load(ORACLE_RECORDS) as z:
                digests, values, shapes, dtypes = iter(z["digests"]), z["values"], iter(z["shapes"]), iter(z["dtypes"])
                at = 0
                for entry in z["names"]:
                    key, name, kind = str(entry).split("|")
                    if kind == "digest":
                        v = Digest(next(digests).tobytes().hex())
                    else:
                        shape = tuple(int(d) for d in next(shapes) if d >= 0)
                        n = int(np.prod(shape))
                        v = values[at:at + n].astype(str(next(dtypes))).reshape(shape)
                        at += n
                        if kind == "sample":
                            v = v.view(PixelSample)
                            v.image_shape = tuple(int(d) for d in next(shapes) if d >= 0)
                    _records.setdefault(key, {})[name] = v
    return _records


def _to_record(outputs, keep):
    out = {}
    for k, v in outputs.items():
        v = np.asarray(v)
        out[k] = PixelSample.of(v) if k in keep else v if v.size <= RECORD_SMALL else Digest.of(v)
    return out


def _write_records(records):
    names, digests, values, shapes, dtypes = [], [], [], [], []
    for key in sorted(records):
        for name, v in records[key].items():
            kind = "digest" if isinstance(v, Digest) else "sample" if isinstance(v, PixelSample) else "array"
            names.append(f"{key}|{name}|{kind}")
            if kind == "digest":
                digests.append(np.frombuffer(bytes.fromhex(v), np.uint8))
                continue
            shapes.append(list(v.shape) + [-1] * (4 - v.ndim))
            if kind == "sample":
                shapes.append(list(v.image_shape) + [-1] * (4 - len(v.image_shape)))
            dtypes.append(np.asarray(v).dtype.str)
            values.append(np.asarray(v, np.float64).reshape(-1))
    np.savez_compressed(ORACLE_RECORDS, names=np.array(names), digests=np.array(digests, np.uint8).reshape(-1, 16), values=np.concatenate(values),
                        shapes=np.array(shapes, np.int64), dtypes=np.array(dtypes))


def _agree(out, rec):
    return sorted(rec) == sorted(out) and all(
        same_bits(out[k], rec[k]) if isinstance(rec[k], Digest) else bit_equal(like(out[k], rec[k]), np.asarray(rec[k])) for k in rec)


@pytest.fixture
def oracle_record(request):
    """oracle_record(label, run, keep=(), live_only=()) -> {name: array or its record}: run(oracle_py) -> {name: array} where the oracle is built
    (checked against the committed record when there is one), else the committed record of this test and label, which leaves out `live_only`."""
    from oracle import oracle_py
    live = oracle_py.available("parity")

    def get(label, run, keep=(), live_only=()):
        path, name = request.node.nodeid.split("::", 1)
        key = os.path.basename(path) + "::" + name + ("/" + label if label else "")
        if live:
            out = {k: np.asarray(v) for k, v in run(oracle_py).items()}
            recordable = {k: v for k, v in out.items() if k not in live_only}
            if os.environ.get("ETXB_RECORD_ORACLE") == "1":
                _recorded[key] = _to_record(recordable, keep)
            elif key in _read_records():
                assert _agree(recordable, _records[key]), f"{key}: the committed oracle record is stale"
            return out
        if key not in _read_records():
            pytest.fail(f"no recorded oracle outputs for {key} (ETXB_RECORD_ORACLE=1 where oracle/_ref is built writes them)")
        return dict(_records[key])

    return get


def pytest_sessionfinish(session):
    if _recorded:
        _write_records({**_read_records(), **_recorded})


@pytest.fixture(scope="session")
def oracle_mod():
    from oracle import oracle_py
    if not oracle_py.available("parity"):
        pytest.skip("oracle/_ref/liboracle_parity.so not built (run oracle/build_oracle.sh where /root/reference exists)")
    return oracle_py
