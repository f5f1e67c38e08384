"""Recorded outputs of the reference's own sources, for tests/test_ref_pin.py.

Every test there runs the same seeded inputs through the reference build (ref_api, oracle/_ref/libvxref.so) and through the hand-written oracle
(oracle_api) and compares the two.  The reference build needs the original project's sources, which a checkout of this repository does not have,
so each test reads the reference side through a `Recording`: while recording (VXS_RECORD_REF_GOLDEN=1 and the library built) it computes each
quantity the test compares with the library and stores it; otherwise it returns the stored quantity.  The oracle side always runs.

What is stored, per quantity, is what its comparison needs:
  value(name, fn)   the value itself (scalars, small arrays, dicts of them), exactly;
  digest(name, fn)  the SHA-256 of the dtype, shape and bytes of an array (or of a tuple of arrays), for bit-exact comparisons of large arrays;
  rows(name, fn)    the row count and a fixed, seeded sample of rows (Rows.idx, Rows.rows) of a large array, for comparisons within a tolerance.
The recording of one test is one .npz under tests/golden/ref_pin/ holding `index` (JSON: name, start, end) and `blob` (the .npy images of the
quantities back to back, deflated as one stream); tests/golden/make_ref_pin_golden.py writes them all.
"""
import hashlib
import io
import json
import os
import re
import zlib

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_pin")
RECORD_ENV = "VXS_RECORD_REF_GOLDEN"
SAMPLE_ROWS = 12           # rows of a sample, fewer for wide rows (at most SAMPLE_VALUES values, at least 2 rows)
SAMPLE_VALUES = 256


def recording():
    return os.environ.get(RECORD_ENV) == "1"


def golden_path(test_name):
    return os.path.join(GOLDEN_DIR, re.sub(r"[^A-Za-z0-9_.-]+", "_", test_name).strip("_") + ".npz")


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(f"{a.dtype.str}{a.shape}".encode())
        h.update(a.tobytes())
    return h.hexdigest()


class Rows:
    """`n` rows in all; `rows` are rows `idx` of the array (ascending, chosen by a seed derived from the quantity's name)"""

    def __init__(self, n, idx, rows):
        self.n, self.idx, self.rows = int(n), idx, rows


class Recording:
    def __init__(self, test_name, record, ref_module):
        self.path, self.record = golden_path(test_name), record
        self.ra = ref_module if record else None        # the library itself, only while recording
        self.data = {}
        if not record:
            if not os.path.exists(self.path):
                raise FileNotFoundError(f"{self.path}: no recording of the reference's outputs for {test_name}; run tests/golden/make_ref_pin_golden.py")
            with np.load(self.path, allow_pickle=False) as z:
                index, blob = json.loads(str(z["index"])), z["blob"].tobytes()
            self.data = {k: np.load(io.BytesIO(blob[a:b]), allow_pickle=False) for k, a, b in index}
        self.used = set()

    def _key(self, name):
        assert re.fullmatch(r"[A-Za-z0-9_.]+", name), name
        assert name not in self.used, f"{name} recorded twice"
        self.used.add(name)
        if not self.record and not any(k == name or k.startswith(name + "/") for k in self.data):
            raise KeyError(f"{self.path} has no {name}: re-record with tests/golden/make_ref_pin_golden.py")
        return name

    def value(self, name, fn):
        k = self._key(name)
        if self.record:
            v = fn()
            if isinstance(v, dict):
                for f, x in v.items():
                    self.data[f"{k}/{f}"] = np.asarray(x)
            else:
                self.data[k] = np.asarray(v)
            return v
        if k in self.data:
            v = self.data[k]
            return v[()] if v.ndim == 0 else v
        return {f[len(k) + 1:]: (x[()] if x.ndim == 0 else x) for f, x in self.data.items() if f.startswith(k + "/")}

    def digest(self, name, fn):
        k = self._key(name)
        if self.record:
            v = fn()
            self.data[k] = np.array(digest(*v) if isinstance(v, tuple) else digest(v))
        return str(self.data[k])

    def rows(self, name, fn):
        key = self._key(name)
        if self.record:
            a = np.asarray(fn())
            k = max(2, min(SAMPLE_ROWS, SAMPLE_VALUES // max(1, a[0].size if len(a) else 1)))
            rng = np.random.default_rng(zlib.crc32(name.encode()))
            idx = np.sort(rng.choice(len(a), min(k, len(a)), replace=False)).astype(np.int64)
            self.data[f"{key}/n"], self.data[f"{key}/idx"], self.data[f"{key}/rows"] = np.array(len(a)), idx, a[idx]
        return Rows(self.data[f"{key}/n"], self.data[f"{key}/idx"], self.data[f"{key}/rows"])

    def finish(self):
        if self.record:
            buf, index = io.BytesIO(), []
            for k, a in self.data.items():
                start = buf.tell()
                np.save(buf, a, allow_pickle=False)
                index.append((k, start, buf.tell()))
            os.makedirs(GOLDEN_DIR, exist_ok=True)
            np.savez_compressed(self.path, index=np.array(json.dumps(index)), blob=np.frombuffer(buf.getvalue(), dtype=np.uint8))
        else:
            unused = sorted({k.split("/")[0] for k in self.data} - self.used)
            assert not unused, f"{self.path}: recorded but not compared: {unused}"
