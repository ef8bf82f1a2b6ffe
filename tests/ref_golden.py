"""Stored results of the reference build (oracle/_ref: the reference's own sources, see oracle/ref.py), so that the tests that
compare against the reference run from a checkout alone.

    G = Golden("ref_extract")
    rk, rd = G("extract_640x480", lambda: R.extract(img, 1000))

returns the value stored under that key in tests/golden/ref_extract.npz.  With ORB_REF_GOLDEN=write (and the reference
build present) the lambda runs instead, and every value it returned is written back to the file when the process exits:

    ORB_REF_GOLDEN=write python -m pytest tests/test_oracle_vs_ref.py tests/test_gpu_facade_vs_ref.py

Values are numpy arrays (structured ones included), Python scalars, strings and tuples / lists / dicts of them.  Large
outputs that the oracle reproduces bit for bit (the reference's keypoints and descriptors) are stored as a digest only:
see extraction()."""
import atexit
import hashlib
import json
import os

import numpy as np

import oracle as O

DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
WRITE = os.environ.get("ORB_REF_GOLDEN") == "write"


def _enc(v, arrays):
    if isinstance(v, np.ndarray):
        k = "a%d" % len(arrays)
        arrays[k] = v
        return {"@": k}
    if isinstance(v, tuple):
        return {"t": [_enc(x, arrays) for x in v]}
    if isinstance(v, list):
        return {"l": [_enc(x, arrays) for x in v]}
    if isinstance(v, dict):
        return {"d": {str(k): _enc(x, arrays) for k, x in v.items()}}
    if isinstance(v, np.generic):
        v = v.item()
    if isinstance(v, (bool, int, float, str)):
        return {"s": v}
    raise TypeError("cannot store %r" % type(v))


def _dec(e, arrays):
    if "@" in e:
        return arrays[e["@"]]
    if "t" in e:
        return tuple(_dec(x, arrays) for x in e["t"])
    if "l" in e:
        return [_dec(x, arrays) for x in e["l"]]
    if "d" in e:
        return {k: _dec(x, arrays) for k, x in e["d"].items()}
    return e["s"]


class Golden:
    def __init__(self, name):
        self.path = os.path.join(DIR, name + ".npz")
        self._values = None
        self._new = {}
        if WRITE:
            atexit.register(self._save)

    def _load(self):
        if self._values is None:
            values = {}
            if os.path.exists(self.path):
                with np.load(self.path, allow_pickle=False) as z:
                    arrays = {k: z[k] for k in z.files}
                schema = json.loads(str(arrays.pop("schema")))
                values = {k: _dec(e, arrays) for k, e in schema.items()}
            self._values = values
        return self._values

    def __call__(self, key, compute):
        if not WRITE:
            values = self._load()
            if key not in values:
                raise KeyError("%s has no entry %r: regenerate it with ORB_REF_GOLDEN=write where the reference build exists"
                               % (self.path, key))
            return values[key]
        arrays = {}
        e = _enc(compute(), arrays)
        self._new[key] = (e, arrays)
        return _dec(e, arrays)

    def _save(self):
        if not self._new:
            return
        values = dict(self._load())
        values.update({k: _dec(e, a) for k, (e, a) in self._new.items()})
        arrays = {}
        schema = {k: _enc(values[k], arrays) for k in sorted(values)}
        np.savez_compressed(self.path, schema=np.array(json.dumps(schema, sort_keys=True)), **arrays)


def digest(*arrays):
    """sha256 over dtype, shape and bytes of each array"""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        h.update(("%s%s" % (a.dtype.descr, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def extraction(golden, key, img, nfeatures, scale_factor, nlevels, score_type, fast_th, reference):
    """The reference's ORBextractor output on `img` (`reference()` returns it where the reference build exists).  Only its
    digest is stored: the oracle with the reference's own retention rule (libstdc++'s nth_element) reproduces it bit for bit,
    so it is recomputed that way here and must match the digest."""
    want = golden(key, lambda: digest(*reference()))
    p = O.make_params(nfeatures, scale_factor, nlevels, score_type, fast_th, ties_mode=O.TIES_NTH_ELEMENT)
    rc, k, d, _ = O.extract(p, img)
    assert rc == 0 and digest(k, d) == want, "%s: the oracle (nth_element retention) differs from the reference's extractor" % key
    return k, d
