"""The reference's outputs, for the tests that compare against them.

A test hands `load()` a name and a function that runs the reference (oracle/_ref, built from the original project) and
returns its outputs as arrays.  Where oracle/_ref was built the function runs and the test compares against the full
arrays.  Elsewhere the outputs come from tests/golden/reference/<name>.npz: small arrays whole, larger ones as a fixed,
seeded sample of 384 rows (pixels, texels, ...) plus the SHA-256 of the whole array; a sample is stored as byte planes
(all first bytes, then all second bytes, ...), which compresses float data better.  Tolerance checks then run on the
sample (`pick` draws the same rows from the test's own array) and bit-exact checks on the digest (`same`).  On 384 rows
the parity tolerance (<= 0.1 % decision-flipped pixels) admits none: the sampled check is the stricter one.

    VPT_RECORD_REFERENCE=DIR python -m pytest -m gpu tests      # on a GPU, with oracle/_ref built: (re)writes DIR/<name>.npz
"""
import hashlib
import json
import os

import numpy as np

import oracle_ref

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference")
ROWS = 384
WHOLE_BYTES = 16384          # arrays up to this size are stored whole


def _numpy(v):
    if hasattr(v, "detach"):
        v = v.detach().cpu().numpy()
    return np.array(v)


def _rows_of(a):
    """(rows, channels) view: a trailing axis of at most 4 is a channel axis, anything else is flattened."""
    return a.reshape(-1, a.shape[-1]) if a.ndim >= 2 and a.shape[-1] <= 4 else a.reshape(-1)


def _sample_rows(n):
    """The rows a recording keeps of an array with n rows: fixed by n alone, so they are recomputed rather than stored."""
    return np.sort(np.random.RandomState(0).choice(n, min(ROWS, n), replace=False))


def _to_planes(a):
    return np.ascontiguousarray(np.moveaxis(a.view(np.uint8).reshape(a.shape + (a.dtype.itemsize,)), -1, 0))


def _from_planes(planes, dtype):
    return np.ascontiguousarray(np.moveaxis(planes, 0, -1)).view(dtype).reshape(planes.shape[1:])


def _digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


class Outputs:
    def __init__(self, name, compute, live, exact=(), live_only=()):
        self.name, self.live, self.exact, self.live_only = name, live, exact, live_only
        if live:
            self.full = {k: _numpy(v) for k, v in compute().items()}
            out = os.environ.get("VPT_RECORD_REFERENCE")
            if out:
                self._save(os.path.join(out, name + ".npz"))
        else:
            with np.load(os.path.join(GOLD, name + ".npz")) as z:
                self.stored = {k: z[k] for k in z.files}
            self.meta = json.loads(str(self.stored.pop("meta")))
            for k, m in self.meta.items():
                if k in self.stored:
                    self.stored[k] = _from_planes(self.stored[k], m["dtype"])

    def _save(self, path):
        os.makedirs(os.path.dirname(path), exist_ok=True)
        d, meta = {}, {}
        for k, a in self.full.items():
            if k in self.live_only:
                continue
            if a.nbytes <= WHOLE_BYTES and k not in self.exact:
                d[k] = a
                continue
            meta[k] = dict(shape=list(a.shape), dtype=a.dtype.str, sha256=_digest(a))
            if k not in self.exact:
                flat = _rows_of(a)
                d[k] = _to_planes(np.ascontiguousarray(flat[_sample_rows(len(flat))]))
        np.savez_compressed(path, meta=np.array(json.dumps(meta, sort_keys=True)), **d)

    def _sampled(self, k):
        return k in self.meta

    def want(self, k):
        """The reference's array: whole when live or small, else its stored sample."""
        return self.full[k] if self.live else self.stored[k]

    def pick(self, k, got):
        """The test's own array, reduced to the rows that `want(k)` holds."""
        got = _numpy(got)
        if self.live or not self._sampled(k):
            return got
        assert list(got.shape) == self.meta[k]["shape"], f"{self.name}:{k}: shape {got.shape} differs from the recorded one"
        flat = _rows_of(got)
        return flat[_sample_rows(len(flat))]

    def same(self, k, got):
        """Bit-exact equality with the reference's whole array."""
        got = _numpy(got)
        if self.live or not self._sampled(k):
            want = self.want(k)
            return got.shape == want.shape and got.dtype == want.dtype and got.tobytes() == want.tobytes()
        return list(got.shape) == self.meta[k]["shape"] and _digest(got) == self.meta[k]["sha256"]


def load(request, compute, live=None, exact=(), live_only=()):
    """Outputs of the reference for this test (named after the test id), live where oracle/_ref exists.  The arrays named in
    `exact` are only ever compared bit for bit: their recording keeps the digest and no sample.  Those named in `live_only`
    are compared only live (their inputs exist only with oracle/_ref) and are not recorded."""
    return Outputs(request.node.name, compute, oracle_ref.available() if live is None else live, exact, live_only)
