"""Stored results of the reference implementation's own CUDA kernels, for the parity tests.

The parity tests compare this package with what the reference's kernels (re-hosted by oracle/refhost.py) computed on
the same seeded inputs.  Those kernels can only be compiled where the reference's source tree is present, so their
results are kept under tests/golden/ref/ as one digest per test case.  Per tensor a digest holds
  shape, sha      (in the JSON entry "meta", with absmax) the SHA-256 of its bytes (-0.0 read as 0.0): bit-exact
                  comparisons,
  absmax          its largest magnitude, the denominator of the relative error,
  whole           the tensor itself, when it has at most WHOLE elements (or the test asks for it);
otherwise
  sketch          for each of SKETCH_BLOCKS runs of consecutive elements, the sum of the elements with fixed
                  pseudo-random signs: every element of the tensor enters one sum, so an error in any one element
                  (any batch item, any face) moves that sum by the error itself;
  idx, val        the TOP largest-magnitude elements;
and for tensors checked per element (`per_element`), the components above 1e-3 of the maximum:
  big, bigval     all of them, when there are at most BIG_WHOLE: their positions (a bit mask) and their values over
                  the maximum in float16 (relative rounding <= 2^-11, which per_element() adds to its error bound),
  idx, val        otherwise a fixed, seeded sample of PER_ELEMENT of them, in float32.

NR_REF_GOLDEN_RECORD=<dir> re-records: the tests then run the reference kernels (oracle/_ref must have been built)
and write the digests into <dir>, which are then copied to tests/golden/ref/.
"""
import hashlib
import json
import os

import numpy as np

from helpers import rel_err

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref")
RECORD_DIR = os.environ.get("NR_REF_GOLDEN_RECORD")
WHOLE = 8192
SKETCH_BLOCKS = 1024
TOP = 64
PER_ELEMENT = 2048
BIG_WHOLE = 16384
F16_EPS = 2.0 ** -11


def _np(a):
    if hasattr(a, "detach"):
        a = a.detach().cpu().numpy()
    return np.ascontiguousarray(a)


def _sha(a):
    if a.dtype.kind == "f":
        a = a + a.dtype.type(0)  # -0.0 -> 0.0: torch.equal does not tell them apart either
        nan = np.isnan(a)
        if nan.any():
            a[nan] = np.nan  # one NaN payload (the GPU's and x86's differ)
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def _sketch(a):
    """signed sums of SKETCH_BLOCKS runs of consecutive elements of `a` (float64); the sign of element i is a bit of
    a multiplicative hash of i, so it does not depend on any random number generator's stream"""
    flat = a.reshape(-1)
    i = np.arange(flat.size, dtype=np.uint32)
    i *= np.uint32(2654435761)  # modulo 2^32
    signed = np.where((i >> np.uint32(15)) & np.uint32(1), -flat, flat)
    starts = (np.arange(min(SKETCH_BLOCKS, flat.size), dtype=np.int64) * flat.size) // min(SKETCH_BLOCKS, flat.size)
    return np.add.reduceat(signed, starts, dtype=np.float64)


class RefGolden:
    """Digests of one test case.  `recording`: the caller runs the reference and `put`s its tensors."""

    def __init__(self, key):
        self.key = key
        self.recording = bool(RECORD_DIR)
        self.meta, self.d = {}, {}
        if not self.recording:
            with np.load(os.path.join(GOLDEN_DIR, key + ".npz")) as z:
                self.d = {k: z[k] for k in z.files if k != "meta"}
                self.meta = json.loads(str(z["meta"]))

    def put(self, name, a, exact_only=False, whole=False, per_element=False):
        """Record tensor `a`.  `exact_only`: only bit-exact comparisons are made with it; `whole`: store it whole
        however large; `per_element`: it is used with per_element(), so its components above 1e-3 of the
        maximum are stored (all of them, or a sample when there are more than BIG_WHOLE)."""
        a = _np(a)
        flat = a.reshape(-1)
        d = self.d
        absmax = float(np.abs(flat.astype(np.float64)).max()) if flat.size else 0.0
        self.meta[name] = {"shape": list(a.shape), "sha": _sha(a), "absmax": absmax}
        if exact_only:
            return
        if whole or flat.size <= WHOLE:
            d[name + ".whole"] = a
            return
        d[name + ".sketch"] = _sketch(a).astype(np.float32)
        if per_element:
            mask = np.abs(flat) > 1e-3 * absmax
            big = np.flatnonzero(mask)
            if big.size <= BIG_WHOLE:
                d[name + ".big"] = np.packbits(mask)
                d[name + ".bigval"] = (flat[big].astype(np.float64) / absmax).astype(np.float16)
                nz = np.flatnonzero(flat)
                idx = nz[np.argpartition(np.abs(flat[nz]), -TOP)[-TOP:]]
            else:
                idx = np.random.default_rng(0).choice(big, PER_ELEMENT, replace=False)
        else:
            nz = np.flatnonzero(flat)
            idx = nz[np.argpartition(np.abs(flat[nz]), -TOP)[-TOP:]] if nz.size > TOP else nz
        idx = np.unique(idx)
        d[name + ".idx"] = idx.astype(np.int32)
        d[name + ".val"] = flat[idx]

    def save(self):
        if self.recording:
            os.makedirs(RECORD_DIR, exist_ok=True)
            np.savez_compressed(os.path.join(RECORD_DIR, self.key + ".npz"), meta=np.array(json.dumps(self.meta)),
                                **self.d)

    def __contains__(self, name):
        return name in self.meta

    def shape(self, name):
        return tuple(self.meta[name]["shape"])

    def absmax(self, name):
        return float(self.meta[name]["absmax"])

    def equal(self, name, got):
        """bit-exact (up to the sign of zero) with the reference tensor"""
        got = _np(got)
        return got.shape == self.shape(name) and _sha(got) == self.meta[name]["sha"]

    def dense(self, name):
        """the whole reference tensor (only for tensors stored whole)"""
        return self.d[name + ".whole"]

    def rel_err(self, name, got):
        """max-abs-error / max-abs-reference.  Stored whole: over every element.  Otherwise the larger of the
        error over the largest elements and the largest change of a signed block sum (an error in any one element
        shows there undiminished; the float32 rounding of the stored sums, <= 6e-8 of each sum, is subtracted)."""
        got = _np(got)
        assert got.shape == self.shape(name), (name, got.shape, self.shape(name))
        if name + ".whole" in self.d:
            return rel_err(got, self.dense(name))
        if not np.isfinite(got).all():
            return float("inf")  # a NaN would vanish from max() below
        den = self.absmax(name)
        idx, val = self.d[name + ".idx"], self.d[name + ".val"].astype(np.float64)
        err = np.abs(got.reshape(-1)[idx].astype(np.float64) - val).max() if idx.size else 0.0
        ref_sums = self.d[name + ".sketch"].astype(np.float64)
        moved = np.abs(_sketch(got) - ref_sums) - np.abs(ref_sums) * 2.0 ** -24
        return float(max(err, moved.max()) / den)

    def per_element(self, name, got, floor=1e-3):
        """max relative error over the components whose magnitude exceeds `floor` x the tensor maximum (all of them,
        unless only a sample was stored), and how many were compared"""
        got = _np(got).reshape(-1).astype(np.float64)
        if name + ".big" in self.d:
            assert floor == 1e-3, floor
            idx = np.flatnonzero(np.unpackbits(self.d[name + ".big"], count=got.size))
            approx = self.d[name + ".bigval"].astype(np.float64) * self.absmax(name)
            # |ref - approx| <= F16_EPS |ref|: a bound on the error against the reference itself
            err = np.abs(got[idx] - approx) * (1 + F16_EPS) / np.abs(approx) + F16_EPS
            return float(err.max()), int(idx.size)
        if name + ".whole" in self.d:
            idx = np.arange(got.size)
            val = self.dense(name).reshape(-1).astype(np.float64)
        else:
            idx, val = self.d[name + ".idx"], self.d[name + ".val"].astype(np.float64)
        big = np.abs(val) > floor * self.absmax(name)
        return float((np.abs(got[idx] - val)[big] / np.abs(val)[big]).max()), int(big.sum())
