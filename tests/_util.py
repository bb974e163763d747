import os

import numpy as np

TOL = 1e-5     # north_star: fp32 results within 1e-5 relative


def load_golden(golden_dir, name):
    p = os.path.join(golden_dir, name)
    if not os.path.exists(p):
        import pytest
        pytest.skip("golden fixture %s not generated yet" % name)
    return np.load(p)


def rel_err(a, b):
    """max |a-b| / max(|b|, tiny) elementwise-max — the parity metric of SURVEY.md §8c."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-30))) if a.size else 0.0


def scaled_err(a, b):
    """max |a-b| / max|b| — for sums whose individual terms cancel (voxel means, gradients via float atomics)."""
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-30)) if a.size else 0.0


class ReferenceOutputs:
    """What the reference's CUDA kernels return on the inputs the GPU parity tests build, kept in one small file
    (tests/golden/reference_outputs.npz) so that the parity tests need nothing outside this repository.  Only outputs the
    tests compare bit for bit are kept (indices, counts, k-NN distances, PPF, grouped features, devox corners and weights),
    each as a SHA-256 digest of the whole array plus a seeded sample of its entries (the sample only makes a failure
    readable); the inputs are regenerated from their seeds by the tests themselves.

    Recording (RI_RECORD_REFERENCE=<file.npz>) needs the reference's CUDA backend built into oracle/_ref
    (oracle/build_ref.py): every check then calls the reference on the same inputs, stores what it returns, compares ours
    with it live, and the file is written when the session ends.

    Provenance of the committed file: the reference backend is not part of this repository, and the file was taken from
    this project's kernels at commit 369b381 (unchanged since), on inputs identical to those of that commit's parity tests,
    whose live torch.equal checks against oracle/_ref on exactly these arrays passed on a B200 (188 GPU tests).  Outputs
    whose inputs changed since (voxel means, devoxelized features of random grids) are not stored: the tests check them
    against the C oracle on the cell indices and corner weights pinned here."""

    SAMPLE = 64

    def __init__(self, path, record_to=None):
        self.record_to = record_to
        self.recorded = {}
        self.backend = None
        if record_to:
            from oracle.build_ref import load_ref
            self.backend = load_ref()
            if self.backend is None:
                raise RuntimeError("recording reference outputs needs oracle/_ref/_multi_shape_pvcnn_backend.so")
            self.data = None
        else:
            self.data = dict(np.load(path))

    @staticmethod
    def _array(t):
        a = t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)
        return np.ascontiguousarray(a)

    @staticmethod
    def _digest(a):
        import hashlib
        return hashlib.sha256(a.dtype.str.encode() + repr(a.shape).encode() + a.tobytes()).hexdigest()

    @classmethod
    def _positions(cls, size, key):
        import zlib
        if size <= cls.SAMPLE:
            return np.arange(size)
        return np.sort(np.random.default_rng(zlib.crc32(key.encode())).choice(size, cls.SAMPLE, replace=False))

    def _want(self, key, suffix):
        if key + suffix not in self.data:
            raise KeyError("no stored reference output %r" % key)
        return self.data[key + suffix]

    def equal(self, key, got, call_reference):
        """Every array of `got` ({name: array}) equals the reference's bit for bit (dtype, shape, every byte).
        `call_reference(backend)` -> {name: array}, the same outputs from the reference backend; called when recording."""
        want = {n: self._array(t) for n, t in call_reference(self.backend).items()} if self.record_to else None
        for name, t in got.items():
            k = key + "/" + name if name else key
            a = self._array(t)
            flat = a.reshape(-1)
            pos = self._positions(flat.size, k)
            if self.record_to:
                w = want[name]
                self.recorded.update({k + ":shape": np.array(w.shape), k + ":sha256": np.array(self._digest(w)),
                                      k + ":val": w.reshape(-1)[self._positions(w.size, k)]})
                assert a.dtype == w.dtype and a.shape == w.shape and np.array_equal(a, w), "%s differs from the reference" % k
                continue
            shape = tuple(int(d) for d in self._want(k, ":shape"))
            val = self._want(k, ":val")
            assert a.shape == shape, "%s: shape %s, the reference returns %s" % (k, a.shape, shape)
            assert a.dtype == val.dtype, "%s: dtype %s, the reference returns %s" % (k, a.dtype, val.dtype)
            assert self._digest(a) == str(self._want(k, ":sha256")), \
                "%s differs from the reference output (%d of %d sampled entries differ)" % (k, int((flat[pos] != val).sum()), pos.size)

    def save(self):
        if self.record_to and self.recorded:
            os.makedirs(os.path.dirname(os.path.abspath(self.record_to)), exist_ok=True)
            np.savez_compressed(self.record_to, **self.recorded)
