"""Compact storage of the reference-executed fixtures: written by make_golden.py and
make_golden_options.py, read by tests/conftest.py.  No import of the reference.

Three kinds of entries, so that a file stays far below 1 MB without dropping a case or an element:
  * seeded inputs are not stored.  Each is kept as the torch recipe that drew it (make_input / randn /
    rand below) and a digest of its bytes; load() draws it again and checks the digest, so a torch whose
    CPU generator draws something else fails loudly instead of testing other inputs.
  * the per-element outputs the tests compare bit for bit (DIGESTED) are kept as a digest of their bytes,
    dtype and shape; test_oracle_golden.eq() compares a computed array against it, every element included.
  * everything else (per-bucket state, points, outputs compared within a tolerance) is stored as is.
"""
import hashlib

import numpy as np
import torch

DIGESTED = frozenset(("q", "xhat", "idx", "idx_rint", "inv_out", "q_nearest", "idx_nearest", "q_midpoint", "idx_midpoint",
                      "q_midpoint2", "idx_midpoint2"))


def make_input(kind, n, seed):
    g = torch.Generator().manual_seed(seed)
    if kind == "weights":
        return torch.randn(n, generator=g) * 0.05
    if kind == "uniform":
        return torch.rand(n, generator=g) * 2 - 1
    if kind == "constant":
        return torch.full((n,), 0.125)
    if kind == "ties":
        # bucket-wise values that land x_hat*S exactly on .5 for S=15 and S=3:
        # x in {0, 1/30, 3/30, ..., 1} scaled so min=0, max=1 inside each bucket.
        base = torch.tensor([0.0, 1.0] + [(2 * k + 1) / 30.0 for k in range(15)] + [(2 * k + 1) / 6.0 for k in range(3)])
        reps = (n + base.numel() - 1) // base.numel()
        return base.repeat(reps)[:n].clone()
    if kind == "mixed_scale":
        x = torch.randn(n, generator=g)
        scale = torch.logspace(-6, 3, n)
        return x * scale
    raise ValueError(kind)


def draw(recipe):
    """recipe = (op, kind, n, seed): op 'input' is make_input(kind, n, seed); 'randn' / 'rand' are n standard normal /
    uniform [0, 1) floats from a CPU generator seeded with seed (kind unused)."""
    op, kind, n, seed = recipe
    if op == "input":
        t = make_input(kind, n, seed)
    elif op in ("randn", "rand"):
        t = getattr(torch, op)(n, generator=torch.Generator().manual_seed(seed))
    else:
        raise ValueError(op)
    return t.numpy()


def _canonical(a):
    a = np.ascontiguousarray(a)
    return a.astype(np.int64) if a.dtype.kind in "iub" else a      # integer results compare by value, floats by bit pattern


def digest(a):
    a = _canonical(a)
    return hashlib.blake2b(a.dtype.str.encode() + a.tobytes(), digest_size=16).hexdigest()


class Digest:
    """Stands for a stored array by its shape, dtype and digest."""

    def __init__(self, key, dtype, shape, hexdigest):
        self.key, self.dtype, self.shape, self.hexdigest = key, np.dtype(dtype), tuple(shape), hexdigest

    def reshape(self, *shape):
        shape = shape[0] if len(shape) == 1 and isinstance(shape[0], (tuple, list)) else shape
        return Digest(self.key, self.dtype, np.empty(self.shape, np.bool_).reshape(shape).shape, self.hexdigest)

    def matches(self, a):
        a = np.asarray(a)
        return a.shape == self.shape and (a.dtype == self.dtype or (a.dtype.kind in "iub" and self.dtype.kind in "iub")) \
            and digest(a) == self.hexdigest


def _suffix(key):
    return key.split("_", 1)[1]


def save(path, arrays, recipes, meta):
    """arrays: every array the reference produced or consumed, by key; recipes: key -> recipe of the seeded inputs."""
    stored, rec, dig = {}, [], []
    for key, a in arrays.items():
        a = np.asarray(a)
        if key in recipes:
            again = draw(recipes[key])
            assert again.dtype == a.dtype and np.array_equal(again.reshape(-1).view(np.uint8), a.reshape(-1).view(np.uint8)), key
            rec.append("|".join([key] + [str(v) for v in recipes[key]] + [a.dtype.str, ",".join(map(str, a.shape)), digest(a)]))
        elif _suffix(key) in DIGESTED:
            dig.append("|".join([key, a.dtype.str, ",".join(map(str, a.shape)), digest(a)]))
        else:
            stored[key] = a
    np.savez_compressed(path, meta=np.array(["|".join(str(v) for v in m) for m in meta]), recipes=np.array(rec),
                        digests=np.array(dig), **stored)


def _shape(s):
    return tuple(int(v) for v in s.split(",") if v)


class Fixture:
    """Read side of save(): fixture[key] is an ndarray (stored or drawn again) or a Digest; .files lists every key."""

    def __init__(self, path):
        self._npz = np.load(path)
        self._recipes, self._digests, self._drawn = {}, {}, {}
        for row in self._npz["recipes"]:
            key, op, kind, n, seed, dtype, shape, hexdigest = str(row).split("|")
            self._recipes[key] = ((op, kind, int(n), int(seed)), np.dtype(dtype), _shape(shape), hexdigest)
        for row in self._npz["digests"]:
            key, dtype, shape, hexdigest = str(row).split("|")
            self._digests[key] = Digest(key, dtype, _shape(shape), hexdigest)
        self.files = [k for k in self._npz.files if k not in ("recipes", "digests")] + list(self._recipes) + list(self._digests)

    def __contains__(self, key):
        return key in self.files

    def __getitem__(self, key):
        if key in self._digests:
            return self._digests[key]
        if key in self._recipes:
            if key not in self._drawn:
                recipe, dtype, shape, hexdigest = self._recipes[key]
                a = draw(recipe).astype(dtype, copy=False).reshape(shape)
                assert digest(a) == hexdigest, f"{key}: torch's CPU generator no longer draws the input the reference saw"
                self._drawn[key] = a
            return self._drawn[key]
        return self._npz[key]


def load(path):
    return Fixture(path)
