"""Generates tests/golden/reference_vectors_options.npz: the UNMODIFIED reference
(antspy/quantized_distillation, mounted at /root/reference) run with the options only its NMT
loop passes (translation_models/model.py:162-164, 198-204) -- ``subtract_mean``, ``max_element``
and ``stochastic_rounding``.  Companion of make_golden.py (whose fixture file stays byte-stable);
run in the build container only:

    python tests/golden/make_golden_options.py

What is executed:
  * quantization.uniformQuantization(..., subtract_mean / max_element)          (quant_functions.py:63-74, 155-194)
  * quantization.ScalingFunction.scale_down / inv_scale_down with the options     (:56-152)
  * quantization.nonUniformQuantization (direct path) with the options           (:196-290)
  * quantization.uniformQuantization(..., stochastic_rounding=True), alone and with the pre-ops (:174-187).
    The reference draws ``torch.rand(tensor.size())`` from torch's default CPU generator; the
    generator is seeded right before the call and the same draw is repeated afterwards, so the stored
    ``u`` is exactly the array the reference compared against -- which pins the deterministic part of
    stochastic rounding (floor, fraction, ``u <= frac`` with equality, the 1/s bump, padded layout).
"""
import os
import sys
import warnings

import numpy as np
import torch

REF = "/root/reference"
sys.path.insert(0, REF)
warnings.filterwarnings("ignore")
import quantization as Q  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from golden_store import make_input, save  # noqa: E402  (same seeded input families)

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_vectors_options.npz")


def option_sets(kind):
    m = {"weights": 0.05, "uniform": 0.5, "mixed_scale": 2.0}[kind]
    return [(True, False), (False, m), (True, m * 0.6), (False, m * 100.0)]      # last: a clamp that clamps nothing


def expected_size(n, b):
    if b is None:
        return (n,)
    if n < b:
        return (1, n)
    return (-(-n // b), b)


def main():
    store, recipes, meta = {}, {}, []       # recipes: seeded inputs, redrawn at load time (golden_store.py)

    def put(k, v):
        store[k] = np.array(v, copy=True)

    # ---------------- pre-ops: uniform forward, scaling state, inverse ----------------
    ci = 0
    for kind in ("weights", "uniform", "mixed_scale"):
        for n in (10, 257, 1000, 2049):
            for b in (256, None, 64):
                for s in (4, 16):
                    if kind == "mixed_scale" and (b == 64 or s == 4):
                        continue
                    for sub, mx in option_sets(kind):
                        x = make_input(kind, n, 8000 + ci)
                        q, sf = Q.uniformQuantization(x, s, bucket_size=b, subtract_mean=sub, max_element=mx)
                        key = f"o{ci}"
                        put(key + "_x", x.numpy())
                        recipes[key + "_x"] = ("input", kind, n, 8000 + ci)
                        put(key + "_q", q.numpy())
                        put(key + "_alpha", sf.alpha.reshape(-1).numpy())
                        put(key + "_beta", sf.beta.reshape(-1).numpy())
                        put(key + "_argmin", sf.idx_min_rows.reshape(-1).numpy())
                        put(key + "_argmax", sf.idx_max_rows.reshape(-1).numpy())
                        put(key + "_mean", np.array([float(sf.mean_tensor)], dtype=np.float32))
                        sf2 = Q.ScalingFunction("linear", mx, sub, b, False)
                        xh = sf2.scale_down(x)
                        put(key + "_xhat", xh.reshape(-1).numpy())
                        if s == 16:                                  # inverse scaling (with the mean added back, :148)
                            y = torch.rand(xh.size(), generator=torch.Generator().manual_seed(11 + ci))
                            put(key + "_inv_in", y.reshape(-1).numpy())
                            recipes[key + "_inv_in"] = ("rand", "-", y.numel(), 11 + ci)
                            put(key + "_inv_out", sf2.inv_scale_down(y).reshape(-1).numpy())
                        meta.append(("pre_uniform", key, kind, n, -1 if b is None else b, s, int(sub), repr(float(mx)) if mx is not False else "no"))
                        ci += 1

    # ---------------- pre-ops: non-uniform direct path ----------------
    ci = 0
    for kind in ("weights", "uniform"):
        for n in (257, 2049):
            for b in (256, None):
                for K in (4, 16):
                    for sub, mx in option_sets(kind)[:3]:
                        x = make_input(kind, n, 9000 + ci)
                        pts = torch.linspace(0, 1, K)
                        q, idx, sf = Q.nonUniformQuantization(x, pts, bucket_size=b, subtract_mean=sub, max_element=mx)
                        key = f"v{ci}"
                        put(key + "_x", x.numpy())
                        recipes[key + "_x"] = ("input", kind, n, 9000 + ci)
                        put(key + "_points", pts.numpy())
                        put(key + "_q", q.numpy())
                        put(key + "_idx", idx.numpy())
                        put(key + "_mean", np.array([float(sf.mean_tensor)], dtype=np.float32))
                        meta.append(("pre_nonuniform", key, kind, n, -1 if b is None else b, K, int(sub), repr(float(mx)) if mx is not False else "no"))
                        ci += 1

    # ---------------- stochastic rounding with the reference's own draws ----------------
    ci = 0
    for kind in ("weights", "uniform"):
        for n in (10, 256, 1000, 2049):
            for b in (256, None, 64):
                for s in (4, 16, 256):
                    for sub, mx in ((False, False), (True, {"weights": 0.04, "uniform": 0.4}[kind])):
                        if (sub or mx) and (s == 256 or b == 64):
                            continue
                        x = make_input(kind, n, 10000 + ci)
                        torch.manual_seed(77000 + ci)
                        q, sf = Q.uniformQuantization(x, s, bucket_size=b, stochastic_rounding=True, subtract_mean=sub, max_element=mx)
                        torch.manual_seed(77000 + ci)
                        u = torch.rand(expected_size(n, b))          # the draw the reference just made (:185)
                        key = f"r{ci}"
                        put(key + "_x", x.numpy())
                        put(key + "_u", u.reshape(-1).numpy())
                        recipes[key + "_x"], recipes[key + "_u"] = ("input", kind, n, 10000 + ci), ("rand", "-", u.numel(), 77000 + ci)
                        put(key + "_q", q.numpy())
                        put(key + "_mean", np.array([float(sf.mean_tensor)], dtype=np.float32))
                        meta.append(("stochastic", key, kind, n, -1 if b is None else b, s, int(sub), repr(float(mx)) if mx is not False else "no"))
                        ci += 1

    save(OUT, store, recipes, meta)
    print("wrote", OUT, os.path.getsize(OUT) // 1024, "KiB;", len(meta), "cases; torch", torch.__version__, "numpy", np.__version__)


if __name__ == "__main__":
    main()
