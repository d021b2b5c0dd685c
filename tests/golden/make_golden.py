"""Generates tests/golden/reference_vectors.npz by running the UNMODIFIED
reference (antspy/quantized_distillation, mounted at /root/reference) on seeded
inputs.  Run in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

The reference has no tests of its own (SURVEY.md section 4), so these vectors
-- outputs of the reference's own code -- are what pins the oracle
(oracle/quant_oracle.py) and, through it, the CUDA path.

What is executed:
  * quantization.uniformQuantization            (quant_functions.py:155-194)
  * quantization.ScalingFunction.scale_down / inv_scale_down   (:56-152)
  * quantization.nonUniformQuantization, direct path           (:196-290)
  * quantization.nonUniformQuantization_variable fwd/bwd with
    pre_process_tensors=True (SearchSorted path)               (:408-573)
  * quantization.uniformQuantization_variable.backward for single-bucket
    inputs: the reference builds the correction vector with torch.mm (:398-400)
    and then fails on a shape bug; torch.mm is wrapped to capture the vector it
    produced, so the stored gradient is g + (the reference's own mm result).
  * quantization.help_functions.initialize_quantization_points (:140-154)
  * quantization.help_functions.get_huffman_encoding_mean_bit_length (:175-232)
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
import quantization.help_functions as QH  # noqa: E402

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from golden_store import make_input, save  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_vectors.npz")


def uniform_cases():
    cases = []
    for kind in ("weights", "uniform"):
        for n in (1, 10, 255, 256, 257, 1000, 4099):
            for b in (256, None, 64):
                for s in (4, 16, 256):
                    cases.append((kind, n, b, s))
    for kind in ("constant", "ties", "mixed_scale"):
        for n in (18, 300, 2048):
            for b in (256, None, 18):
                for s in (4, 16):
                    cases.append((kind, n, b, s))
    cases.append(("weights", 3 * 5 * 7 * 11, 100, 8))      # odd bucket, odd s
    cases.append(("weights", 40000, 1024, 16))
    cases.append(("weights", 40001, 4096, 2))
    return cases


def main():
    class _CopyStore(dict):
        def __setitem__(self, k, v):            # .numpy() aliases torch storage: snapshot now
            super().__setitem__(k, np.array(v, copy=True))
    store = _CopyStore()
    recipes = {}                                 # seeded inputs: redrawn at load time (golden_store.py)
    meta = []

    # ---------------- uniform forward + scaling state -----------------------
    for ci, (kind, n, b, s) in enumerate(uniform_cases()):
        x = make_input(kind, n, 1000 + ci)
        q, sf = Q.uniformQuantization(x, s, bucket_size=b)
        key = f"u{ci}"
        store[key + "_x"] = x.numpy()
        recipes[key + "_x"] = ("input", kind, n, 1000 + ci)
        store[key + "_q"] = q.numpy()
        store[key + "_alpha"] = sf.alpha.reshape(-1).numpy()
        store[key + "_beta"] = sf.beta.reshape(-1).numpy()
        store[key + "_argmin"] = sf.idx_min_rows.reshape(-1).numpy()
        store[key + "_argmax"] = sf.idx_max_rows.reshape(-1).numpy()
        # integer levels the way the reference recovers them (help_functions.py:213-218)
        sf2 = Q.ScalingFunction("linear", False, False, b, False)
        xh = sf2.scale_down(x)
        store[key + "_xhat"] = xh.reshape(-1).numpy()
        lv = np.rint(xh.reshape(-1).numpy() * np.float32(s - 1))[:n]
        qs = sf.scale_down(q.clone()).view(-1)[0:n].numpy()  # sf has modify_in_place=True
        dig = np.digitize(qs, [k / (s - 1) - 1e-5 for k in range(s)]) - 1
        store[key + "_idx"] = dig.astype(np.int64)
        store[key + "_idx_rint"] = lv.astype(np.int64)
        # inverse scaling of an arbitrary row tensor
        y = torch.rand(xh.size(), generator=torch.Generator().manual_seed(7 + ci))
        store[key + "_inv_in"] = y.reshape(-1).numpy()
        recipes[key + "_inv_in"] = ("rand", "-", y.numel(), 7 + ci)
        store[key + "_inv_out"] = sf2.inv_scale_down(y).reshape(-1).numpy()
        meta.append(("uniform", key, kind, n, -1 if b is None else b, s))

    # ---------------- 'complicated' backward, single bucket -----------------
    orig_mm = torch.mm
    for ci, (n, b, s) in enumerate([(200, 256, 16), (256, 256, 16), (256, 256, 4), (100, 128, 256),
                                    (64, 64, 16), (1000, 1024, 4), (37, 64, 8)]):
        x = make_input("weights", n, 2000 + ci)
        g = torch.randn(n, generator=torch.Generator().manual_seed(3000 + ci))
        f = Q.uniformQuantization_variable(s, bucket_size=b)
        f.forward(x)
        cap = {}

        def mm(a, bb):
            r = orig_mm(a, bb)
            cap["r"] = r
            return r
        torch.mm = mm
        try:
            f.backward(g)
        except RuntimeError:
            pass                                   # the known shape bug at :398-402
        finally:
            torch.mm = orig_mm
        key = f"c{ci}"
        store[key + "_x"] = x.numpy()
        store[key + "_g"] = g.numpy()
        recipes[key + "_x"], recipes[key + "_g"] = ("input", "weights", n, 2000 + ci), ("randn", "-", n, 3000 + ci)
        store[key + "_gout"] = (g + cap["r"].view(-1)).numpy()
        meta.append(("minmax_bwd", key, "weights", n, b, s))

    # ---------------- non-uniform, both index rules --------------------------
    nu = []
    for kind in ("weights", "uniform"):
        for n in (1, 10, 256, 257, 1000, 4099):
            for b in (256, None):
                for K in (3, 4, 16):
                    nu.append((kind, n, b, K))
    nu.append(("ties", 300, 256, 4))
    nu.append(("weights", 5000, 256, 40))
    for ci, (kind, n, b, K) in enumerate(nu):
        x = make_input(kind, n, 4000 + ci)
        sf = Q.ScalingFunction("linear", False, False, b, False)
        if ci % 2 == 0 and n >= K:
            pts = QH.initialize_quantization_points(x, sf, K)
        else:
            pts = torch.linspace(0, 1, K)
        if kind == "ties":
            pts = torch.tensor([0.0, 0.2, 0.6, 1.0])   # x_hat hits exact midpoints / equidistant cases
        key = f"n{ci}"
        store[key + "_x"] = x.numpy()
        recipes[key + "_x"] = ("input", kind, n, 4000 + ci)
        store[key + "_points"] = pts.numpy()
        # direct path = nearest rule
        q, idx, sfn = Q.nonUniformQuantization(x, pts, bucket_size=b)
        store[key + "_q_nearest"] = q.numpy()
        store[key + "_idx_nearest"] = idx.numpy()
        store[key + "_alpha"] = sfn.alpha.reshape(-1).numpy()
        # pre-processed path = midpoint rule, plus backward
        f = Q.nonUniformQuantization_variable(bucket_size=b, pre_process_tensors=True, tensor=x)
        q2 = f.forward(None, pts)
        store[key + "_q_midpoint"] = q2.numpy()
        store[key + "_idx_midpoint"] = f.savedForBackward["indices"].numpy()
        # second query with moved points exercises the incremental update (:555-561)
        pts2 = torch.sort(pts + 0.01 * torch.randn(K, generator=torch.Generator().manual_seed(ci)))[0].clamp(0, 1)
        q3 = f.forward(None, pts2)
        store[key + "_points2"] = pts2.numpy()
        store[key + "_q_midpoint2"] = q3.numpy()
        store[key + "_idx_midpoint2"] = f.savedForBackward["indices"].numpy()
        g = torch.randn(n, generator=torch.Generator().manual_seed(5000 + ci))
        Q.USE_CUDA = False
        gi, gp = f.backward(g)
        store[key + "_g"] = g.numpy()
        recipes[key + "_g"] = ("randn", "-", n, 5000 + ci)
        store[key + "_gpoints2"] = gp.numpy()
        meta.append(("nonuniform", key, kind, n, -1 if b is None else b, K))

    # ---------------- centroid initialisation -------------------------------
    for ci, (n, b, K) in enumerate([(1000, 256, 4), (4099, 256, 16), (4099, None, 3), (10, 256, 4)]):
        x = make_input("weights", n, 6000 + ci)
        sf = Q.ScalingFunction("linear", False, False, b, False)
        pts = QH.initialize_quantization_points(x, sf, K)
        key = f"p{ci}"
        store[key + "_x"] = x.numpy()
        recipes[key + "_x"] = ("input", "weights", n, 6000 + ci)
        store[key + "_points"] = pts.numpy()
        meta.append(("init_points", key, "weights", n, -1 if b is None else b, K))

    # ---------------- Huffman mean bit length over a small "model" ----------
    for ci, (b, s) in enumerate([(256, 4), (256, 16), (None, 4)]):
        params = [make_input("weights", n, 7000 + 10 * ci + j) for j, n in enumerate((300, 1000, 4099, 10))]
        fun = lambda t, s=s, b=b: Q.uniformQuantization(t, s, bucket_size=b)  # noqa: E731
        mbl = QH.get_huffman_encoding_mean_bit_length(iter(params), fun, "uniform", s=s)
        key = f"h{ci}"
        for j, p in enumerate(params):
            store[f"{key}_x{j}"] = p.numpy()
            recipes[f"{key}_x{j}"] = ("input", "weights", p.numel(), 7000 + 10 * ci + j)
        store[key + "_mean_bits"] = np.array([mbl], dtype=np.float64)
        meta.append(("huffman", key, "weights", len(params), -1 if b is None else b, s))

    save(OUT, store, recipes, meta)
    print("wrote", OUT, os.path.getsize(OUT) // 1024, "KiB;", len(meta), "cases; torch", torch.__version__,
          "numpy", np.__version__)


if __name__ == "__main__":
    main()
