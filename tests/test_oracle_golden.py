"""Pins oracle/quant_oracle.py against outputs of the reference itself
(tests/golden/reference_vectors.npz, produced by tests/golden/make_golden.py).
Bit-exact for everything except sums the reference accumulates in float32."""
import numpy as np
from golden_store import Digest

from oracle import quant_oracle as O


def eq(a, b):
    a = np.asarray(a)
    if isinstance(b, Digest):                                       # every element, by digest (tests/golden/golden_store.py)
        assert b.matches(a), (b.key, a.shape, b.shape, a.dtype, b.dtype)
        return
    b = np.asarray(b)
    assert a.shape == b.shape, (a.shape, b.shape)
    if a.dtype.kind == "f":
        assert a.dtype == b.dtype, (a.dtype, b.dtype)
        bits = {4: np.uint32, 8: np.uint64}[a.dtype.itemsize]
        assert np.array_equal(a.view(bits), b.view(bits))          # bit pattern: +0 / -0 and NaN payloads count
    else:
        assert np.array_equal(a, b)


def test_uniform_forward_bit_exact(golden):
    data, cases = golden
    assert len(cases["uniform"]) > 150
    for c in cases["uniform"]:
        k = c["key"]
        x = data[k + "_x"]
        q, idx, st = O.uniform_fwd(x, c["s"], c["bucket"])
        eq(q, data[k + "_q"])
        eq(st["alpha"], data[k + "_alpha"])
        eq(st["beta"], data[k + "_beta"])
        eq(st["argmin"], data[k + "_argmin"])
        eq(st["argmax"], data[k + "_argmax"])
        eq(idx.reshape(-1), data[k + "_idx_rint"])
        # the reference's own index recovery (np.digitize on the re-scaled q with its 1e-5 slack,
        # help_functions.py:213-218) gives the same integer level on EVERY element of every case
        # (229,548 elements, incl. the constant and mixed-scale buckets): no exemptions
        eq(idx.reshape(-1).astype(np.int64), data[k + "_idx"])                  # integer digests compare by value


def test_scale_down_and_inverse_bit_exact(golden):
    data, cases = golden
    for c in cases["uniform"]:
        k = c["key"]
        xh, st = O.scale_down(data[k + "_x"], c["bucket"])
        eq(xh.reshape(-1), data[k + "_xhat"])
        y = data[k + "_inv_in"].reshape(xh.shape)
        eq(O.inv_scale_down(y, st).reshape(-1), data[k + "_inv_out"])


def test_minmax_backward_matches_reference_mm(golden):
    data, cases = golden
    for c in cases["minmax_bwd"]:
        k = c["key"]
        gout, info = O.uniform_bwd_minmax(data[k + "_x"], data[k + "_g"], c["s"], c["bucket"])
        ref = data[k + "_gout"]
        # positions: identical; values: float32 mm sum vs float64 sum
        changed_ref = np.nonzero(ref != data[k + "_g"])[0]
        changed = np.nonzero(gout != data[k + "_g"])[0]
        assert np.array_equal(changed, changed_ref)
        scale = np.abs(data[k + "_g"]).sum() / c["s"]
        assert np.abs(gout.astype(np.float64) - ref).max() <= 1e-6 * scale + 1e-7


def test_nonuniform_both_rules_bit_exact(golden):
    data, cases = golden
    for c in cases["nonuniform"]:
        k = c["key"]
        x = data[k + "_x"]
        pts = data[k + "_points"]
        q, idx, st = O.nonuniform_fwd(x, pts, c["bucket"], rule="nearest")
        eq(idx, data[k + "_idx_nearest"])
        eq(q, data[k + "_q_nearest"])
        q, idx, st = O.nonuniform_fwd(x, pts, c["bucket"], rule="midpoint")
        eq(idx, data[k + "_idx_midpoint"])
        eq(q, data[k + "_q_midpoint"])
        q, idx, st = O.nonuniform_fwd(x, data[k + "_points2"], c["bucket"], rule="midpoint")
        eq(idx, data[k + "_idx_midpoint2"])
        eq(q, data[k + "_q_midpoint2"])
        eq(st["alpha"], data[k + "_alpha"])
        gp = O.nonuniform_bwd_points(data[k + "_g"], idx, st["alpha"], pts.size, c["bucket"])
        ref = data[k + "_gpoints2"].astype(np.float64)
        a_rep = np.abs(data[k + "_g"]).astype(np.float64).sum() * float(st["alpha"].max())
        assert np.abs(gp - ref).max() <= 1e-6 * a_rep + 1e-12


def test_points_initialisation(golden):
    data, cases = golden
    for c in cases["init_points"]:
        k = c["key"]
        eq(O.initialize_points(data[k + "_x"], c["bucket"], c["s"]), data[k + "_points"])


def test_huffman_mean_bit_length(golden):
    data, cases = golden
    for c in cases["huffman"]:
        k = c["key"]
        counts = np.zeros(c["s"], dtype=np.int64)
        for j in range(c["n"]):
            _, idx, _ = O.uniform_fwd(data[f"{k}_x{j}"], c["s"], c["bucket"])
            counts += np.bincount(idx.reshape(-1), minlength=c["s"])
        assert abs(O.huffman_mean_bit_length(counts) - float(data[k + "_mean_bits"][0])) < 1e-9


def test_bucket_geometry_edges():
    assert O.bucket_geometry(10, 256) == (1, 10, 10)
    assert O.bucket_geometry(256, 256) == (1, 256, 256)
    assert O.bucket_geometry(257, 256) == (2, 256, 512)
    assert O.bucket_geometry(1000, None) == (1, 1000, 1000)
    assert O.bucketed(np.arange(5, dtype=np.float32), 2).tolist() == [[0, 1], [2, 3], [4, 4]]


def test_torch_chain_matches_golden(golden):
    """oracle/torch_chain.py (the CPU baseline that is timed) is the same
    function as the reference, bit for bit, on every golden case."""
    import torch
    from oracle import torch_chain as T
    data, cases = golden
    for c in cases["uniform"]:
        k = c["key"]
        q, st = T.uniform_fwd(torch.from_numpy(data[k + "_x"].copy()), c["s"], c["bucket"])
        eq(q.numpy(), data[k + "_q"])
        eq(st.alpha.reshape(-1).numpy(), data[k + "_alpha"])
    for c in cases["nonuniform"]:
        k = c["key"]
        x = torch.from_numpy(data[k + "_x"].copy())
        pts = torch.from_numpy(data[k + "_points"].copy())
        q, idx, st = T.nonuniform_fwd(x, pts, c["bucket"], "nearest")
        eq(q.numpy(), data[k + "_q_nearest"])
        eq(idx.numpy(), data[k + "_idx_nearest"])
        q, idx, st = T.nonuniform_fwd(x, torch.from_numpy(data[k + "_points2"].copy()), c["bucket"], "midpoint")
        eq(q.numpy(), data[k + "_q_midpoint2"])
        eq(idx.numpy(), data[k + "_idx_midpoint2"])
        gp = T.nonuniform_bwd_points(torch.from_numpy(data[k + "_g"].copy()), idx, st, pts.numel(), c["bucket"])
        eq(gp.numpy(), data[k + "_gpoints2"])
    for c in cases["minmax_bwd"]:
        k = c["key"]
        gout = T.uniform_bwd_minmax(torch.from_numpy(data[k + "_x"].copy()), torch.from_numpy(data[k + "_g"].copy()),
                                    c["s"], c["bucket"])
        assert np.abs(gout.numpy() - data[k + "_gout"]).max() <= 1e-6 * np.abs(data[k + "_g"]).sum() / c["s"] + 1e-7


def test_c_oracle_matches_golden(golden):
    """oracle/quant_oracle.c (gcc, -ffp-contract=off) reproduces the reference bit for bit."""
    from oracle import c_oracle as CO
    data, cases = golden
    for c in cases["uniform"]:
        k = c["key"]
        q, idx, st = CO.uniform_fwd(data[k + "_x"], c["s"], c["bucket"])
        eq(q, data[k + "_q"].reshape(-1))
        eq(st["alpha"], data[k + "_alpha"])
        eq(st["argmin"], data[k + "_argmin"])
        eq(st["argmax"], data[k + "_argmax"])
        eq(idx, data[k + "_idx_rint"])
    for c in cases["nonuniform"]:
        k = c["key"]
        q, idx, st = CO.nonuniform_fwd(data[k + "_x"], data[k + "_points"], c["bucket"], "nearest")
        eq(q, data[k + "_q_nearest"].reshape(-1))
        eq(idx, data[k + "_idx_nearest"].reshape(-1))
        q, idx, st = CO.nonuniform_fwd(data[k + "_x"], data[k + "_points2"], c["bucket"], "midpoint")
        eq(q, data[k + "_q_midpoint2"].reshape(-1))
        eq(idx, data[k + "_idx_midpoint2"].reshape(-1))
        gp = CO.nonuniform_bwd_points(data[k + "_g"], idx, st["alpha"], data[k + "_points"].size, c["bucket"])
        scale = np.abs(data[k + "_g"]).astype(np.float64).sum() * float(st["alpha"].max())
        assert np.abs(gp - data[k + "_gpoints2"]).max() <= 1e-6 * scale + 1e-12
    for c in cases["minmax_bwd"]:
        k = c["key"]
        out = CO.uniform_bwd_minmax(data[k + "_x"], data[k + "_g"], c["s"], c["bucket"])
        assert np.abs(out - data[k + "_gout"]).max() <= 1e-6 * np.abs(data[k + "_g"]).sum() / c["s"] + 1e-7


# ----------------------------------------------------------------------------------------------------------------
# the options only the NMT loop passes (translation_models/model.py:162-164): fixtures of make_golden_options.py
# ----------------------------------------------------------------------------------------------------------------
def _mean_close(x, got, ref):
    """The reference's mean is a float32 torch reduction: equal to the float64 mean up to the summation order."""
    x64 = np.asarray(x, dtype=np.float64)
    assert abs(float(got) - float(ref)) <= 1e-6 * np.abs(x64).mean() + 1e-30, (float(got), float(ref))


def test_pre_ops_uniform_forward_bit_exact(golden_options):
    data, cases = golden_options
    assert len(cases["pre_uniform"]) >= 200
    clamped = 0
    for c in cases["pre_uniform"]:
        k, x = c["key"], data[c["key"] + "_x"]
        ref_mean = data[k + "_mean"][0]
        opts = dict(subtract_mean=c["subtract_mean"], max_element=c["max_element"])
        # everything downstream of the mean, bit for bit, given the reference's own mean ...
        q, idx, st = O.uniform_fwd(x, c["s"], c["bucket"], mean=ref_mean, **opts)
        eq(q, data[k + "_q"])
        eq(st["alpha"], data[k + "_alpha"])
        eq(st["beta"], data[k + "_beta"])
        eq(st["argmin"], data[k + "_argmin"])
        eq(st["argmax"], data[k + "_argmax"])
        xh, st2 = O.scale_down(x, c["bucket"], mean=ref_mean, **opts)
        eq(xh.reshape(-1), data[k + "_xhat"])
        if k + "_inv_in" in data.files:                                  # inverse adds the mean back (:148)
            eq(O.inv_scale_down(data[k + "_inv_in"].reshape(xh.shape), st2).reshape(-1), data[k + "_inv_out"])
        # ... and the oracle's own mean inside the summation-order tolerance
        if c["subtract_mean"]:
            _mean_close(x, O.pre_ops(x, True, False)[1], ref_mean)
        else:
            assert ref_mean == 0
        if c["max_element"] is not False:
            clamped += int((np.abs(x - ref_mean) > c["max_element"]).any())
    assert clamped >= 100                                                 # the clamp is active in most clamp cases


def test_pre_ops_nonuniform_direct_path_bit_exact(golden_options):
    data, cases = golden_options
    assert len(cases["pre_nonuniform"]) >= 40
    for c in cases["pre_nonuniform"]:
        k = c["key"]
        q, idx, st = O.nonuniform_fwd(data[k + "_x"], data[k + "_points"], c["bucket"], rule="nearest", mean=data[k + "_mean"][0],
                                      subtract_mean=c["subtract_mean"], max_element=c["max_element"])
        eq(idx.reshape(-1).astype(np.int64), data[k + "_idx"].reshape(-1))
        eq(q, data[k + "_q"])


def test_stochastic_rounding_given_the_reference_draws_bit_exact(golden_options):
    """quant_functions.py:174-187 with the very ``torch.rand`` array the reference drew: floor, fraction, ``u <= frac``
    (equality included), the 1/s bump and the padded layout of ``u`` are all pinned; only the draw itself is random."""
    data, cases = golden_options
    assert len(cases["stochastic"]) >= 80
    ups = total = 0
    for c in cases["stochastic"]:
        k, x, u = c["key"], data[c["key"] + "_x"], data[c["key"] + "_u"]
        q, st = O.uniform_fwd_stochastic(x, c["s"], c["bucket"], u, subtract_mean=c["subtract_mean"], max_element=c["max_element"],
                                         mean=data[k + "_mean"][0])
        eq(q, data[k + "_q"])
        # not vacuous: the rounded-up fraction is neither 0 nor 1
        det = O.uniform_fwd(x, c["s"], c["bucket"], subtract_mean=c["subtract_mean"], max_element=c["max_element"], mean=data[k + "_mean"][0])[0]
        ups += int((q != det).sum())
        total += q.size
    assert 0.1 < ups / total < 0.9
