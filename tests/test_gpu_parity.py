"""GPU parity: the CUDA path (through the C ABI / the reference-shaped Python
surface) against (1) the golden vectors produced by the reference itself and
(2) the oracle on seeded inputs.  Bit-exact for q / idx / alpha / beta /
argmin / argmax; stated tolerance only for float32 sums whose order differs."""
import numpy as np
import pytest
import torch
from golden_store import Digest

from oracle import quant_oracle as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def Q():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import quantized_distillation_b200.quantization as Q
    return Q


def bits(a):
    a = np.ascontiguousarray(np.asarray(a))
    return a.view(np.uint32) if a.dtype == np.float32 else a


def assert_same(a, b, what=""):
    if isinstance(b, Digest):                             # every element, by digest (tests/golden/golden_store.py)
        a = np.asarray(a)
        assert b.matches(a), (what, a.shape, b.shape, a.dtype, b.dtype)
        return
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if a.dtype.kind == "f":                               # NaN payload / sign bits are not part of the contract
        both_nan = np.isnan(a) & np.isnan(b)
        if both_nan.any():
            a, b = np.where(both_nan, 0, a).astype(a.dtype), np.where(both_nan, 0, b).astype(b.dtype)
    if not np.array_equal(bits(a), bits(b)):
        # -0.0 vs +0.0 can never come out of the chain, so a plain bit compare is the bar
        bad = np.nonzero(bits(a).reshape(-1) != bits(b).reshape(-1))[0]
        raise AssertionError(f"{what}: {bad.size} mismatches, first at {bad[:5]}: {a.reshape(-1)[bad[:5]]} vs {b.reshape(-1)[bad[:5]]}")


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def assert_minmax_gradient(out, g, ref, argmax, argmin, abs_sum, r, what=""):
    """a5 parity bar.  Untouched elements are bit-identical to g.  At the two positions of bucket b
    the only freedom is the ORDER of the sum r_b = sum_j v_j (float64 here, float32 torch.mm in the
    reference): |out - ref| <= 1e-6 * sum_j |v_j|  + one float32 ulp of r_b (its rounding) + one
    ulp of the result (the final add)."""
    out, g, ref = (np.asarray(a, dtype=np.float32).reshape(-1) for a in (out, g, ref))
    pos = np.concatenate([np.asarray(argmax), np.asarray(argmin)]).astype(np.int64)
    rows = np.concatenate([np.arange(len(argmax)), np.arange(len(argmin))])
    touched = np.zeros(out.size, bool)
    touched[pos] = True
    assert np.array_equal(out[~touched].view(np.uint32), g[~touched].view(np.uint32)), f"{what}: element outside argmin'/argmax' changed"
    ulp = 2.0 ** -23
    tol = 1e-6 * abs_sum[rows] + ulp * np.abs(r[rows]) + ulp * np.maximum(np.abs(ref[pos]), np.abs(g[pos])) + 1e-37
    err = np.abs(out[pos].astype(np.float64) - ref[pos].astype(np.float64))
    bad = np.nonzero(err > tol)[0]
    assert bad.size == 0, f"{what}: {bad.size} positions off, worst {err[bad].max():.3e} vs tol {tol[bad][err[bad].argmax()]:.3e}"


# ----------------------------------------------------------------------- golden vectors
def test_uniform_forward_golden(Q, golden):
    data, cases = golden
    for c in cases["uniform"]:
        k = c["key"]
        q, sf = Q.uniformQuantization(dev(data[k + "_x"]), c["s"], bucket_size=c["bucket"])
        assert_same(q.cpu().numpy(), data[k + "_q"], f"{k} q {c}")
        assert_same(sf.alpha.reshape(-1).cpu().numpy(), data[k + "_alpha"], f"{k} alpha")
        assert_same(sf.beta.reshape(-1).cpu().numpy(), data[k + "_beta"], f"{k} beta")
        assert_same(sf.idx_min_rows.reshape(-1).cpu().numpy(), data[k + "_argmin"], f"{k} argmin {c}")
        assert_same(sf.idx_max_rows.reshape(-1).cpu().numpy(), data[k + "_argmax"], f"{k} argmax")


def test_scale_down_inverse_golden(Q, golden):
    data, cases = golden
    for c in cases["uniform"]:
        k = c["key"]
        sf = Q.ScalingFunction("linear", False, False, c["bucket"], False)
        xh = sf.scale_down(dev(data[k + "_x"]))
        assert_same(xh.reshape(-1).cpu().numpy(), data[k + "_xhat"], f"{k} xhat {c}")
        y = dev(data[k + "_inv_in"]).view(xh.size())
        assert_same(sf.inv_scale_down(y).reshape(-1).cpu().numpy(), data[k + "_inv_out"], f"{k} inv")


def test_nonuniform_golden(Q, golden):
    data, cases = golden
    for c in cases["nonuniform"]:
        k = c["key"]
        x = dev(data[k + "_x"])
        pts = dev(data[k + "_points"])
        q, idx, sf = Q.nonUniformQuantization(x, pts, bucket_size=c["bucket"])
        assert idx.dtype == torch.int64
        assert_same(idx.cpu().numpy(), data[k + "_idx_nearest"], f"{k} idx nearest {c}")
        assert_same(q.cpu().numpy(), data[k + "_q_nearest"], f"{k} q nearest")
        assert_same(sf.alpha.reshape(-1).cpu().numpy(), data[k + "_alpha"], f"{k} alpha")
        f = Q.nonUniformQuantization_variable(bucket_size=c["bucket"], pre_process_tensors=True, tensor=x)
        q1 = f.forward(None, pts)
        assert_same(q1.cpu().numpy(), data[k + "_q_midpoint"], f"{k} q midpoint")
        assert_same(f.savedForBackward["indices"].cpu().numpy().astype(np.int64), data[k + "_idx_midpoint"], f"{k} idx midpoint")
        q2 = f.forward(None, dev(data[k + "_points2"]))
        assert_same(q2.cpu().numpy(), data[k + "_q_midpoint2"], f"{k} q midpoint2")
        g = dev(data[k + "_g"])
        gin, gp = f.backward(g)
        assert gin is g
        ref = data[k + "_gpoints2"].astype(np.float64)
        scale = np.abs(data[k + "_g"]).astype(np.float64).sum() * float(data[k + "_alpha"].max())
        assert np.abs(gp.cpu().numpy() - ref).max() <= 1e-6 * scale + 1e-12, (k, gp, ref)
        # the hand-driven pre-processed path of the reference docstring (:218-227)
        sfp = Q.ScalingFunction("linear", False, False, c["bucket"], False)
        sso = Q.SearchSorted(sfp.scale_down(x).view(-1))
        q3, idx3, _ = Q.nonUniformQuantization(None, pts, bucket_size=c["bucket"], pre_processed_values=True,
                                               search_sorted_obj=sso, scaling_function=sfp, tensors_info=(x.type(), True))
        assert_same(q3.cpu().numpy(), data[k + "_q_midpoint"], f"{k} q preprocessed")
        assert_same(idx3.cpu().numpy(), data[k + "_idx_midpoint"], f"{k} idx preprocessed")


def test_minmax_backward_golden(Q, golden):
    data, cases = golden
    for c in cases["minmax_bwd"]:
        k = c["key"]
        f = Q.uniformQuantization_variable(c["s"], bucket_size=c["bucket"])
        f.forward(dev(data[k + "_x"]))
        gout = f.backward(dev(data[k + "_g"])).cpu().numpy()
        ref = data[k + "_gout"]
        assert np.array_equal(np.nonzero(gout != data[k + "_g"])[0], np.nonzero(ref != data[k + "_g"])[0]), k
        scale = np.abs(data[k + "_g"]).sum() / c["s"]
        assert np.abs(gout.astype(np.float64) - ref).max() <= 1e-6 * scale + 1e-7, k


def test_points_initialisation_golden(Q, golden):
    data, cases = golden
    for c in cases["init_points"]:
        k = c["key"]
        sf = Q.ScalingFunction("linear", False, False, c["bucket"], False)
        pts = Q.help_functions.initialize_quantization_points(dev(data[k + "_x"]), sf, c["s"])
        assert_same(pts.cpu().numpy(), data[k + "_points"], k)


def test_huffman_golden(Q, golden):
    data, cases = golden
    for c in cases["huffman"]:
        k = c["key"]
        params = [dev(data[f"{k}_x{j}"]) for j in range(c["n"])]
        fun = lambda t, s=c["s"], b=c["bucket"]: Q.uniformQuantization(t, s, bucket_size=b)  # noqa: E731
        mbl = Q.help_functions.get_huffman_encoding_mean_bit_length(iter(params), fun, "uniform", s=c["s"])
        assert abs(mbl - float(data[k + "_mean_bits"][0])) < 1e-9


# ----------------------------------------------------------------------- oracle sweeps
SIZES = [1, 3, 4, 5, 31, 127, 128, 129, 255, 256, 257, 511, 512, 513, 1023, 1024, 1025, 4096, 5000, 65536 + 17, 200003]
# 1026 / 3002: rows alternate between 16-byte aligned and unaligned (bulk-copied vs ld.global-staged rows of
# the staged path inherit each other's ring slots); 12000: two-chunk rows; 49152: the shared-memory limit
BUCKETS = [None, 256, 384, 512, 768, 1024, 100, 7, 1026, 2048, 3000, 3002, 4096, 8192, 12000, 20000, 49152]


@pytest.mark.parametrize("bucket", BUCKETS)
def test_uniform_all_paths_vs_oracle(Q, bucket):
    """Every execution path: warp (vec / scalar, R=2,4,8), block (TMA-staged), grid."""
    rng = np.random.default_rng(7)
    for n in SIZES + [300001]:
        for s in (4, 16, 256):
            x = (rng.standard_normal(n) * 0.05).astype(np.float32)
            if n > 10:
                x[rng.integers(0, n, 3)] = x[0]          # duplicate extremes: first-occurrence ties
            q, idx, st = O.uniform_fwd(x, s, bucket)
            qd, sf = Q.uniformQuantization(dev(x), s, bucket_size=bucket)
            assert_same(qd.cpu().numpy(), q, f"n={n} b={bucket} s={s}")
            assert_same(sf.alpha.reshape(-1).cpu().numpy(), st["alpha"], "alpha")
            assert_same(sf.beta.reshape(-1).cpu().numpy(), st["beta"], "beta")
            assert_same(sf.idx_min_rows.reshape(-1).cpu().numpy(), st["argmin"], f"argmin n={n} b={bucket}")
            assert_same(sf.idx_max_rows.reshape(-1).cpu().numpy(), st["argmax"], "argmax")


def test_uniform_large_bucket_none_grid_path(Q):
    rng = np.random.default_rng(11)
    n = 3_000_017
    x = rng.uniform(-1, 1, n).astype(np.float32)
    q, idx, st = O.uniform_fwd(x, 16, None)
    qd, sf = Q.uniformQuantization(dev(x), 16, bucket_size=None)
    assert_same(qd.cpu().numpy(), q, "grid path q")
    assert_same(sf.idx_min_rows.cpu().numpy(), st["argmin"], "grid argmin")
    assert_same(sf.idx_max_rows.cpu().numpy(), st["argmax"], "grid argmax")


def test_unaligned_views_and_in_place(Q):
    rng = np.random.default_rng(3)
    base = dev((rng.standard_normal(5000 + 3) * 0.1).astype(np.float32))
    for off in (1, 2, 3):
        v = base[off:off + 4097]                          # 4-byte aligned only
        ref, _, _ = O.uniform_fwd(v.cpu().numpy(), 16, 256)
        q, _ = Q.uniformQuantization(v, 16, bucket_size=256)
        assert_same(q.cpu().numpy(), ref, f"offset {off}")
    t = base[:4096].clone()
    ref, _, _ = O.uniform_fwd(t.cpu().numpy(), 4, 256)
    out, _ = Q.uniformQuantization(t, 4, bucket_size=256, modify_in_place=True)
    assert out.data_ptr() == t.data_ptr()
    assert_same(t.cpu().numpy(), ref, "in place")
    # shape is preserved
    w = dev(rng.standard_normal((7, 5, 3, 3)).astype(np.float32))
    q, sf = Q.uniformQuantization(w, 16, bucket_size=256)
    assert q.shape == w.shape and sf.alpha.shape == (2, 1) and sf.idx_min_rows.dtype == torch.int64


def test_edge_inputs(Q):
    # constant bucket (alpha -> 1), exact .5 ties (round half even), denormals, huge range
    for x in (np.full(300, 0.125, np.float32),
              np.array([0.0, 1.0] + [(2 * k + 1) / 30.0 for k in range(15)], np.float32),
              np.array([0.0, 1e-40, 3e-39, 1e-38], np.float32),
              np.array([-3e38, 3e38, 1.0, 0.0], np.float32),
              np.array([1.0, 1.0 + 1e-7, 1.0 + 2e-7], np.float32)):
        for s in (4, 16):
            for b in (256, None, 2):
                with np.errstate(all="ignore"):
                    q, _, st = O.uniform_fwd(x, s, b)
                qd, sf = Q.uniformQuantization(dev(x), s, bucket_size=b)
                assert_same(qd.cpu().numpy(), q, f"edge {x[:4]} s={s} b={b}")
    # NaN propagates through the whole bucket like torch.min/max do
    x = np.arange(600, dtype=np.float32)
    x[300] = np.nan
    qd, _ = Q.uniformQuantization(dev(x), 16, bucket_size=256)
    out = qd.cpu().numpy()
    assert np.isnan(out[256:512]).all() and not np.isnan(out[:256]).any() and not np.isnan(out[512:]).any()


def test_rounding_boundary_stress(Q):
    """Inputs engineered so that x_hat*S sits on, or a few ulps around, every rounding boundary
    k+0.5: the fast level path must hand exactly these to the exact IEEE chain."""
    rng = np.random.default_rng(41)
    for s in (2, 4, 16, 256):
        S = s - 1
        for lo, span in ((0.0, 1.0), (-0.731, 0.0371), (5.0, 3.3e-5), (-100.0, 7777.7), (1e-20, 1e-21)):
            rows = []
            for _ in range(64):
                ks = (rng.integers(0, S, 254) + 0.5) / S
                jit = 1 + rng.integers(-6, 7, 254) * 2.0 ** -24
                row = lo + span * np.concatenate([[0.0, 1.0], ks * jit])
                rows.append(row)
            x = np.concatenate(rows).astype(np.float32)
            with np.errstate(all="ignore"):
                q, idx, st = O.uniform_fwd(x, s, 256)
            qd, sf = Q.uniformQuantization(dev(x), s, bucket_size=256)
            assert_same(qd.cpu().numpy(), q, f"boundary stress s={s} lo={lo} span={span}")
            from quantized_distillation_b200 import _native as N
            xd = dev(x)
            i8 = torch.empty(x.size, dtype=torch.uint8, device="cuda")
            ws = N.workspace(x.size, 256, xd.device)
            N.check(N.lib().qd_uniform_fwd(N.ptr(xd), None, N.ptr(i8), None, None, None, None, x.size, 256, s, None, 0.0, 0, 0, 0,
                                           N.ptr(ws), ws.numel(), N.stream_ptr()))
            assert_same(i8.cpu().numpy().astype(np.int64), idx, f"levels s={s}")


def test_large_level_counts_use_exact_path(Q):
    rng = np.random.default_rng(43)
    x = (rng.standard_normal(10000) * 0.05).astype(np.float32)
    for s in (257, 1024, 65536):
        q, _, _ = O.uniform_fwd(x, s, 256)
        qd, _ = Q.uniformQuantization(dev(x), s, bucket_size=256)
        assert_same(qd.cpu().numpy(), q, f"s={s}")


@pytest.mark.parametrize("bucket", [256, 384, 512, 768, 1000, 1024, 100, 1026, 2048, 3002, 4096, 8192, 12000, 20000, 49152])
def test_minmax_backward_vs_oracle(Q, bucket):
    rng = np.random.default_rng(5)
    for n in (1, 100, 256, 257, 1000, 4099, 20000, 150001):
        for s in (4, 16, 256):
            x = (rng.standard_normal(n) * 0.05).astype(np.float32)
            g = rng.standard_normal(n).astype(np.float32)
            ref, info = O.uniform_bwd_minmax(x, g, s, bucket)
            f = Q.uniformQuantization_variable(s, bucket_size=bucket)
            f.forward(dev(x))
            out = f.backward(dev(g)).cpu().numpy()
            assert_minmax_gradient(out, g, ref, info["argmax"], info["argmin"], info["abs_sum"], info["r"], f"n={n} s={s} b={bucket}")


def test_minmax_backward_in_place_and_degenerate_rows(Q):
    """gout aliasing g (what the training loop does), constant rows (alpha -> 1, argmin' == argmax': no change),
    rows whose quantized values collapse onto few floats (large offset), through warp / two-pass / staged paths."""
    from quantized_distillation_b200 import _native as N
    rng = np.random.default_rng(55)
    for bucket in (256, 1024, 2048, 8192, 20000):
        n = bucket * 9 + 17
        x = (rng.standard_normal(n) * 0.05).astype(np.float32)
        x[:bucket] = 0.25                                      # constant row
        x[bucket:2 * bucket] = 1000.0 + rng.standard_normal(bucket).astype(np.float32) * 1e-4   # q values collapse
        x[2 * bucket:3 * bucket] = np.repeat(rng.standard_normal(bucket // 8).astype(np.float32), 8)   # many ties
        g = rng.standard_normal(n).astype(np.float32)
        ref, info = O.uniform_bwd_minmax(x, g, 16, bucket)
        xd, gd = dev(x), dev(g)
        ws = N.workspace(n, bucket, xd.device)
        N.check(N.lib().qd_uniform_bwd(N.ptr(xd), N.ptr(gd), N.ptr(gd), n, bucket, 16, N.BWD_MINMAX, N.ptr(ws), ws.numel(),
                                       N.stream_ptr()))
        assert_minmax_gradient(gd.cpu().numpy(), g, ref, info["argmax"], info["argmin"], info["abs_sum"], info["r"], f"in place b={bucket}")


def test_fused_fwd_bwd_capi(Q):
    """qd_uniform_fwd_bwd through ctypes: q identical to the forward op, gout identical to the backward op."""
    from quantized_distillation_b200 import _native as N
    rng = np.random.default_rng(9)
    for n, b in ((4096, 256), (100000, 256), (5000, 512), (70001, 1024), (30000, 4096), (200000, 8192), (100000, 3002),
                 (300000, 49152)):
        x = dev((rng.standard_normal(n) * 2).astype(np.float32))
        g = dev(rng.standard_normal(n).astype(np.float32))
        ws = N.workspace(n, b, x.device)
        for mode in (N.BWD_STE, N.BWD_TRUNCATED, N.BWD_MINMAX):
            q, go = torch.empty_like(x), torch.empty_like(g)
            N.check(N.lib().qd_uniform_fwd_bwd(N.ptr(x), N.ptr(g), N.ptr(q), N.ptr(go), n, b, 16, mode, N.ptr(ws), ws.numel(),
                                               N.stream_ptr()))
            qref, _, _ = O.uniform_fwd(x.cpu().numpy(), 16, b)
            assert_same(q.cpu().numpy(), qref, f"fused q mode {mode}")
            go2 = torch.empty_like(g)
            N.check(N.lib().qd_uniform_bwd(N.ptr(x), N.ptr(g), N.ptr(go2), n, b, 16, mode, N.ptr(ws), ws.numel(), N.stream_ptr()))
            if mode == N.BWD_MINMAX:
                # the fused pass and the stand-alone backward may add the terms of r_b in a different order (each uses
                # the faster one, qd_api.cu): same positions, both inside the a5 tolerance of the oracle
                ref, info = O.uniform_bwd_minmax(x.cpu().numpy(), g.cpu().numpy(), 16, b)
                for out in (go, go2):
                    assert_minmax_gradient(out.cpu().numpy(), g.cpu().numpy(), ref, info["argmax"], info["argmin"], info["abs_sum"],
                                           info["r"], f"fused/unfused min/max n={n} b={b}")
                assert np.array_equal(np.nonzero((go != g).cpu().numpy())[0], np.nonzero((go2 != g).cpu().numpy())[0])
            else:
                assert_same(go.cpu().numpy(), go2.cpu().numpy(), f"fused gout mode {mode}")
            if mode == N.BWD_STE:
                assert_same(go.cpu().numpy(), g.cpu().numpy(), "ste")
            if mode == N.BWD_TRUNCATED:
                assert_same(go.cpu().numpy(), O.uniform_bwd_truncated(x.cpu().numpy(), g.cpu().numpy()), "trunc")


@pytest.mark.parametrize("bucket", [None, 256, 1024, 100, 1026, 4096, 8192, 3002, 20000, 49152])
def test_nonuniform_vs_oracle(Q, bucket):
    rng = np.random.default_rng(13)
    for n in (1, 10, 256, 257, 5000, 70001, 200003):
        for K in (1, 2, 3, 4, 5, 8, 9, 16, 17, 32, 33, 40, 256):
            x = (rng.standard_normal(n) * 0.05).astype(np.float32)
            pts = np.sort(rng.random(K)).astype(np.float32)
            if K >= 4:
                pts[1] = pts[2]                          # duplicate centroids
            for rule, kw in (("nearest", {}), ("midpoint", {"pre": True})):
                q, idx, st = O.nonuniform_fwd(x, pts, bucket, rule=rule)
                if rule == "nearest":
                    qd, idxd, sf = Q.nonUniformQuantization(dev(x), dev(pts), bucket_size=bucket)
                    qd8, idx8, _ = Q.nonUniformQuantization(dev(x), dev(pts), bucket_size=bucket, index_dtype=torch.uint8)
                    assert_same(idx8.cpu().numpy().astype(np.int64), idx, "u8 idx")
                else:
                    f = Q.nonUniformQuantization_variable(bucket_size=bucket, pre_process_tensors=True, tensor=dev(x))
                    qd = f.forward(None, dev(pts))
                    idxd = f.savedForBackward["indices"].to(torch.int64)
                assert_same(idxd.cpu().numpy(), idx, f"{rule} idx n={n} K={K} b={bucket}")
                assert_same(qd.cpu().numpy(), q, f"{rule} q n={n} K={K} b={bucket}")


def test_nonuniform_tiny_and_degenerate_rows(Q):
    """Rows that push x_hat's division outside the hoisted-reciprocal domain: tiny non-zero
    distances from the minimum, huge / tiny alpha, constant rows."""
    pts = np.array([0.0, 1e-30, 0.5, 1.0], np.float32)
    rows = [np.array([0.0, 1e-38, 1e-30, 1e-12, 0.5, 1.0, 3e-39, 1e-20] * 32, np.float32),
            np.array([0.0, 3e38, 1e10, 1.0] * 64, np.float32),
            np.array([1.0, 1.0 + 1e-7] * 128, np.float32),
            np.full(256, -2.5, np.float32),
            (np.arange(256) * 1e-42).astype(np.float32)]
    x = np.concatenate(rows)
    for rule in ("nearest", "midpoint"):
        with np.errstate(all="ignore"):
            q, idx, st = O.nonuniform_fwd(x, pts, 256, rule=rule)
        if rule == "nearest":
            qd, idxd, _ = Q.nonUniformQuantization(dev(x), dev(pts), bucket_size=256)
        else:
            f = Q.nonUniformQuantization_variable(bucket_size=256, pre_process_tensors=True, tensor=dev(x))
            qd = f.forward(None, dev(pts))
            idxd = f.savedForBackward["indices"].to(torch.int64)
        assert_same(idxd.cpu().numpy(), idx, f"tiny {rule} idx")
        assert_same(qd.cpu().numpy(), q, f"tiny {rule} q")


@pytest.mark.parametrize("bucket", [None, 256, 100])
def test_points_gradient_vs_oracle(Q, bucket):
    rng = np.random.default_rng(17)
    for n in (1, 300, 4099, 300001):
        for K in (2, 4, 8, 9, 16, 40):
            x = (rng.standard_normal(n) * 0.05).astype(np.float32)
            g = rng.standard_normal(n).astype(np.float32)
            pts = np.linspace(0, 1, K).astype(np.float32)
            f = Q.nonUniformQuantization_variable(bucket_size=bucket, pre_process_tensors=True, tensor=dev(x))
            f.forward(None, dev(pts))
            _, gp = f.backward(dev(g))
            _, idx, st = O.nonuniform_fwd(x, pts, bucket, rule="midpoint")
            ref = O.nonuniform_bwd_points(g, idx, st["alpha"], K, bucket)
            # float64 accumulation of float32 products: only the final cast to float32 differs from the exact sum
            assert np.abs(gp.cpu().numpy().astype(np.float64) - ref).max() <= 1e-6 * np.abs(ref).max() + 1e-30, (n, K, bucket)
            # deterministic: a second run is bit-identical
            f.forward(None, dev(pts))
            _, gp2 = f.backward(dev(g))
            assert_same(gp.cpu().numpy(), gp2.cpu().numpy(), "determinism")


def test_pre_ops_mean_and_clamp(Q):
    rng = np.random.default_rng(19)
    x = (rng.standard_normal(5000) * 2 + 0.3).astype(np.float32)
    for b in (256, None):
        # clamp only: bit exact
        q, _, _ = O.uniform_fwd(x, 16, b, max_element=1.5)
        qd, _ = Q.uniformQuantization(dev(x), 16, bucket_size=b, max_element=1.5)
        assert_same(qd.cpu().numpy(), q, "max_element")
        # mean: the reference's mean is a float32 torch reduction (order dependent) -> tolerance
        qd, sf = Q.uniformQuantization(dev(x), 16, bucket_size=b, subtract_mean=True)
        mean = float(sf.mean_tensor)
        assert abs(mean - x.astype(np.float64).mean()) < 1e-5
        q2, _, _ = O.uniform_fwd(x - np.float32(mean), 16, b)
        assert np.abs(qd.cpu().numpy() - (q2 + np.float32(mean))).max() < 1e-5


def test_stochastic_rounding_distribution(Q):
    torch.manual_seed(0)
    n, s = 1 << 20, 4
    x = torch.rand(n).cuda()
    x[0], x[1] = 0.0, 1.0
    x = x.view(-1)
    q, sf = Q.uniformQuantization(x, s, stochastic_rounding=True, bucket_size=None)
    lv = torch.round(q * (s - 1))
    assert torch.allclose(lv / (s - 1), q, atol=1e-6)
    lo = torch.floor(x * (s - 1))
    assert bool(((lv == lo) | (lv == lo + 1)).all())
    frac = x * (s - 1) - lo
    up = (lv == lo + 1).float()
    # E[up] = frac: compare in 10 bins of frac
    for k in range(10):
        m = (frac >= k / 10) & (frac < (k + 1) / 10)
        assert abs(up[m].mean().item() - frac[m].mean().item()) < 0.01
    q2, _ = Q.uniformQuantization(x, s, stochastic_rounding=True, bucket_size=None)
    assert not torch.equal(q, q2)                       # a fresh stream per call


def _stochastic(x, s, bucket, seed, offset=0):
    """qd_uniform_fwd with stochastic rounding through the C ABI: (q, integer levels, alpha, beta)."""
    from quantized_distillation_b200 import _native as N
    n = x.numel()
    b = 0 if bucket is None else bucket
    rows = N.geometry(n, b)[0]
    q = torch.empty_like(x)
    idx = torch.empty(n, dtype=torch.uint8, device=x.device)
    alpha, beta = torch.empty(rows, device=x.device), torch.empty(rows, device=x.device)
    ws = N.workspace(n, b, x.device)
    N.check(N.lib().qd_uniform_fwd(N.ptr(x), N.ptr(q), N.ptr(idx), N.ptr(alpha), N.ptr(beta), None, None, n, b, s, None, 0.0,
                                   1, seed, offset, N.ptr(ws), ws.numel(), N.stream_ptr()))
    return q, idx, alpha, beta


@pytest.mark.parametrize("s", [4, 16])
@pytest.mark.parametrize("bucket", [256, 512, 1024, 2048, 4096, 8192, None])
def test_stochastic_rounding_every_path(Q, bucket, s):
    """Stochastic rounding (quant_functions.py:174-187) on the warp (R=2,4,8), two-pass, CTA-staged and
    grid paths.  Exact part: the level is floor(x_hat*S) or that plus one, with x_hat, alpha, beta the
    oracle's bits, and q is bit-identical to the reference chain GIVEN the up/down decisions.  Random
    part (the reference draws torch.rand on the host, so only the distribution can match): E[up | frac]
    = frac inside 4 sigma in ten bins, decisions independent of the row (no Philox block reused),
    reproducible per seed, different across seeds."""
    rng = np.random.default_rng(31)
    n = (1 << 20) + 37
    xh_np = (rng.standard_normal(n) * 0.05).astype(np.float32)
    x = dev(xh_np)
    q, lv, alpha, beta = _stochastic(x, s, bucket, seed=1234)
    xh, st = O.scale_down(xh_np, bucket)
    assert_same(alpha.cpu().numpy(), st["alpha"], "alpha")
    assert_same(beta.cpu().numpy(), st["beta"], "beta")
    S = np.float32(s - 1)
    prob = (S * xh).astype(np.float32).reshape(-1)[:n]
    lo = np.floor(prob)
    frac = (prob - lo).astype(np.float32)
    lvh = lv.cpu().numpy().astype(np.float32)
    up = lvh == lo + 1
    assert np.all(up | (lvh == lo)), "level is neither floor nor floor + 1"
    assert not np.any(up & (frac == 0) & (lo == s - 1)), "rounded up past the top level"
    # q given the decisions: the oracle's chain with u = 0 where the kernel went up and u = 2 where it did not
    u = np.full(xh.size, 2.0, np.float32)
    u[:n][up] = 0.0
    qref, _ = O.uniform_fwd_stochastic(xh_np, s, bucket, u)
    assert_same(q.cpu().numpy(), qref, f"stochastic q b={bucket} s={s}")
    # distribution
    for k in range(10):
        m = (frac >= k / 10) & (frac < (k + 1) / 10)
        cnt = int(m.sum())
        assert cnt > 1000
        p = frac[m].astype(np.float64)
        sigma = np.sqrt((p * (1 - p)).sum()) / cnt
        assert abs(up[m].mean() - p.mean()) < 4 * sigma + 2.0 ** -24, (k, up[m].mean(), p.mean(), sigma)
    # streams: same seed -> same bits; other seed / other offset -> a different draw
    q_again, lv_again, _, _ = _stochastic(x, s, bucket, seed=1234)
    assert torch.equal(lv_again, lv) and torch.equal(q_again, q)
    for other in (_stochastic(x, s, bucket, seed=1235)[1], _stochastic(x, s, bucket, seed=1234, offset=1 << 20)[1]):
        differ = (other != lv).float().mean().item()
        assert differ > 0.05, differ


@pytest.mark.parametrize("bucket", [256, 1024, 4096, 8192])
def test_stochastic_rounding_rows_get_distinct_random_blocks(Q, bucket):
    """Every row holds the SAME values: if two rows (or two warps, or two CTAs) consumed the same Philox
    counters their up/down patterns would coincide.  No two rows may agree, and no row may be periodic
    with the 4-element period of one Philox block."""
    rng = np.random.default_rng(37)
    rows = 512
    row = rng.random(bucket).astype(np.float32)
    row[0], row[1] = 0.0, 1.0
    x = dev(np.tile(row, rows))
    _, lv, _, _ = _stochastic(x, 4, bucket, seed=99)
    pat = lv.view(rows, bucket).cpu().numpy()
    uniq = np.unique(pat, axis=0)
    assert uniq.shape[0] == rows, f"{rows - uniq.shape[0]} rows share their random pattern with another row"
    same_next = (pat[1:] == pat[:-1]).mean()
    base = (pat == np.floor(row * 3)[None, :]).mean()            # P(two independent draws agree) is far below 1
    assert same_next < 0.95 and base < 0.95, (same_next, base)


def test_cpu_tensors_run_on_gpu_and_come_back(Q):
    rng = np.random.default_rng(23)
    x = (rng.standard_normal(3000) * 0.05).astype(np.float32)
    ref, idx, st = O.uniform_fwd(x, 16, 256)
    q, sf = Q.uniformQuantization(torch.from_numpy(x.copy()), 16, bucket_size=256)
    assert not q.is_cuda and not sf.alpha.is_cuda
    assert_same(q.numpy(), ref, "cpu tensor")
    qn, idxn, _ = Q.nonUniformQuantization(torch.from_numpy(x.copy()), [0.0, 0.3, 0.7, 1.0], bucket_size=256)
    qo, io, _ = O.nonuniform_fwd(x, np.array([0.0, 0.3, 0.7, 1.0], np.float32), 256)
    assert_same(qn.numpy(), qo, "cpu nonuniform")
    assert_same(idxn.numpy(), io, "cpu nonuniform idx")


def test_host_buffer_capi_pipeline(Q):
    from quantized_distillation_b200 import _native as N
    rng = np.random.default_rng(29)
    for n, b in ((10_000_003, 256), (5_000_000, 0), (9_000_000, 4096)):
        x = torch.from_numpy((rng.standard_normal(n) * 0.05).astype(np.float32)).pin_memory()
        g = torch.from_numpy(rng.standard_normal(n).astype(np.float32)).pin_memory()
        q = torch.empty(n, dtype=torch.float32).pin_memory()
        go = torch.empty(n, dtype=torch.float32).pin_memory()
        N.check(N.lib().qd_uniform_fwd_bwd_host(N.ptr(x), N.ptr(g), N.ptr(q), N.ptr(go), n, b, 16, N.BWD_TRUNCATED,
                                                torch.cuda.current_device()))
        qd, _ = Q.uniformQuantization(x.cuda(), 16, bucket_size=b or None)
        assert torch.equal(q, qd.cpu()), (n, b)
        assert torch.equal(go, g)                        # |x| <= 1 everywhere here
        q.zero_()
        N.check(N.lib().qd_uniform_fwd_host(N.ptr(x), N.ptr(q), n, b, 16, torch.cuda.current_device()))
        assert torch.equal(q, qd.cpu())
    # min/max backward is row-local, so the host entry point equals the resident call bit for bit whatever the staging:
    # one launch straight on the pinned buffers (<= 8 Mi elements), the chunked pipeline (larger, or pageable memory)
    for n, b, pinned in ((1000, 256, True), (1_000_003, 256, True), (3_000_000, 1000, True), (2_000_001, 256, False),
                         (30_000_001, 256, True), (26_000_123, 1000, True)):
        pin = (lambda t: t.pin_memory()) if pinned else (lambda t: t)
        x = pin(torch.from_numpy((rng.standard_normal(n) * 0.05).astype(np.float32)))
        g = pin(torch.from_numpy(rng.standard_normal(n).astype(np.float32)))
        q = pin(torch.zeros(n, dtype=torch.float32))
        go = pin(torch.zeros(n, dtype=torch.float32))
        N.check(N.lib().qd_uniform_fwd_bwd_host(N.ptr(x), N.ptr(g), N.ptr(q), N.ptr(go), n, b, 16, N.BWD_MINMAX,
                                                torch.cuda.current_device()))
        xd, gd = x.cuda(), g.cuda()
        qd, god = torch.empty_like(xd), torch.empty_like(gd)
        ws = N.workspace(n, b, xd.device)
        N.check(N.lib().qd_uniform_fwd_bwd(N.ptr(xd), N.ptr(gd), N.ptr(qd), N.ptr(god), n, b, 16, N.BWD_MINMAX, N.ptr(ws), ws.numel(),
                                           N.stream_ptr()))
        assert torch.equal(q, qd.cpu()), (n, b)
        assert torch.equal(go, god.cpu()), (n, b)


def test_multi_tensor_plan_matches_per_tensor(Q):
    from quantized_distillation_b200.plan import QuantizationPlan
    rng = np.random.default_rng(31)
    sizes = [5000, 10, 5625, 75, 93750, 50, 62500, 50, 31250, 25, 800000, 500, 75, 75, 50, 50, 25, 25, 500, 500, 1, 257]
    for bucket in (256, 1024, None, 4096):
        params = [dev((rng.standard_normal(n) * 0.05).astype(np.float32)) for n in sizes]
        ref = [Q.uniformQuantization(p, 16, bucket_size=bucket)[0] for p in params]
        plan = QuantizationPlan(params, levels=16, bucket_size=bucket)
        master = plan.save_master()
        plan.quantize_()
        for p, r in zip(params, ref):
            assert torch.equal(p, r)
        plan.restore_master()
        for p, m in zip(params, master):
            assert torch.equal(p, m)
        originals = [p.clone() for p in params]
        fused_master = plan.save_and_quantize_()          # one pass: shadow copy + in-place quantization
        for p, r, m, o in zip(params, ref, fused_master, originals):
            assert torch.equal(p, r) and torch.equal(m, o)
        plan.restore_master()
        if bucket is not None:
            grads = [dev(rng.standard_normal(n).astype(np.float32)) for n in sizes]
            expect = []
            for p, g in zip(params, grads):
                f = Q.uniformQuantization_variable(16, bucket_size=bucket)
                f.forward(p)
                expect.append(f.backward(g))
            plan.backward_(grads, "complicated")
            for g, e in zip(grads, expect):
                assert torch.equal(g, e)
        # 'truncated' fix-up (also on the long-row plan of bucket None: one launch for all tensors)
        for p in params:
            p.mul_(30.0)                                   # some |w| > 1
        grads = [dev(rng.standard_normal(n).astype(np.float32)) for n in sizes]
        expect = [torch.where(p.abs() > 1, torch.zeros_like(g), g) for p, g in zip(params, grads)]
        plan.backward_(grads, "truncated")
        for g, e in zip(grads, expect):
            assert torch.equal(g, e)
        if bucket is None:
            with pytest.raises(NotImplementedError):
                plan.backward_(grads, "complicated")


def test_long_row_plan_wrn_sized_model_bucket_none(Q):
    """bucket_size=None on a model with tensors far beyond one SM's shared memory (the post-mortem setting,
    cifar10_test.py:305-317): three launches for the whole model, bit-identical to the per-tensor op."""
    from quantized_distillation_b200.plan import QuantizationPlan
    gen = torch.Generator(device="cuda").manual_seed(8)
    sizes = [432, 16, 4_460_544, 352, 1_115_136, 10, 123_904, 49_153, 16_384, 16_385, 3]
    params = [torch.randn(n, generator=gen, device="cuda") * 0.05 for n in sizes]
    params[2] = params[2].view(352, 352, 6, 6)[:, :, :, :]                     # a 4-D view, like a conv weight
    for levels in (4, 256):
        work = [p.clone() for p in params]
        ref = [Q.uniformQuantization(p, levels, bucket_size=None)[0] for p in work]
        plan = QuantizationPlan(work, levels=levels, bucket_size=None)
        master = plan.save_and_quantize_()
        for w, r, m, o in zip(work, ref, master, params):
            assert torch.equal(w, r) and torch.equal(m.view(-1), o.reshape(-1))


def test_centroid_plan_matches_per_tensor_ops_and_oracle(Q):
    """qd_plan_nonuniform_fwd / _bwd: every tensor of a model in one forward launch and two gradient
    launches.  q and idx bit-identical to the per-tensor op and to the oracle (midpoint rule), centroid
    gradients equal to the oracle's float64 sums within float32 rounding, deterministic across calls."""
    from quantized_distillation_b200.plan import CentroidPlan
    rng = np.random.default_rng(41)
    sizes = [5000, 10, 5625, 75, 93750, 50, 800000, 500, 25, 1, 257, 255]          # student-like mix incl. tiny tensors
    for bucket in (256, 1024, 100, None):
        if bucket is None:
            use = [n for n in sizes if n <= 1024]
        else:
            use = sizes
        Ks = [int(rng.integers(1, 33)) for _ in use]
        Ks[0], Ks[1] = 4, 32
        xs = [(rng.standard_normal(n) * 0.05).astype(np.float32) for n in use]
        pts = [np.sort(rng.random(k)).astype(np.float32) for k in Ks]
        gs = [rng.standard_normal(n).astype(np.float32) for n in use]
        src = [dev(x) for x in xs]
        dst = [torch.empty_like(t) for t in src]
        pd = [dev(p) for p in pts]
        plan = CentroidPlan(src, dst, pd, bucket)
        plan.forward_()
        grads = plan.backward_([dev(g) for g in gs])
        first = [g.clone() for g in grads]
        for i, (x, p, g) in enumerate(zip(xs, pts, gs)):
            q, idx, st = O.nonuniform_fwd(x, p, bucket, rule="midpoint")
            assert_same(dst[i].cpu().numpy(), q, f"plan q tensor {i} b={bucket}")
            assert_same(plan.indices[i].cpu().numpy().astype(np.int64).reshape(-1), idx.reshape(-1), f"plan idx tensor {i}")
            assert_same(plan.alpha[i].cpu().numpy(), st["alpha"], "plan alpha")
            f = Q.nonUniformQuantization_variable(bucket_size=bucket, pre_process_tensors=True, tensor=src[i])
            assert torch.equal(f.forward(None, pd[i]).view(-1), dst[i].view(-1))
            ref = O.nonuniform_bwd_points(g, idx, st["alpha"], len(p), bucket)
            got = first[i].cpu().numpy().astype(np.float64)
            mag = np.array([np.abs(g.reshape(-1)[idx.reshape(-1) == k]).sum() for k in range(len(p))]) * float(st["alpha"].max())
            assert np.all(np.abs(got - ref) <= 1e-6 * mag + 2.0 ** -23 * np.abs(ref) + 1e-30), (i, bucket, got, ref)
        # new points, same plan: the table is re-read at every launch; gradients reproducible bit for bit
        for p in pd:
            p.copy_(torch.sort(torch.rand_like(p))[0])
        plan.forward_()
        for i, x in enumerate(xs):
            q, idx, _ = O.nonuniform_fwd(x, pd[i].cpu().numpy(), bucket, rule="midpoint")
            assert_same(dst[i].cpu().numpy(), q, f"plan q after point update, tensor {i}")
        a = [g.clone() for g in plan.backward_([dev(g) for g in gs])]
        b = [g.clone() for g in plan.backward_([dev(g) for g in gs])]
        assert all(torch.equal(u, v) for u, v in zip(a, b))
    big = torch.randn(5000, device="cuda")
    with pytest.raises(NotImplementedError):                    # more than 32 points
        CentroidPlan([big], [torch.empty_like(big)], [torch.linspace(0, 1, 33, device="cuda")], 256)
    with pytest.raises(NotImplementedError):                    # rows longer than 1024 elements
        CentroidPlan([big], [torch.empty_like(big)], [torch.linspace(0, 1, 4, device="cuda")], 2048)


def test_order_statistics_select_is_exact(Q):
    """qd_order_statistics (value histogram + compaction + radix select) against a full sort, bit for
    bit: uniform / peaked / constant / heavy-tie inputs, values outside [0, 1], tiny tensors, up to 512
    ranks, unaligned views."""
    from quantized_distillation_b200.quantization import help_functions as H
    gen = torch.Generator(device="cuda").manual_seed(3)
    cases = []
    for n in (1, 2, 5, 257, 4099, 100003, 5_000_017):
        cases.append(torch.rand(n, generator=gen, device="cuda"))
        cases.append((torch.randn(n, generator=gen, device="cuda") * 0.02 + 0.5).clamp_(0, 1))      # peaked: few value bins hold everything
    cases.append(torch.full((70001,), 0.25, device="cuda"))
    cases.append(torch.randint(0, 4, (300000,), generator=gen, device="cuda").float() / 3)           # four distinct values
    cases.append(torch.randn(200001, generator=gen, device="cuda") * 5)                                # far outside [0, 1]
    cases.append(torch.rand(100004, generator=gen, device="cuda")[3:])                                 # 12-byte offset view
    for v in cases:
        n = v.numel()
        ref = torch.sort(v)[0]
        for R in (1, 8, 32, 512):
            ranks = torch.randint(0, n, (R,), generator=gen, device="cuda").cpu().numpy()
            ranks[0], ranks[-1] = 0, n - 1
            got = H.order_statistics(v, ranks)
            want = ref[torch.as_tensor(ranks, device="cuda")]
            assert torch.equal(got, want), (n, R)


def test_gradient_norms_multi_tensor(Q):
    from quantized_distillation_b200.quantization import help_functions as H
    gen = torch.Generator(device="cuda").manual_seed(4)
    ts = [torch.randn(n, generator=gen, device="cuda") * (i + 1) for i, n in enumerate((1, 10, 5000, 16384, 16385, 800000, 75))]
    got = H.gradient_norms(ts)
    want = torch.stack([t.double().norm() for t in ts])
    assert torch.allclose(got.double(), want, rtol=2e-7, atol=0), (got, want)
    assert torch.equal(got, H.gradient_norms(ts))                 # fixed summation order: reproducible bits


def test_absmax_absnorm_extension_matches_the_intended_semantics(Q):
    """Row a10: PARITY UNPINNED -- the reference lines (quant_functions.py:109-127) cannot execute, so this only checks
    that the opt-in extension computes the intended semantics restated in oracle/quant_oracle.py: refused by default,
    then scale_down / inv_scale_down / uniformQuantization bit-exact given the per-bucket scale (absmax: exact scale;
    absnorm: float64 sum rounded once, so the scale itself is compared to one ulp)."""
    from quantized_distillation_b200.quantization import quant_functions as QF
    x0 = torch.randn(1000, device="cuda")
    with pytest.raises(NotImplementedError):
        Q.uniformQuantization(x0, 8, type_of_scaling="absmax", bucket_size=256)
    QF.ALLOW_UNPINNED_SCALING = True
    try:
        rng = np.random.default_rng(61)
        for kind in ("absmax", "absnorm"):
            for bucket in (256, 100, None, 4096):
                for n in (1, 255, 256, 257, 5000, 70001):
                    x = (rng.standard_normal(n) * 0.05).astype(np.float32)
                    if n > 10:
                        x[3] = 0.0
                        x[7] = -x[5]
                    sf = Q.ScalingFunction(kind, False, False, bucket, False)
                    xh = sf.scale_down(dev(x))
                    norm_d = sf.norm_scaling.reshape(-1).cpu().numpy()
                    oxh, osign, onorm, _ = O.abs_scale_down(x, bucket, kind)
                    if kind == "absmax":
                        assert_same(norm_d, onorm, f"{kind} norm b={bucket} n={n}")
                    else:
                        assert np.all(np.abs(norm_d - onorm) <= np.spacing(onorm)), (kind, bucket, n)
                        oxh, osign, onorm, _ = O.abs_scale_down(x, bucket, kind, norm=norm_d)
                    assert_same(xh.cpu().numpy().reshape(oxh.shape), oxh, f"{kind} x_hat b={bucket} n={n}")
                    assert_same(sf.tensor_sign.cpu().numpy().reshape(osign.shape), osign, f"{kind} sign")
                    back = sf.inv_scale_down(xh).cpu().numpy().reshape(-1)
                    want = ((oxh * onorm[:, None]).astype(np.float32) * osign).astype(np.float32).reshape(-1)[:n]
                    assert_same(back, want, f"{kind} inverse")
                    for s in (2, 8, 128):
                        q, sf2 = Q.uniformQuantization(dev(x), s, type_of_scaling=kind, bucket_size=bucket)
                        nd = sf2.norm_scaling.reshape(-1).cpu().numpy()
                        oq, _, _ = O.uniform_fwd_abs(x, s, bucket, kind, norm=nd)
                        assert_same(q.cpu().numpy(), oq, f"{kind} q b={bucket} n={n} s={s}")
                        lv = np.unique(np.abs(q.cpu().numpy().reshape(-1)[:min(n, bucket or n)]) / max(nd[0], 1e-30) * (s - 1)).round(3)
                        assert lv.size <= s
        with pytest.raises(NotImplementedError):
            Q.uniformQuantization(x0, 8, type_of_scaling="absmax", bucket_size=256, stochastic_rounding=True)
    finally:
        QF.ALLOW_UNPINNED_SCALING = False


def test_compiled_front_door_equals_ctypes_path(Q):
    """The optional pybind/ATen module in front of the per-tensor ops (csrc/qd_torch_fast.cpp) is plumbing only: with it
    and without it (ctypes) every output -- q, alpha, beta, argmin, argmax, shapes, dtypes, the backward -- is identical."""
    from quantized_distillation_b200 import _native as N
    if N.fast() is None:
        pytest.skip("fast-call module not built")
    rng = np.random.default_rng(71)
    saved = N._fast
    try:
        for n, bucket in ((5000, 256), (10, 256), (257, 100), (70001, 1024), (100000, 4096), (300001, None)):
            x = dev((rng.standard_normal(n) * 0.05).astype(np.float32)).view(-1, 1) if n == 5000 else dev((rng.standard_normal(n) * 0.05).astype(np.float32))
            g = dev(rng.standard_normal(n).astype(np.float32)).view(x.shape)
            outs = []
            for use_fast in (True, False):
                N._fast = saved if use_fast else None
                q, sf = Q.uniformQuantization(x, 16, bucket_size=bucket)
                res = [q, sf.alpha, sf.beta, sf.idx_min_rows, sf.idx_max_rows]
                meta = (sf.original_tensor_size, sf.original_tensor_length, sf.expected_tensor_size, sf.mean_tensor)
                if bucket is not None:
                    f = Q.uniformQuantization_variable(16, bucket_size=bucket)
                    f.forward(x)
                    res.append(f.backward(g))
                outs.append((res, meta))
            for a, b in zip(outs[0][0], outs[1][0]):
                assert a.shape == b.shape and a.dtype == b.dtype and torch.equal(a, b)
            assert outs[0][1] == outs[1][1]
        N._fast = saved
        xin = dev((rng.standard_normal(4096) * 0.05).astype(np.float32))
        keep = xin.clone()
        q, _ = Q.uniformQuantization(xin, 4, bucket_size=256, modify_in_place=True)
        assert q.data_ptr() == xin.data_ptr() and not torch.equal(xin, keep)
        with pytest.raises(ValueError):
            Q.uniformQuantization(xin, 1, bucket_size=256)                      # levels < 2: the C ABI's INVALID_ARG -> ValueError
    finally:
        N._fast = saved


def test_error_mapping(Q):
    x = torch.randn(100).cuda()
    with pytest.raises(ValueError):
        Q.uniformQuantization(x, 1, bucket_size=256)                 # s < 2
    with pytest.raises(ValueError):
        Q.ScalingFunction("cubic", False, False, None)
    with pytest.raises(ValueError):
        Q.ScalingFunction("linear", False, False, -3)
    f = Q.uniformQuantization_variable(16, bucket_size=None)
    f.forward(x)
    with pytest.raises(NotImplementedError):
        f.backward(x)
    with pytest.raises(ValueError):
        Q.uniformQuantization_variable(16, bucket_size=256).backward(x)
    with pytest.raises(ValueError):
        Q.nonUniformQuantization(x, [0.0, 1.0], pre_processed_values=True)
    with pytest.raises(ValueError):
        Q.nonUniformQuantization_variable(pre_process_tensors=True)
    sf = Q.ScalingFunction("linear", False, False, 64)
    sf.scale_down(x)
    with pytest.raises(ValueError):
        sf.inv_scale_down(torch.zeros(3, 64).cuda())


def test_division_selftest_on_device(Q):
    import ctypes as C
    from quantized_distillation_b200 import _native as N
    bad = C.c_int64(-1)
    N.check(N.lib().qd_selftest_division(1 << 26, 1234, C.byref(bad), N.stream_ptr()))
    assert bad.value == 0


def test_full_size_properties_64M(Q):
    """BASELINE size (64 Mi floats): size-independent properties instead of an oracle run.
    idempotence (q(q(x)) == q(x)), level count <= s per bucket, range preserved, and the
    first/last 1 Mi elements against the oracle."""
    n, s, b = 1 << 26, 16, 256
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(n, generator=g, device="cuda") * 0.05
    q, sf = Q.uniformQuantization(x, s, bucket_size=b)
    q2, _ = Q.uniformQuantization(q, s, bucket_size=b)
    assert float((q2 - q).abs().max()) <= 1e-6 * float(q.abs().max())
    rows = q.view(-1, b)
    assert torch.equal(rows.min(dim=1)[0], x.view(-1, b).min(dim=1)[0])
    assert float((rows.max(dim=1)[0] - x.view(-1, b).max(dim=1)[0]).abs().max()) <= 1e-6
    lv = torch.round((rows - sf.beta) / sf.alpha * (s - 1))
    assert float(lv.min()) == 0 and float(lv.max()) == s - 1
    for sl in (slice(0, 1 << 20), slice(n - (1 << 20), n)):
        ref, _, _ = O.uniform_fwd(x[sl].cpu().numpy(), s, b)
        assert_same(q[sl].cpu().numpy(), ref, "64M slice")
    # the whole 64 Mi tensor, bit for bit, against the C restatement (oracle/quant_oracle.c)
    from oracle import c_oracle as CO
    xh = x.cpu().numpy()
    qc, idxc, stc = CO.uniform_fwd(xh, s, b)
    assert_same(q.cpu().numpy(), qc, "64M full tensor vs C oracle")
    assert_same(sf.alpha.view(-1).cpu().numpy(), stc["alpha"], "64M alpha")
    assert_same(sf.idx_max_rows.view(-1).cpu().numpy(), stc["argmax"], "64M argmax")
    del qc, idxc
    # fused forward+backward at full size: q identical, gout within the float32-sum tolerance per bucket
    from quantized_distillation_b200 import _native as N
    gd = torch.randn(n, generator=g, device="cuda")
    qq, go = torch.empty_like(x), torch.empty_like(gd)
    ws = N.workspace(n, b, x.device)
    N.check(N.lib().qd_uniform_fwd_bwd(N.ptr(x), N.ptr(gd), N.ptr(qq), N.ptr(go), n, b, s, N.BWD_MINMAX, N.ptr(ws), ws.numel(),
                                       N.stream_ptr()))
    assert torch.equal(qq, q)
    gh = gd.cpu().numpy()
    ref, abs_sum, r = CO.uniform_bwd_minmax_ex(xh, gh, s, b)
    # positions: first argmax' / argmin' of the QUANTIZED rows (quant_functions.py:350-363)
    qrows = q.view(-1, b)
    base = torch.arange(n // b, device="cuda") * b
    amax = (qrows.argmax(dim=1) + base).cpu().numpy()          # torch.argmax / argmin: first occurrence
    amin = (qrows.argmin(dim=1) + base).cpu().numpy()
    assert_minmax_gradient(go.cpu().numpy(), gh, ref, amax, amin, abs_sum, r, "64M fused min/max backward")


def test_packed_codec_round_trip(Q):
    """encode -> (bit-packed codes, alpha, beta) -> decode reproduces the fused fake-quant output bit for bit."""
    from quantized_distillation_b200 import codec
    rng = np.random.default_rng(47)
    for n in (1, 7, 8, 9, 255, 256, 257, 5000, 300001):
        x = dev((rng.standard_normal(n) * 0.05).astype(np.float32))
        for s, bucket in ((2, 256), (4, 256), (16, 256), (256, 256), (16, None), (3, 100), (200, 4096)):
            pt = codec.encode_uniform(x, s, bucket)
            assert pt.bits == codec.bits_for(s) and pt.packed.numel() == (n * pt.bits + 7) // 8
            q, _ = Q.uniformQuantization(x, s, bucket_size=bucket)
            assert torch.equal(codec.decode(pt), q), (n, s, bucket)
        for K, rule in ((4, "nearest"), (16, "midpoint"), (3, "nearest")):
            pts = np.sort(rng.random(K)).astype(np.float32)
            pt = codec.encode_nonuniform(x, pts, 256, rule=rule)
            if rule == "nearest":
                qn, _, _ = Q.nonUniformQuantization(x, dev(pts), bucket_size=256)
            else:
                qn = Q.nonUniformQuantization_variable(bucket_size=256, pre_process_tensors=True, tensor=x).forward(None, dev(pts))
            assert torch.equal(codec.decode(pt), qn), (n, K, rule)
    big = codec.encode_uniform(dev(rng.standard_normal(1 << 20).astype(np.float32)), 16, 256)
    assert abs(big.nbytes / (4 << 20) - 1 / codec.get_size_reduction(4, 256)) < 1e-6      # 4-bit + 8 B per 256 weights
    assert codec.get_size_reduction(4, None) == 8


def test_packed_codec_many_tiles_and_unaligned_views(Q):
    """The tiled pack / unpack / inv_scale kernels past one tile per CTA (the row cursor advances by tile steps),
    with ragged buckets, and on views whose pointers are not 16-byte aligned (byte-wise fallbacks)."""
    from quantized_distillation_b200 import _native as N
    from quantized_distillation_b200 import codec
    g = torch.Generator(device="cuda").manual_seed(5)
    n = 40_000_003
    x = torch.randn(n, generator=g, device="cuda") * 0.05
    for s, bucket in ((16, 256), (4, 100), (256, 1000), (2, None)):
        pt = codec.encode_uniform(x, s, bucket)
        q, sf = Q.uniformQuantization(x, s, bucket_size=bucket)
        assert torch.equal(codec.decode(pt), q), (s, bucket)
        # inv_scale(scale(x)) against the two stock-torch ops of the reference (mul_, add_: no FMA)
        f = Q.ScalingFunction("linear", False, False, bucket, False)
        y = f.scale_down(x)
        back = f.inv_scale_down(y)
        if bucket is None:
            want = y * f.alpha + f.beta
        else:
            rows = -(-n // bucket)
            yp = torch.zeros(rows * bucket, device="cuda")
            yp[:n] = y.view(-1)[:n]
            want = (yp.view(rows, bucket) * f.alpha.view(-1, 1) + f.beta.view(-1, 1)).view(-1)[:n]
        assert torch.equal(back.view(-1), want.view(-1)), (s, bucket)
    # unaligned device pointers straight through the C ABI
    lib, sp = N.lib(), N.stream_ptr()
    m = 100_001
    idx_store = torch.randint(0, 16, (m + 3,), dtype=torch.uint8, device="cuda", generator=g)
    for off in (0, 1, 3):
        for bits in (1, 2, 4, 8):
            codes = (idx_store & ((1 << bits) - 1))[off:off + m]          # a view: pointer offset by `off` bytes
            out_store = torch.zeros((m * bits + 7) // 8 + 3, dtype=torch.uint8, device="cuda")
            packed = out_store[off:off + (m * bits + 7) // 8]
            N.check(lib.qd_pack_indices(N.ptr(codes), N.ptr(packed), m, bits, sp))
            c = codes.cpu().numpy().astype(np.uint64)
            per = 8 // bits
            pad = np.zeros(-(-m // per) * per, dtype=np.uint64)
            pad[:m] = c
            want = np.zeros(len(pad) // per, dtype=np.uint64)
            for j in range(per):
                want |= pad[j::per] << np.uint64(j * bits)
            assert np.array_equal(packed.cpu().numpy(), want.astype(np.uint8)), (off, bits)
            # unpack from the unaligned view into an unaligned float view
            alpha = torch.full((1,), 2.0, device="cuda")
            beta = torch.full((1,), -1.0, device="cuda")
            q_store = torch.zeros(m + 3, device="cuda")
            qv = q_store[off:off + m]
            levels = 1 << bits
            N.check(lib.qd_unpack_dequant_uniform(N.ptr(packed), bits, N.ptr(alpha), N.ptr(beta), N.ptr(qv), m, 0, levels, sp))
            # a tensor divisor: torch's CUDA division by a Python scalar multiplies by the reciprocal instead
            wantq = (codes.float() / torch.full((m,), float(levels - 1), device="cuda")) * 2.0 + (-1.0)
            assert torch.equal(qv, wantq), (off, bits)


def test_size_accounting_matches_reference_formula(Q):
    from quantized_distillation_b200 import codec
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Linear(64, 300), torch.nn.ReLU(), torch.nn.Linear(300, 10)).cuda()
    fun = lambda t: Q.uniformQuantization(t, 16, bucket_size=256)  # noqa: E731
    mb = codec.get_size_quantized_model(model, 4, fun, bucket_size=256, quantizeFirstLastLayer=False)
    params = list(model.parameters())
    mbl = Q.help_functions.get_huffman_encoding_mean_bit_length(iter(params[1:-1]), fun, "uniform", s=16)
    count_q = sum(p.numel() for p in params[1:-1])
    count_u = params[0].numel() + params[-1].numel()
    assert abs(mb - (count_u * 4 + mbl * count_q / 8 + count_q / 256 * 8) / 1e6) < 1e-12
    assert codec.get_size_quantized_model(model, None, fun) == sum(p.numel() for p in params) * 4 / 1e6


def test_c_abi_is_reentrant_across_threads_and_streams(Q):
    """Four Python threads, each on its own CUDA stream, hammer the library concurrently;
    every result must equal the single-threaded one (no shared mutable state in the ABI)."""
    import threading
    rng = np.random.default_rng(53)
    xs = [dev((rng.standard_normal(200_003) * 0.05).astype(np.float32)) for _ in range(4)]
    expect = [Q.uniformQuantization(x, 16, bucket_size=256)[0].clone() for x in xs]
    expect_none = [Q.uniformQuantization(x, 16, bucket_size=None)[0].clone() for x in xs]
    torch.cuda.synchronize()
    errors = []

    def work(i):
        try:
            s = torch.cuda.Stream()
            with torch.cuda.stream(s):
                for _ in range(20):
                    q, _ = Q.uniformQuantization(xs[i], 16, bucket_size=256)
                    qn, _ = Q.uniformQuantization(xs[i], 16, bucket_size=None)       # grid path: needs its own workspace
                    f = Q.nonUniformQuantization_variable(bucket_size=256, pre_process_tensors=True, tensor=xs[i])
                    f.forward(None, torch.linspace(0, 1, 4, device="cuda"))
                    f.backward(xs[i])
                s.synchronize()
                if not (torch.equal(q, expect[i]) and torch.equal(qn, expect_none[i])):
                    errors.append(i)
        except Exception as e:  # pragma: no cover
            errors.append((i, repr(e)))

    threads = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors, errors
