"""Parity of the CUDA product path with the oracle / reference golden vectors (needs a B200).

Tolerances are BASELINE.json's: relative L2 <= 1e-5 on the FP32 direct path, <= 1e-4 on the
tensor-core (3xTF32) path.  Everything goes through the plugin or the C ABI; the oracle only checks.
"""
import ctypes

import numpy as np
import pytest

from conftest import golden_names, load_golden, product_golden_names
from oracle import bruteforce_oracle as orc
from oracle import c_oracle

pytestmark = pytest.mark.gpu

TOL_DIRECT = 1e-5
TOL_TENSOR = 1e-4
PRODUCT_CASES = product_golden_names()

def run_plugin(kernel, y, x, b, *, same_points=False, normalize_rows=False, density=False, path="auto"):
    """The call sequence of runner.py:73-143."""
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Product

    algo = B200Product(kernel=kernel, dimension=y.shape[1], normalize_rows=normalize_rows, precision="float32", path=path)
    try:
        algo.prepare_data(source_points=y, target_points=y if x is None else x, same_points=same_points,
                          density_estimation=density)
        algo.fit()
        algo.prepare_query(source_signal=b)
        algo.query()
        out = algo.get_result()
        extra = algo.get_additional()
    finally:
        algo.done()
    assert out.dtype == np.float64 and out.flags["C_CONTIGUOUS"]
    return out, extra


@pytest.mark.parametrize("name", PRODUCT_CASES)
def test_golden_vectors(name):
    g = load_golden(name)
    D = g["source_points"].shape[1]
    out, extra = run_plugin(g["kernel"], g["source_points"], g["target_points"], g["source_signal"],
                            same_points=g["same_points"], normalize_rows=g["normalize_rows"], density=g["density_estimation"])
    assert out.shape == g["truth"].shape
    tol = TOL_DIRECT if D <= 16 else TOL_TENSOR
    err = orc.rel_l2(out, g["truth"])
    assert err <= tol, f"{name}: rel-L2 {err:.3e} > {tol:g}"
    assert extra["gpu_launches"] >= 1


@pytest.mark.parametrize("name", [n for n in PRODUCT_CASES if "gaussian" in n and "d64" not in n and "d784" not in n])
def test_golden_vectors_difference_form(name):
    """The Gaussian golden cases again with the product form switched off (path='direct_diff')."""
    g = load_golden(name)
    out, extra = run_plugin(g["kernel"], g["source_points"], g["target_points"], g["source_signal"], same_points=g["same_points"],
                            normalize_rows=g["normalize_rows"], density=g["density_estimation"], path="direct_diff")
    assert orc.rel_l2(out, g["truth"]) <= TOL_DIRECT
    assert extra["form"] in ("difference", "n/a")


def test_gaussian_form_selection():
    """Unit-scale data -> product form; spread-out data -> difference form (decided on the device);
    both within tolerance of the float64 oracle evaluated on the same float32-rounded inputs."""
    rng = np.random.RandomState(3)
    for scale, offset, want in [(1.0, 0.0, "product"), (1.0, 1000.0, "product"), (4.0, 0.0, "difference"), (30.0, -7.0, "difference")]:
        y = (scale * rng.rand(3000, 3) + offset).astype(np.float32).astype(np.float64)
        x = (scale * rng.rand(1111, 3) + offset).astype(np.float32).astype(np.float64)
        b = rng.randn(3000, 2)
        for norm in (False, True):
            out, extra = run_plugin("gaussian", y, x, b, normalize_rows=norm)
            assert extra["form"] == want, (scale, offset, extra)
            assert orc.rel_l2(out, c_oracle.kernel_product("gaussian", y, x, b, normalize_rows=norm)) <= TOL_DIRECT, (scale, offset, norm)


@pytest.mark.parametrize("kernel", ["gaussian", "absolute-exponential", "inverse-distance"])
@pytest.mark.parametrize("N,M", [(1, 1), (7, 513), (255, 1), (2049, 511), (4097, 1537), (300, 40000)])
def test_ragged_sizes(kernel, N, M):
    rng = np.random.RandomState(N * 131 + M)
    y, x, b = rng.rand(M, 3), rng.rand(N, 3), rng.randn(M, 1)
    out, _ = run_plugin(kernel, y, x, b)
    want = c_oracle.kernel_product(kernel, y, x, b)
    assert orc.rel_l2(out, want) <= TOL_DIRECT


@pytest.mark.parametrize("D", [1, 2, 3, 4, 5, 8, 11, 16])
@pytest.mark.parametrize("E", [1, 2, 3, 4, 5, 9])
def test_dims(D, E):
    rng = np.random.RandomState(D * 17 + E)
    r = (3.0 / max(D, 3)) ** 0.5
    y, x, b = r * rng.rand(700, D), r * rng.rand(333, D), rng.randn(700, E)
    out, _ = run_plugin("gaussian", y, x, b)
    assert orc.rel_l2(out, c_oracle.kernel_product("gaussian", y, x, b)) <= TOL_DIRECT
    out, _ = run_plugin("gaussian", y, x, b, normalize_rows=True)
    assert orc.rel_l2(out, c_oracle.kernel_product("gaussian", y, x, b, normalize_rows=True)) <= TOL_DIRECT


@pytest.mark.parametrize("kernel", ["gaussian", "absolute-exponential"])
def test_attention_survives_fp32_underflow(kernel):
    """Rows far from every source: exp(-d2) underflows in FP32 (d2 > 104) but not in the float64
    reference (d2 < 745); the online max-rescale must still normalise them."""
    rng = np.random.RandomState(5)
    y, b = rng.rand(900, 3), rng.randn(900, 2)
    x = rng.rand(64, 3) + (12.0 if kernel == "gaussian" else 150.0)
    out, _ = run_plugin(kernel, y, x, b, normalize_rows=True)
    want = orc.kernel_product(kernel, y, x, b, normalize_rows=True)
    assert np.isfinite(out).all()
    assert orc.rel_l2(out, want) <= 2e-4  # the exponent itself is ~1e3 ulps of FP32 away from zero here


def test_inverse_distance_zeroing_follows_global_rows():
    """row_offset shifts the zeroed column (bruteforce.py:12-14 works on the global flat index)."""
    import torch
    from kernel_matrix_benchmarks_b200.product import kernel_product

    g = load_golden("product_invdist_tall_d3")
    y = torch.tensor(g["source_points"], dtype=torch.float32, device="cuda")
    x = torch.tensor(g["target_points"], dtype=torch.float32, device="cuda")
    b = torch.tensor(g["source_signal"], dtype=torch.float32, device="cuda")
    lo, hi = 40, 120
    part = kernel_product(x[lo:hi].contiguous(), y, b, kernel="inverse-distance", row_offset=lo).cpu().numpy()
    assert orc.rel_l2(part, g["truth"][lo:hi]) <= TOL_DIRECT


def test_config_c1_full():
    """BASELINE config 1: Gaussian N=M=10k, D=3, E=1, all rows against the float64 oracle."""
    from kernel_matrix_benchmarks_b200 import datasets

    ds = datasets.config_c1()
    out, extra = run_plugin("gaussian", ds.source_points, None, ds.source_signal, same_points=True)
    want = c_oracle.kernel_product("gaussian", ds.source_points, None, ds.source_signal)
    err = orc.rel_l2(out, want)
    print(f"C1 rel-L2 {err:.2e} {extra}")
    assert err <= TOL_DIRECT


def test_config_c2_full_size_sampled_and_properties():
    """BASELINE config 2 at full size (N=M=1M, D=3): sampled rows against the oracle, plus
    size-independent properties: bitwise determinism, linearity in b, density == product with ones."""
    import torch
    from kernel_matrix_benchmarks_b200 import datasets
    from kernel_matrix_benchmarks_b200.product import kernel_product

    ds = datasets.config_c2()
    n = ds.N
    out, extra = run_plugin("gaussian", ds.source_points, None, ds.source_signal, same_points=True)
    rows = np.random.RandomState(0).choice(n, 768, replace=False)
    want = c_oracle.kernel_product("gaussian", ds.source_points, None, ds.source_signal, rows=rows)
    err = orc.rel_l2(out[rows], want)
    print(f"C2 sampled rel-L2 {err:.2e} {extra}")
    assert err <= TOL_DIRECT

    y = torch.tensor(ds.source_points, dtype=torch.float32, device="cuda")
    b1 = torch.tensor(ds.source_signal, dtype=torch.float32, device="cuda")
    b2 = torch.randn(n, 1, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    a1 = kernel_product(y, y, b1)
    assert torch.equal(a1, kernel_product(y, y, b1)), "stream-K combination must be deterministic"
    assert np.array_equal(a1.cpu().numpy().astype(np.float64), out)
    a2 = kernel_product(y, y, b2)
    a12 = kernel_product(y, y, 0.5 * b1 - 2.0 * b2)
    lin = (a12 - (0.5 * a1 - 2.0 * a2)).norm() / a12.norm()
    assert float(lin) <= 1e-5
    dens = kernel_product(y, y, None, density_estimation=True)
    ones = kernel_product(y, y, torch.ones_like(b1))
    assert torch.equal(dens, ones)
    att = kernel_product(y, y, torch.full_like(b1, 3.25), normalize_rows=True)
    assert float((att - 3.25).abs().max()) <= 3.25e-5  # 1e-5 relative, worst row of 10^6


def test_degenerate_attention_rows_are_nan_like_the_reference():
    """1 x 1 inverse-distance attention is 0/0: the reference returns NaN (bruteforce.py:145), so do we."""
    one = np.array([[0.3, 0.2, 0.1]])
    out, _ = run_plugin("inverse-distance", one, one, np.array([[2.0]]), same_points=True, normalize_rows=True)
    want = orc.kernel_product("inverse-distance", one, None, np.array([[2.0]]), normalize_rows=True)
    assert np.isnan(want).all() and np.isnan(out).all()


def test_density_attention_is_ones():
    g = load_golden("density_attention_gaussian_cube_d3")
    out, _ = run_plugin("gaussian", g["source_points"], None, g["source_signal"], same_points=True, normalize_rows=True, density=True)
    assert np.array_equal(out, np.ones_like(g["truth"]))


def test_c_abi_error_paths():
    import torch
    from kernel_matrix_benchmarks_b200 import _lib
    from kernel_matrix_benchmarks_b200.product import kernel_product

    lib = _lib.load()
    x = torch.rand(10, 3, device="cuda")
    b = torch.rand(10, 1, device="cuda")
    out = torch.empty(10, 1, device="cuda")
    P = lambda t: ctypes.c_void_p(t.data_ptr())
    # workspace too small
    rc = lib.kmb_product_f32(P(x), P(x), P(b), P(out), 10, 10, 3, 1, 0, 0, 0, 0, P(out), 4, None)
    assert rc == _lib.KMB_ERR_WORKSPACE and b"workspace too small" in lib.kmb_last_error()
    # NULL signal without the density flag
    rc = lib.kmb_product_f32(P(x), P(x), None, P(out), 10, 10, 3, 1, 0, 0, 0, 0, P(out), 4, None)
    assert rc == _lib.KMB_ERR_INVALID
    with pytest.raises(NotImplementedError):
        kernel_product(x, x, b, kernel="laplace")
    with pytest.raises(ValueError):
        kernel_product(x.double(), x, b)
    with pytest.raises(NotImplementedError):
        kernel_product(torch.rand(4, 20, device="cuda"), torch.rand(4, 20, device="cuda"), torch.rand(4, 1, device="cuda"), path="direct")


# ---------------------------------------------------------------- tensor-core (3xTF32) path


TENSOR_PATHS = ["tensor_f16", "tensor_tf32"]   # FP16 hi/lo operands (what "auto" picks) and the TF32 hi/lo ones


@pytest.mark.parametrize("path", TENSOR_PATHS)
@pytest.mark.parametrize("kernel", ["gaussian", "absolute-exponential", "inverse-distance"])
@pytest.mark.parametrize("N,M,D,E", [(1, 1, 17, 1), (130, 257, 33, 1), (300, 1000, 64, 2), (129, 640, 100, 5), (257, 129, 784, 1)])
def test_tensor_path_shapes(kernel, N, M, D, E, path):
    rng = np.random.RandomState(N + M + D)
    r = (3.0 / D) ** 0.5
    y, x, b = r * rng.rand(M, D), r * rng.rand(N, D), rng.randn(M, E)
    for norm in (False, True):
        out, extra = run_plugin(kernel, y, x, b, normalize_rows=norm, path=path)
        want = c_oracle.kernel_product(kernel, y, x, b, normalize_rows=norm)
        if np.isnan(want).any():  # 0/0 rows (e.g. the 1 x 1 inverse-distance matrix): the reference returns NaN too
            assert np.array_equal(np.isnan(out), np.isnan(want))
            continue
        err = orc.rel_l2(out, want)
        assert err <= TOL_TENSOR, (kernel, norm, err)


def test_tensor_path_agrees_with_direct_path_on_small_d():
    """Same D = 8 problem through both paths: FP32 FMA distances vs tcgen05 3xTF32 distances."""
    rng = np.random.RandomState(8)
    y, x, b = 0.6 * rng.rand(5000, 8), 0.6 * rng.rand(700, 8), rng.randn(5000, 2)
    want = c_oracle.kernel_product("gaussian", y, x, b)
    direct, _ = run_plugin("gaussian", y, x, b, path="direct")
    tensor, _ = run_plugin("gaussian", y, x, b, path="tensor")
    assert orc.rel_l2(direct, want) <= TOL_DIRECT
    assert orc.rel_l2(tensor, want) <= TOL_TENSOR
    assert orc.rel_l2(tensor, direct) <= TOL_TENSOR


@pytest.mark.parametrize("path", TENSOR_PATHS)
def test_tensor_path_uncentred_data(path):
    """Offset data (all coordinates near 50): the prepass centres on the source mean, so the
    cancellation in |x|^2 + |y|^2 - 2x.y stays at the scale of the spread, not of the offset."""
    rng = np.random.RandomState(9)
    y = (50.0 + 0.2 * rng.rand(2000, 64)).astype(np.float32).astype(np.float64)
    x = (50.0 + 0.2 * rng.rand(300, 64)).astype(np.float32).astype(np.float64)
    b = rng.randn(2000, 1)
    out, _ = run_plugin("gaussian", y, x, b, path=path)
    assert orc.rel_l2(out, c_oracle.kernel_product("gaussian", y, x, b)) <= TOL_TENSOR


@pytest.mark.parametrize("path", TENSOR_PATHS)
@pytest.mark.parametrize("N,M,D", [(20000, 3000, 40), (128 * 79, 256 * 9 + 1, 48), (128 * 149, 300, 20), (5000, 70000, 32)])
def test_tensor_path_wave_schedule(N, M, D, path):
    """Shapes that exercise the wave schedule: several waves, row tiles split over many CTAs (combined by
    the last CTA to arrive), a last wave with a different split, more row tiles than CTAs.  Sampled rows."""
    rng = np.random.RandomState(N + M)
    r = (3.0 / D) ** 0.5
    y, x, b = r * rng.rand(M, D), r * rng.rand(N, D), rng.randn(M, 1)
    rows = np.unique(np.concatenate([np.arange(0, N, 97), [N - 1]]))
    for norm in (False, True):
        out, _ = run_plugin("gaussian", y, x, b, normalize_rows=norm, path=path)
        want = c_oracle.kernel_product("gaussian", y, x, b, normalize_rows=norm, rows=rows)
        err = orc.rel_l2(out[rows], want)
        assert err <= TOL_TENSOR, (norm, err)
    again, _ = run_plugin("gaussian", y, x, b, normalize_rows=True, path=path)
    assert np.array_equal(again, out)   # deterministic: fixed combine order


def test_tensor_f16_scaling_range():
    """FP16 operand planes: the power-of-two scale follows the data (tiny and huge coordinates, one outlier
    column) and the result keeps FP32-class accuracy."""
    rng = np.random.RandomState(11)
    D = 48
    base_y, base_x, b = rng.rand(3000, D), rng.rand(400, D), rng.randn(3000, 1)
    r = (3.0 / D) ** 0.5
    for name, scale in (("unit", r), ("tiny", 1e-3 * r), ("wide", 4.0 * r)):
        y, x = scale * base_y, scale * base_x
        out, _ = run_plugin("gaussian", y, x, b, path="tensor_f16")
        err = orc.rel_l2(out, c_oracle.kernel_product("gaussian", y, x, b))
        assert err <= 1e-5, (name, err)
    # one far outlier among the sources stretches the scale by 2^7: the other points keep their accuracy
    y = r * base_y
    y[0, :] += 100.0 * r
    out, _ = run_plugin("gaussian", y, r * base_x, b, path="tensor_f16")
    err = orc.rel_l2(out, c_oracle.kernel_product("gaussian", y, r * base_x, b))
    assert err <= TOL_TENSOR, err


def test_prepared_points_give_the_same_product():
    """kmb_product_prepare_f32 + KMB_FLAG_PREPARED == the product doing its own prepass, bit for bit; the plugin does
    the prepass in fit(), prepares again when the workspace has to grow for a wider signal, and reuses it afterwards."""
    import torch
    from kernel_matrix_benchmarks_b200 import product
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Product

    rng = np.random.RandomState(21)
    D = 96
    r = (3.0 / D) ** 0.5
    yh, xh = r * rng.rand(3000, D), r * rng.rand(700, D)
    y = torch.tensor(yh, dtype=torch.float32, device="cuda")
    x = torch.tensor(xh, dtype=torch.float32, device="cuda")
    for E in (1, 40):
        b = torch.tensor(rng.randn(3000, E), dtype=torch.float32, device="cuda")
        plain = product.kernel_product(x, y, b, kernel="gaussian", workspace=product.Workspace())
        ws = product.Workspace()
        token = product.prepare_points(x, y, kernel="gaussian", workspace=ws,
                                       min_bytes=product.workspace_bytes(700, 3000, D, E, kernel="gaussian"))
        assert token is not None
        again = product.kernel_product(x, y, b, kernel="gaussian", workspace=ws, prepared=token)
        assert torch.equal(plain, again)
        # a stale token (the workspace was reallocated) is ignored: the product does the prepass itself
        stale = product.kernel_product(x, y, b, kernel="gaussian", workspace=product.Workspace(), prepared=token)
        assert torch.equal(plain, stale)
    assert product.prepare_points(x[:, :3].contiguous(), y[:, :3].contiguous(), kernel="gaussian") is None   # direct path: no-op

    algo = B200Product(kernel="gaussian", dimension=D, precision="float32")
    algo.prepare_data(source_points=yh, target_points=xh)
    algo.fit()
    first = algo._prepared
    assert first is not None
    outs = []
    for E in (1, 40, 40, 1):
        bh = np.random.RandomState(E).randn(3000, E)
        algo.prepare_query(source_signal=bh)
        algo.query()
        outs.append((E, algo.get_result(), algo._prepared))
        assert orc.rel_l2(outs[-1][1], c_oracle.kernel_product("gaussian", yh, xh, bh)) <= 1e-5
    assert outs[0][2] is first and outs[1][2] is not first and outs[2][2] is outs[1][2] and outs[3][2] is outs[1][2]
    assert np.array_equal(outs[1][1], outs[2][1])
    algo.done()


def test_config_c3_sampled():
    """BASELINE config 3 at full size (M = 60k sources, N = 10k targets, D = 784, E = 1):
    every 40th target row against the float64 oracle."""
    from kernel_matrix_benchmarks_b200 import datasets

    ds = datasets.config_c3()
    rows = np.arange(0, ds.N, 40)
    want = c_oracle.kernel_product("gaussian", ds.source_points, ds.target_points, ds.source_signal, rows=rows)
    for path in TENSOR_PATHS:
        out, extra = run_plugin("gaussian", ds.source_points, ds.target_points, ds.source_signal, path=path)
        err = orc.rel_l2(out[rows], want)
        print(f"C3 sampled rel-L2 {path} {err:.2e} {extra}")
        assert err <= TOL_TENSOR


def test_config_c4_reduced():
    """BASELINE config 4 (row-normalised exponential kernel, D = 64, E = 64) at N = M = 16k:
    sampled rows against the oracle; a constant signal must come back unchanged."""
    from kernel_matrix_benchmarks_b200 import datasets

    ds = datasets.config_c4(n=16384)
    out, extra = run_plugin(ds.kernel, ds.source_points, ds.target_points, ds.source_signal, normalize_rows=True)
    rows = np.arange(0, ds.N, 64)
    want = c_oracle.kernel_product(ds.kernel, ds.source_points, ds.target_points, ds.source_signal, normalize_rows=True, rows=rows)
    err = orc.rel_l2(out[rows], want)
    print(f"C4 (16k) sampled rel-L2 {err:.2e} {extra}")
    assert err <= TOL_TENSOR
    const, _ = run_plugin(ds.kernel, ds.source_points, ds.target_points, np.full((ds.M, 1), -2.5), normalize_rows=True)
    assert np.abs(const + 2.5).max() <= 2.5e-5


def test_config_c4_full_size_sampled():
    """BASELINE config 4 at FULL size (N = M = 262 144, D = 64, E = 64, row-normalised exponential kernel): 2048 row
    tiles in 14 waves of CTA pairs -- the schedule the reduced case never reaches.  256 sampled target rows (every
    1024th, shifted so that first/last tiles and both CTAs of a pair are hit) against the float64 C oracle."""
    from kernel_matrix_benchmarks_b200 import datasets

    ds = datasets.config_c4()
    assert (ds.N, ds.M, ds.D, ds.E) == (262144, 262144, 64, 64)
    rows = np.unique(np.concatenate((np.arange(0, ds.N, 1024) + (np.arange(256) * 37) % 1024, [0, 127, 128, 255, ds.N - 1])))
    want = c_oracle.kernel_product(ds.kernel, ds.source_points, ds.target_points, ds.source_signal, normalize_rows=True, rows=rows)
    for kernel in (ds.kernel, "gaussian"):
        if kernel != ds.kernel:
            want = c_oracle.kernel_product(kernel, ds.source_points, ds.target_points, ds.source_signal, normalize_rows=True, rows=rows)
        out, extra = run_plugin(kernel, ds.source_points, ds.target_points, ds.source_signal, normalize_rows=True)
        assert out.shape == (ds.N, ds.E) and np.isfinite(out).all()
        err = orc.rel_l2(out[rows], want)
        worst = np.max(np.linalg.norm(out[rows] - want, axis=1) / np.linalg.norm(want, axis=1))
        print(f"C4 full size {kernel}: sampled rel-L2 {err:.2e} (worst row {worst:.2e}) over {len(rows)} rows {extra}")
        assert err <= TOL_TENSOR and worst <= 5 * TOL_TENSOR


@pytest.mark.parametrize("kernel, path, norm", [("inverse-distance", "auto", False), ("inverse-distance", "auto", True),
                                                ("gaussian", "tensor_tf32", True), ("gaussian", "auto", False)])
def test_wide_signal_tensor_kernels_over_many_source_blocks(kernel, path, norm):
    """M = 262 144 sources against a few row tiles, D = 64, E = 16: the P.B accumulators of the E > 4 tensor kernels
    (kprod_tensor_pv.cu for the inverse-distance kernel and the TF32 planes, kprod_tensor_pv16.cu otherwise) collect
    thousands of source blocks per row tile.  The tensor cores truncate when they add into the FP32 accumulator, which
    grew to 2.4e-4 relative at this M before the accumulators were flushed to FP32 sums every few dozen blocks."""
    rng = np.random.RandomState(17)
    m, n, d, e = 262_144, 384, 64, 16
    r = (3.0 / d) ** 0.5
    y, x, b = r * rng.rand(m, d), r * rng.rand(n, d), rng.randn(m, e)
    out, extra = run_plugin(kernel, y, x, b, normalize_rows=norm, path=path)
    rows = np.arange(0, n, 3)
    want = c_oracle.kernel_product(kernel, y, x, b, normalize_rows=norm, rows=rows)   # global row indices: inverse-distance zeroing
    err = orc.rel_l2(out[rows], want)
    print(f"{kernel} path={path} norm={norm}: rel-L2 {err:.2e} {extra}")
    assert err <= 0.5 * TOL_TENSOR


@pytest.mark.parametrize("kernel", ["gaussian", "absolute-exponential"])
def test_wide_signal_with_small_d_takes_the_tensor_kernel(kernel):
    """D <= 16 with E >= 32 under path="auto": K b is a dense contraction, so the P.B kernel (tcgen05, FP16 planes) runs
    instead of ceil(E / 16) passes of the direct kernel (6x faster at D = 3, E = 64); path="direct" keeps the FP32 kernel."""
    rng = np.random.RandomState(23)
    y, x, b = rng.rand(3000, 3), rng.rand(700, 3), rng.randn(3000, 64)
    for norm in (False, True):
        want = c_oracle.kernel_product(kernel, y, x, b, normalize_rows=norm)
        out, extra = run_plugin(kernel, y, x, b, normalize_rows=norm)
        assert extra["path_used"] == "tensor_f16" and extra["form"] == "n/a", extra
        assert orc.rel_l2(out, want) <= TOL_TENSOR
        out, extra = run_plugin(kernel, y, x, b, normalize_rows=norm, path="direct")
        assert extra["path_used"] == "direct"
        assert orc.rel_l2(out, want) <= TOL_DIRECT
    out, extra = run_plugin(kernel, y, x, b[:, :16].copy())
    assert extra["path_used"] == "direct"


def test_empty_row_shard_is_a_no_op():
    """shard_bounds gives the last ranks empty shards when ceil(n / world) * rank >= n (n = 9 on 8 ranks): the C ABI
    must treat N == 0 as a no-op even though an empty tensor has a NULL data pointer (every other rank would
    otherwise hang in the next collective)."""
    import torch
    from kernel_matrix_benchmarks_b200 import product
    from kernel_matrix_benchmarks_b200.solver import shard_bounds

    y = torch.rand(9, 3, device="cuda")
    b = torch.rand(9, 1, device="cuda")
    lo, hi, _ = shard_bounds(9, 7, 8)
    assert lo == hi
    out = product.kernel_product(y[lo:hi], y, b)
    assert out.shape == (0, 1)
    out64 = product.kernel_product_f64(y[lo:hi].double(), y.double(), b.double())
    assert out64.shape == (0, 1)


# ------------------------------------------- tensor path with the second contraction on tcgen05 (E > 4)


@pytest.mark.parametrize("path", TENSOR_PATHS)
@pytest.mark.parametrize("kernel", ["gaussian", "absolute-exponential", "inverse-distance"])
@pytest.mark.parametrize("norm", [False, True])
@pytest.mark.parametrize("N,M,D,E", [(100, 20000, 64, 64), (300, 1000, 32, 5), (129, 641, 100, 33), (1000, 130, 128, 70),
                                     (128 * 150 + 3, 700, 48, 8)])
def test_tensor_pv_shapes(kernel, norm, N, M, D, E, path):
    """P.B on the tensor cores: one row tile split over many CTAs (combined by the last to arrive), ragged
    sizes, E not a multiple of 32, two passes over the signal (E > 64), more row tiles than CTAs.
    tensor_f16: kprod_tensor_pv16 (inverse-distance: the TF32 kernel); tensor_tf32: kprod_tensor_pv."""
    rng = np.random.RandomState(N + M + D + E)
    r = (3.0 / D) ** 0.5
    y, x, b = r * rng.rand(M, D), r * rng.rand(N, D), rng.randn(M, E) * (1.0 + 100.0 * (np.arange(E) % 3 == 0))
    out, _ = run_plugin(kernel, y, x, b, normalize_rows=norm, path=path)
    want = c_oracle.kernel_product(kernel, y, x, b, normalize_rows=norm)
    assert out.shape == want.shape
    assert orc.rel_l2(out, want) <= TOL_TENSOR
    # every column on its own: the columns scaled by 101 carry ~99 % of the norm and would hide the others
    col_err = np.linalg.norm(out - want, axis=0) / np.linalg.norm(want, axis=0)
    assert col_err.max() <= 10 * TOL_TENSOR, (int(col_err.argmax()), col_err.max())


@pytest.mark.parametrize("path", TENSOR_PATHS)
@pytest.mark.parametrize("kernel", ["gaussian", "absolute-exponential"])
def test_tensor_pv_lazy_rescale(kernel, path):
    """Sources ordered far -> near: the running reference exponent must be rescaled (growth > 2^64)
    and rows that only ever see far sources must still normalise (FP32 exp would underflow)."""
    rng = np.random.RandomState(4)
    D, E = 64, 16
    far = 4.0 if kernel == "gaussian" else 30.0
    near = 0.2 * rng.rand(500, D)
    y = np.concatenate((near + far / np.sqrt(D) * 3, near + far / np.sqrt(D), near), axis=0)  # far, closer, near
    x = np.concatenate((0.2 * rng.rand(200, D), 0.2 * rng.rand(56, D) - far / np.sqrt(D)), axis=0)
    b = rng.randn(y.shape[0], E)
    out, _ = run_plugin(kernel, y, x, b, normalize_rows=True, path=path)
    want = orc.kernel_product(kernel, y, x, b, normalize_rows=True)
    assert np.isfinite(out).all()
    assert orc.rel_l2(out, want) <= 5e-4  # |u||v| ~ 1e4 here: the 3xTF32 cancellation error of d^2 is ~1e-2


@pytest.mark.parametrize("norm", [False, True])
@pytest.mark.parametrize("kernel", ["gaussian", "absolute-exponential"])
def test_tensor_pv16_reference_moves_block_after_block(kernel, norm):
    """Sources sorted from far to near in small steps: the lazy reference of every row moves in many of the 128-source
    blocks of a row tile, so the fused pass of kprod_tensor_pv16 (exponent with the reference the row already has) is
    redone in two phases again and again, with accumulators to rescale and long accumulators already flushed
    (M > 64 blocks).  E = 64, D = 64: the shape of config C4."""
    rng = np.random.RandomState(11)
    D, E, M, N = 64, 64, 128 * 150 + 37, 300
    step = np.linspace(6.0 if kernel == "gaussian" else 40.0, 0.0, M)[:, None] / np.sqrt(D)   # distance to the targets shrinks
    y = 0.15 * rng.rand(M, D) + step
    x = 0.15 * rng.rand(N, D)
    b = rng.randn(M, E)
    out, extra = run_plugin(kernel, y, x, b, normalize_rows=norm, path="tensor")
    assert extra["path_used"] == "tensor_f16"
    want = orc.kernel_product(kernel, y, x, b, normalize_rows=norm)
    assert np.isfinite(out).all()
    # exponential kernel: the sources span 40 length units, |u||v| ~ 300 in log2 units, and the cancellation error of the
    # three-term d^2 (2^-22 |u||v|) goes through a square root at the near sources -- as in test_tensor_pv_lazy_rescale
    assert orc.rel_l2(out, want) <= (TOL_TENSOR if kernel == "gaussian" else 5e-4)


@pytest.mark.parametrize("M", [1, 63, 64, 65, 127, 129, 200])
@pytest.mark.parametrize("kernel", ["gaussian", "absolute-exponential"])
def test_tensor_pv16_padded_sources_weigh_nothing(kernel, M):
    """Blocks that are partly or (for one column group) wholly padding: padded sources carry |v|^2 = 3.39e38 and must come
    out as exact zero weights without a branch, whatever the row's reference exponent is (also when a group never sees a
    real source: M <= 64)."""
    rng = np.random.RandomState(M)
    D, E, N = 64, 40, 260
    r = (3.0 / D) ** 0.5
    y, x, b = r * rng.rand(M, D), r * rng.rand(N, D), rng.randn(M, E)
    for norm in (False, True):
        out, _ = run_plugin(kernel, y, x, b, normalize_rows=norm, path="tensor")
        want = orc.kernel_product(kernel, y, x, b, normalize_rows=norm)
        assert np.isfinite(out).all()
        assert orc.rel_l2(out, want) <= TOL_TENSOR


# ---- symmetric (same_points) Gaussian product: kprod_sym --------------------------------------------

def _sym_case(n, D, radius=1.0, kernel="gaussian", round_inputs=False):
    from kernel_matrix_benchmarks_b200 import datasets

    ds = datasets.uniform_cube(n, D, radius, kernel)
    if round_inputs:   # singular kernels: compare on the float32-rounded points the GPU sees (as test_gaussian_form_selection does)
        ds.source_points = ds.target_points = ds.source_points.astype(np.float32).astype(np.float64)
    rows = np.unique(np.concatenate([np.arange(0, n, max(1, n // 192)), [0, n - 1, n // 2]]))
    want = orc.kernel_product(kernel, ds.source_points, None, ds.source_signal, rows=rows)
    return ds, rows, want


@pytest.mark.parametrize("n, D", [(300, 3), (4096, 2), (5000, 1), (40000, 3), (65553, 2), (131072 + 5, 3)])
def test_symmetric_product_matches_oracle(n, D):
    """kmb_product_f32(path=DIRECT_SYM) == K b of bruteforce.py:25-58,153 with target_points=None."""
    import torch
    from kernel_matrix_benchmarks_b200 import product

    ds, rows, want = _sym_case(n, D)
    y = torch.tensor(ds.source_points, dtype=torch.float32, device="cuda")
    b = torch.tensor(ds.source_signal, dtype=torch.float32, device="cuda")
    got = product.kernel_product(y, y, b, path="direct_sym").cpu().numpy().astype(np.float64)
    assert got.shape == (n, 1)
    assert orc.rel_l2(got[rows], want) <= TOL_DIRECT
    # row-by-row against the general kernel on all rows (catches a wrong tile / column block)
    ref = product.kernel_product(y, y, b, path="direct").cpu().numpy().astype(np.float64)
    assert np.max(np.abs(got - ref)) <= 2e-5 * np.max(np.abs(ref))


@pytest.mark.parametrize("kernel", ["absolute-exponential", "inverse-distance"])
@pytest.mark.parametrize("n, D", [(300, 3), (5000, 2), (40000, 3), (65553 + 4096, 3)])
def test_symmetric_product_other_kernels(kernel, n, D):
    """Every kernel of bruteforce.py:18-22 is symmetric (inverse-distance: zero diagonal when N == M, :12-14): the
    difference form of kprod_sym against the oracle and, row by row, against the general kernel.  (1 / |x - y| is
    dominated by the nearest neighbours, whose distances move by 1e-3 relative when the coordinates are rounded to float32:
    the oracle therefore sees the rounded points, and D = 1 -- where 7 10^4 float32 points collide -- is left out.)"""
    import torch
    from kernel_matrix_benchmarks_b200 import product

    ds, rows, want = _sym_case(n, D, kernel=kernel, round_inputs=True)
    y = torch.tensor(ds.source_points, dtype=torch.float32, device="cuda")
    b = torch.tensor(ds.source_signal, dtype=torch.float32, device="cuda")
    got = product.kernel_product(y, y, b, kernel=kernel, path="direct_sym").cpu().numpy().astype(np.float64)
    assert got.shape == (n, 1) and np.isfinite(got).all()
    assert orc.rel_l2(got[rows], want) <= TOL_DIRECT
    ref = product.kernel_product(y, y, b, kernel=kernel, path="direct").cpu().numpy().astype(np.float64)
    assert np.max(np.abs(got - ref)) <= 2e-5 * np.max(np.abs(ref))
    parts = sum(product.kernel_product_sym_part(y, b, p, 3, kernel=kernel).double() for p in range(3)).cpu().numpy()
    assert orc.rel_l2(parts[rows], want) <= TOL_DIRECT
    # density estimation (b == 1, bruteforce.py:150) through the same kernels
    dens = product.kernel_product(y, y, None, kernel=kernel, density_estimation=True, path="direct_sym").cpu().numpy().astype(np.float64)
    want_d = orc.kernel_product(kernel, ds.source_points, None, None, density_estimation=True, rows=rows)
    assert orc.rel_l2(dens[rows], want_d) <= TOL_DIRECT


def test_symmetric_workspace_is_linear_in_n():
    """The hand-over buffers are O(n sqrt(CTAs)) floats (strip order), not one column vector per row tile."""
    from kernel_matrix_benchmarks_b200 import _lib

    lib, need = _lib.load(), ctypes.c_size_t(0)
    _lib.check(lib.kmb_product_sym_workspace_bytes(1_000_000, 3, 0, 1, ctypes.byref(need)))
    assert need.value < 200 << 20, need.value          # was 0.98 GB of column sums
    _lib.check(lib.kmb_product_sym_workspace_bytes(4_000_000, 3, 0, 1, ctypes.byref(need)))
    assert need.value < 1 << 30, need.value            # was 15.6 GB
    _lib.check(lib.kmb_product_sym_workspace_bytes(10_000_000, 3, 3, 8, ctypes.byref(need)))
    assert need.value < 2 << 30, need.value


def test_symmetric_product_at_4m_points():
    """N = 4 10^6 (beyond what the per-tile column buffers of round 1 allowed within a few GB): sampled rows vs the C oracle."""
    import torch
    from kernel_matrix_benchmarks_b200 import datasets, product
    from oracle import c_oracle

    n = 4_000_000
    ds = datasets.uniform_cube(n, 3, 1.0, "gaussian")
    rows = np.sort(np.random.RandomState(5).choice(n, 64, replace=False))
    want = c_oracle.kernel_product("gaussian", ds.source_points, None, ds.source_signal, rows=rows)
    y = torch.tensor(ds.source_points, dtype=torch.float32, device="cuda")
    b = torch.tensor(ds.source_signal, dtype=torch.float32, device="cuda")
    ws = product.Workspace()
    got = product.kernel_product(y, y, b, path="direct_sym", workspace=ws)
    assert ws.buf.numel() < 1 << 30
    got = got[torch.as_tensor(rows, device="cuda")].cpu().numpy().astype(np.float64)
    assert orc.rel_l2(got, want) <= TOL_DIRECT


@pytest.mark.parametrize("n_parts", [2, 3, 8])
def test_symmetric_parts_add_up(n_parts):
    """The unit list cut into n_parts ranges (one per GPU): the partial outputs sum to the product."""
    import torch
    from kernel_matrix_benchmarks_b200 import product

    ds, rows, want = _sym_case(50000, 3)
    y = torch.tensor(ds.source_points, dtype=torch.float32, device="cuda")
    b = torch.tensor(ds.source_signal, dtype=torch.float32, device="cuda")
    total = torch.zeros((ds.N, 1), dtype=torch.float64, device="cuda")
    for part in range(n_parts):
        total += product.kernel_product_sym_part(y, b, part, n_parts).double()
    assert orc.rel_l2(total.cpu().numpy()[rows], want) <= TOL_DIRECT


def test_symmetric_falls_back_to_difference_form_on_spread_data():
    import torch
    from kernel_matrix_benchmarks_b200 import product

    ds, rows, want = _sym_case(20000, 3, radius=6.0)
    y = torch.tensor(ds.source_points, dtype=torch.float32, device="cuda")
    b = torch.tensor(ds.source_signal, dtype=torch.float32, device="cuda")
    got = product.kernel_product(y, y, b, path="direct_sym").cpu().numpy().astype(np.float64)
    assert product.direct_stats()["form"] == "difference"
    assert orc.rel_l2(got[rows], want) <= TOL_DIRECT
    parts = sum(product.kernel_product_sym_part(y, b, p, 3).double() for p in range(3)).cpu().numpy()
    assert orc.rel_l2(parts[rows], want) <= TOL_DIRECT


def test_symmetric_is_deterministic_and_checks_its_arguments():
    import torch
    from kernel_matrix_benchmarks_b200 import _lib, product

    ds, _, _ = _sym_case(40000, 3)
    y = torch.tensor(ds.source_points, dtype=torch.float32, device="cuda")
    b = torch.tensor(ds.source_signal, dtype=torch.float32, device="cuda")
    a1 = product.kernel_product(y, y, b, path="direct_sym").clone()
    a2 = product.kernel_product(y, y, b, path="direct_sym").clone()
    assert torch.equal(a1, a2)
    with pytest.raises(ValueError):  # a copy of the points is not "the same points"
        product.kernel_product(y.clone(), y, b, path="direct_sym")
    with pytest.raises(NotImplementedError):   # attention is not symmetric
        product.kernel_product(y, y, b, normalize_rows=True, path="direct_sym")
    need = ctypes.c_size_t(0)
    lib = _lib.load()
    assert lib.kmb_product_sym_workspace_bytes(40000, 4, 0, 1, ctypes.byref(need)) == _lib.KMB_ERR_UNSUPPORTED
    assert lib.kmb_product_sym_workspace_bytes(40000, 3, 2, 2, ctypes.byref(need)) == _lib.KMB_ERR_INVALID


def test_plugin_takes_the_symmetric_path_for_same_points():
    """runner.py passes same_points=True together with target_points == source_points (runner.py:77-84)."""
    ds, rows, want = _sym_case(40000, 3)
    out, extra = run_plugin("gaussian", ds.source_points, ds.source_points, ds.source_signal, same_points=True)
    assert extra["path_used"] == "direct_sym" and extra["form"] == "product"
    assert orc.rel_l2(out[rows], want) <= TOL_DIRECT
    # without the flag the arrays are copied separately and the general kernel runs
    out2, extra2 = run_plugin("gaussian", ds.source_points, ds.source_points.copy(), ds.source_signal, same_points=False)
    assert extra2["path_used"] != "direct_sym"
    assert orc.rel_l2(out2[rows], want) <= TOL_DIRECT


# ---- precision variants of the plugin (bruteforce.py:64-87; algos.yaml:156-162 sweeps float16/32/64) -----

def run_plugin_precision(precision, g, **kw):
    from kernel_matrix_benchmarks_b200.algorithms.b200 import B200Product

    algo = B200Product(kernel=g["kernel"], dimension=g["source_points"].shape[1], normalize_rows=g["normalize_rows"],
                       precision=precision, **kw)
    try:
        algo.prepare_data(source_points=g["source_points"], target_points=g["target_points"], same_points=g["same_points"],
                          density_estimation=g["density_estimation"])
        algo.fit()
        algo.prepare_query(source_signal=g["source_signal"])
        algo.query()
        return algo.get_result(), algo.get_additional(), str(algo)
    finally:
        algo.done()


@pytest.mark.parametrize("name", PRODUCT_CASES)
def test_float64_precision_matches_reference_float64(name):
    """precision=float64: the reference's own float64 outputs (tests/golden) to round-off -- every golden case, also
    D = 64 / D = 784 (the tiled float64 kernel: what the ground truth of the C3 / C4 datasets is written with)."""
    g = load_golden(name)
    out, extra, label = run_plugin_precision("float64", g)
    assert out.dtype == np.float64 and out.shape == g["truth"].shape and "float64" in label
    assert extra["path_used"] in ("direct_f64", "None") or g["normalize_rows"] and g["density_estimation"]
    if np.isnan(g["truth"]).any():
        assert np.array_equal(np.isnan(out), np.isnan(g["truth"]))
    else:
        assert orc.rel_l2(out, g["truth"]) <= 1e-12


def test_float64_precision_properties_at_size():
    from kernel_matrix_benchmarks_b200 import datasets

    ds = datasets.uniform_cube(20000, 3, 1.0, "gaussian")
    g = dict(kernel="gaussian", source_points=ds.source_points, target_points=ds.source_points, source_signal=ds.source_signal,
             same_points=True, normalize_rows=False, density_estimation=False)
    out, _, _ = run_plugin_precision(np.float64, g)
    rows = np.arange(0, 20000, 100)
    want = orc.kernel_product("gaussian", ds.source_points, None, ds.source_signal, rows=rows)
    assert orc.rel_l2(out[rows], want) <= 1e-13


def test_float64_wide_kernel_ragged_shapes():
    """The tiled float64 kernel (D > 16): tile edges in N, M, D and E, more than 64 signal columns (two passes), all three
    kernels incl. the inverse-distance zeroing rule with a row offset that is not a multiple of the tile."""
    import torch
    from kernel_matrix_benchmarks_b200 import product

    rng = np.random.RandomState(8)
    for kernel, N, M, D, E, norm in (("gaussian", 65, 130, 17, 1, False), ("absolute-exponential", 200, 63, 100, 70, True),
                                     ("inverse-distance", 150, 37, 33, 3, False), ("gaussian", 1, 1, 784, 1, False)):
        r = (3.0 / D) ** 0.5
        y, x, b = r * rng.rand(M, D), r * rng.rand(N, D), rng.randn(M, E)
        want = orc.kernel_product(kernel, y, x, b, normalize_rows=norm)
        got = product.kernel_product_f64(torch.tensor(x, device="cuda"), torch.tensor(y, device="cuda"), torch.tensor(b, device="cuda"),
                                         kernel=kernel, normalize_rows=norm).cpu().numpy()
        assert got.shape == want.shape and orc.rel_l2(got, want) <= 1e-12, (kernel, N, M, D, E)
    # sharded rows: the zeroing rule follows the global row index
    y, x, b = rng.rand(37, 20), rng.rand(150, 20), rng.randn(37, 2)
    want = orc.kernel_product("inverse-distance", y, x, b)
    lo = 70
    got = product.kernel_product_f64(torch.tensor(x[lo:], device="cuda"), torch.tensor(y, device="cuda"), torch.tensor(b, device="cuda"),
                                     kernel="inverse-distance", row_offset=lo).cpu().numpy()
    assert orc.rel_l2(got, want[lo:]) <= 1e-12


def test_float16_precision_rounds_the_inputs_like_the_reference():
    """precision=float16: inputs go through half precision (bruteforce.py:100-106 astype), arithmetic in FP32."""
    g = load_golden(PRODUCT_CASES[0]) if False else None
    from kernel_matrix_benchmarks_b200 import datasets

    ds = datasets.uniform_cube(4096, 3, 1.0, "gaussian")
    g = dict(kernel="gaussian", source_points=ds.source_points, target_points=ds.source_points, source_signal=ds.source_signal,
             same_points=True, normalize_rows=False, density_estimation=False)
    out, _, label = run_plugin_precision("float16", g)
    y16 = ds.source_points.astype(np.float16).astype(np.float64)
    b16 = ds.source_signal.astype(np.float16).astype(np.float64)
    want = orc.kernel_product("gaussian", y16, None, b16)
    assert "float16" in label
    assert orc.rel_l2(out, want) <= TOL_DIRECT
    # and it is a float16-class result w.r.t. the unrounded problem (the reference's own float16 run: ~1e-3)
    exact = orc.kernel_product("gaussian", ds.source_points, None, ds.source_signal)
    assert 1e-5 < orc.rel_l2(out, exact) < 5e-3
