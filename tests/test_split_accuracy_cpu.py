"""The arithmetic claim behind the tensor path, checked on the CPU with NumPy: a three-term hi/lo split of the operands
(hi.hi + hi.lo + lo.hi, accumulated in higher precision) reproduces FP32-class dot products, both with TF32 planes
(KMB_PATH_TENSOR_3XTF32) and with FP16 planes of power-of-two scaled data (KMB_PATH_TENSOR_3XF16: the scale the device
prepass picks puts the largest operand in [2^13, 2^14)).  DESIGN.md section 7 states the error model tested here."""
import numpy as np
import pytest


def split_f16(w):
    """What split_points_f16_kernel does: p with 2^p max|w| in [2^13, 2^14); hi = fp16(2^p w), lo = fp16(2^p w - hi)."""
    p = 13 - int(np.floor(np.log2(np.abs(w).max())))
    s = np.float32(w) * np.float32(2.0 ** p)
    hi = s.astype(np.float16)
    lo = (s - hi.astype(np.float32)).astype(np.float16)
    return hi.astype(np.float64), lo.astype(np.float64), 2.0 ** (-2 * p)


def signal_scale(m):
    """What signal_scale_kernel (kprod_tensor_pv16.cu) does for a signal column whose largest |b| is m: q = 13 - ilogb(m),
    clamped to [-114, 126], the range in which 2^q and 2^-q are both finite FP32 normals."""
    q = 13 - (np.frexp(np.float32(m))[1] - 1) if 0 < m < np.inf else 0
    return int(np.clip(q, -114, 126))


def test_signal_scale_maps_every_normal_column_into_fp16_range():
    """The FP16 signal planes of kprod_tensor_pv16 hold 2^q b per column.  For every column whose largest |b| is an FP32
    normal number, 2^q max|b| lands in [2^13, 2^14) (in [1, 2^14) below 2^-113), so hi never overflows FP16 (65504) and
    hi + lo keep 22 bits of the column's largest value: lo never sinks into FP16 subnormals far enough to lose them.  The
    earlier clamp to [-100, 100] put max|b| = 1e35 at 7.9e4 (hi = inf, lo = -inf: NaN results) and max|b| = 1e-36 at 1.3e-6
    (hi an FP16 subnormal: ~2e-2 relative)."""
    rng = np.random.RandomState(9)
    tiny = np.finfo(np.float32).tiny
    for k in range(-126, 128):
        m = np.float32(2.0 ** k * rng.uniform(1.0, 1.99))
        q = signal_scale(m)
        s, inv = np.float32(2.0 ** q), np.float32(2.0 ** -q)
        assert np.isfinite(s) and np.isfinite(inv) and s >= tiny and inv >= tiny, k
        top = float(m) * 2.0 ** q
        assert (2.0 ** 13 <= top < 2.0 ** 14) if m >= 2.0 ** -113 else (1.0 <= top < 2.0 ** 14), (k, top)
        col = np.float32(m) * np.float32(rng.uniform(-1.0, 1.0, 2000))
        col[0] = m
        v = col * s                                      # exact: a power of two
        hi = v.astype(np.float16)
        lo = (v - hi.astype(np.float32)).astype(np.float16)
        assert np.isfinite(hi).all() and np.isfinite(lo).all(), k
        rec = hi.astype(np.float64) + lo.astype(np.float64)
        assert np.abs(rec - v.astype(np.float64)).max() <= 2.0 ** -22 * top, k
    old = lambda m: int(np.clip(13 - (np.frexp(np.float32(m))[1] - 1), -100, 100))   # noqa: E731
    assert np.float32(1e35) * 2.0 ** old(1e35) > 65504 and np.float32(1e-36) * 2.0 ** old(1e-36) < 2.0 ** -14


def to_tf32(x):
    """cvt.rna.tf32.f32: round to nearest (ties away) on the 13 dropped mantissa bits."""
    u = np.float32(x).view(np.uint32).astype(np.uint64)
    u = ((u + 0x1000) & 0xFFFFE000).astype(np.uint32)
    return u.view(np.float32)


def split_tf32(w):
    hi = to_tf32(w)
    lo = to_tf32(np.float32(w) - hi)
    return hi.astype(np.float64), lo.astype(np.float64), 1.0


def three_term(split, u, v):
    uh, ul, su = split(u)
    vh, vl, sv = split(v)
    assert su == sv
    return (uh @ vh.T + uh @ vl.T + ul @ vh.T) * su


@pytest.mark.parametrize("split", [split_f16, split_tf32])
@pytest.mark.parametrize("D", [64, 784])
def test_three_term_split_is_fp32_class(split, D):
    rng = np.random.RandomState(D)
    r = (3.0 / D) ** 0.5
    pts = np.float32(r * rng.rand(400, D))
    pts = (pts - pts.mean(0)).astype(np.float32)      # the prepass centres on the column means
    u, v = pts[:150], pts[150:]
    if split is split_f16:   # one common scale for both operand sets, as the prepass uses
        both = lambda w: split_f16(np.concatenate([w, pts]))   # noqa: E731
        uh, ul, s = both(u); vh, vl, _ = both(v)
        got = (uh[:150] @ vh[:250].T + uh[:150] @ vl[:250].T + ul[:150] @ vh[:250].T) * s
    else:
        got = three_term(split, u, v)
    exact = u.astype(np.float64) @ v.astype(np.float64).T
    scale = np.linalg.norm(u, axis=1)[:, None] * np.linalg.norm(v, axis=1)[None, :]
    err = np.abs(got - exact) / scale
    assert err.max() <= 2.0 ** -20, err.max()         # dropped lo.lo term + plane rounding: ~2^-22 per product
    # the squared distances the kernel forms from it keep 1e-6 of the typical distance
    d2 = (u.astype(np.float64) ** 2).sum(1)[:, None] + (v.astype(np.float64) ** 2).sum(1)[None, :] - 2 * got
    d2_exact = ((u[:, None, :].astype(np.float64) - v[None, :, :]) ** 2).sum(-1)
    assert np.abs(d2 - d2_exact).max() <= 2e-6 * d2_exact.mean()


def test_f16_planes_with_an_outlier_and_tiny_coordinates():
    """One far point stretches the power-of-two scale; coordinates far below the largest fall into FP16 subnormals for
    lo.  The absolute error stays at 2^-24 of the LARGEST operand, i.e. the accuracy of the bulk degrades gracefully
    (what tests/test_product_gpu.py::test_tensor_f16_scaling_range sees on the device)."""
    rng = np.random.RandomState(1)
    D = 48
    pts = np.float32(0.25 * rng.rand(300, D))
    pts[0] += 25.0                                     # outlier, 100x the spread
    pts[:, 5] *= 1e-4                                  # one tiny column
    hi, lo, s = split_f16(pts)
    rec = (hi + lo) * np.sqrt(s)
    big = np.abs(pts).max()
    assert np.abs(rec - pts).max() <= big * 2.0 ** -23
    got = (hi @ hi.T + hi @ lo.T + lo @ hi.T) * s
    exact = pts.astype(np.float64) @ pts.astype(np.float64).T
    bulk = slice(1, None)
    assert np.abs(got - exact)[bulk, bulk].max() <= big * np.abs(pts[1:]).max() * D * 2.0 ** -22


def test_per_group_lazy_online_softmax_merges_exactly():
    """The epilogue of kprod_tensor_pv16 restated: four column groups keep independent running sums with LAZY reference
    exponents (rescaled only when the block maximum outgrows the reference by 2^8), weights split into FP16 hi + lo,
    merged at the end with 2^(ref_g - ref).  Against the plain row-normalised product in float64."""
    rng = np.random.RandomState(3)
    n_rows, n_src, E, block, groups, lazy = 16, 2048, 8, 128, 4, 8.0
    # log2 kernel values with a strong trend (far -> near sources) so that references must move, plus rows that only
    # ever see tiny values (FP32 exp would underflow)
    logk = -40.0 * rng.rand(n_rows, n_src) - np.linspace(300.0, 0.0, n_src)[None, :]
    logk[3] -= 400.0
    b = rng.randn(n_src, E)
    want = (np.exp2(logk - logk.max(1, keepdims=True)) @ b) / np.exp2(logk - logk.max(1, keepdims=True)).sum(1, keepdims=True)

    O = np.zeros((groups, n_rows, E)); ks = np.zeros((groups, n_rows)); ref = np.full((groups, n_rows), -np.inf)
    for j0 in range(0, n_src, block):
        for g in range(groups):
            cols = slice(j0 + 32 * g, j0 + 32 * g + 32)
            s = logk[:, cols]
            cm = s.max(1)
            first = np.isinf(ref[g])
            need = ~first & (cm > ref[g] + lazy)
            sc = np.where(need, np.exp2(ref[g] - cm), 1.0)
            O[g] *= sc[:, None]; ks[g] *= sc
            ref[g] = np.where(first | need, cm, ref[g])
            p = np.float32(np.exp2(s - ref[g][:, None]))
            assert p.max() <= 2.0 ** lazy * 1.0001          # fits FP16 with room to spare
            hi = (p.view(np.uint32) & 0xFFFFE000).view(np.float32)   # 11 significant bits: exact in FP16
            lo = (p - hi).astype(np.float16).astype(np.float64)
            assert np.array_equal(hi.astype(np.float16).astype(np.float32), np.where(hi >= 2.0 ** -14, hi, hi.astype(np.float16).astype(np.float32)))
            O[g] += (hi.astype(np.float16).astype(np.float64) + lo) @ b[cols]
            ks[g] += p.astype(np.float64).sum(1)
    rmax = ref.max(0)
    w = np.exp2(ref - rmax[None, :])
    got = (w[:, :, None] * O).sum(0) / (w * ks).sum(0)[:, None]
    assert np.abs(got - want).max() <= 2e-6 * np.abs(want).max()


# ---- the squared norms as one more (BF16) K step of the S contraction, and the F2FP + FHADD split of the weights ------
# (kprod_tensor_pv16.cu: norm_tiles_kernel, the `weight` step of the epilogue) restated in NumPy

def to_bf16(x):
    """__float2bfloat16_rn: round to nearest even on the 16 dropped bits (finite inputs)."""
    u = np.float32(x).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32)


def norm_pieces(val):
    """Three BF16 pieces of val, each the rounding of what is left (norm_tiles_kernel)."""
    val = np.float32(val)
    pieces = []
    for _ in range(3):
        p = to_bf16(val)
        pieces.append(p)
        val = np.float32(val - p)
    return pieces


def test_three_bf16_pieces_carry_a_squared_norm_to_fp32_precision():
    rng = np.random.RandomState(3)
    # -|u|^2 / sscale for data scaled into [2^13, 2^14) per coordinate, D = 1 ... 128; and tiny / zero norms
    val = -np.float32(np.concatenate([rng.rand(20000) * 128 * 2.0 ** 28, rng.rand(2000) * 1e-3, [0.0, 1.0, 2.0 ** 34]]))
    p0, p1, p2 = norm_pieces(val)
    back = p0.astype(np.float64) + p1.astype(np.float64) + p2.astype(np.float64)
    nz = val != 0
    assert np.abs(back[nz] - val[nz].astype(np.float64)).max() <= 0   # 8 + 8 + 8 significant bits: the FP32 value exactly
    assert (back[~nz] == 0).all()
    # what the tensor cores add up for one (row, source): the ones columns pick the pieces of both norms, in FP32
    un, vn = val[:1000].astype(np.float64), val[1000:2000].astype(np.float64)
    a, b = norm_pieces(val[:1000]), norm_pieces(val[1000:2000])
    acc = sum(x.astype(np.float64) for x in a) + sum(x.astype(np.float64) for x in b)
    assert np.abs(acc - (un + vn)).max() == 0


def test_padded_sources_get_a_finite_marker_that_no_norm_can_offset():
    p0, p1, p2 = norm_pieces(np.float32(-3.0e38))
    back = float(p0) + float(p1) + float(p2)
    assert np.isfinite([p0, p1, p2]).all() and back < -2.9e38
    # the largest -|u|^2 / sscale a row can carry (128 coordinates below 2^14) does not move it, nor does sscale below 1 make it a NaN
    assert np.isfinite(np.float32(back) + np.float32(-128 * 2.0 ** 28))
    for sscale in (2.0 ** -40, 1.0, 2.0 ** 40):
        d2 = -np.float32(sscale) * np.float32(back)          # what the epilogue turns the accumulator into
        assert d2 > 1e20 and not np.isnan(d2)                 # weight 2^-d2 (Gaussian) or 2^-sqrt(.) (exponential): an exact zero


def test_f2fp_fhadd_split_of_a_weight_keeps_22_bits():
    """hi = fp16_rn(w); -lo = fp16_rn(hi - w), the difference exact in FP32 (FHADD); the MMA negates the lo plane."""
    rng = np.random.RandomState(5)
    w = np.float32(2.0 ** rng.uniform(-3.0, 8.0, 200000))    # weights 2^(log2 k - ref) <= 2^8 whose lo part is a normal FP16
    hi = w.astype(np.float16)
    nl = (hi.astype(np.float32) - w).astype(np.float32)       # exact: |hi - w| <= 2^-11 w, both on w's FP32 grid
    assert (nl.astype(np.float64) == hi.astype(np.float64) - w.astype(np.float64)).all()
    neg_lo = nl.astype(np.float16)
    back = hi.astype(np.float64) - neg_lo.astype(np.float64)
    assert (np.abs(back - w.astype(np.float64)) / w).max() <= 2.0 ** -22
    # smaller weights: the lo part (then hi as well) falls into FP16's subnormals and the planes lose bits, but the absolute
    # error stays at half a subnormal step, 2^-25 -- of a row whose largest weight is at least 1 (the lazy reference)
    small = np.float32(2.0 ** rng.uniform(-40.0, -3.0, 100000))
    h2 = small.astype(np.float16)
    d2 = (h2.astype(np.float32) - small).astype(np.float32)
    assert (d2.astype(np.float64) == h2.astype(np.float64) - small.astype(np.float64)).all()
    l2 = d2.astype(np.float16)
    assert np.abs(h2.astype(np.float64) - l2.astype(np.float64) - small).max() <= 2.0 ** -25
