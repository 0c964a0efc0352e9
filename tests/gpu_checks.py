"""Parity checks of the CUDA path against the CPU oracle, shared by `pytest -m gpu` (tests/test_gpu_*.py)
and tools/gpu_probe.py.  Every check calls the product through the C ABI (rten_b200.ops -> ctypes ->
librten_b200.so) and the oracle through oracle/oracle.py.

Tolerances
  integer / index work, elementwise f32 math, Softmax, LayerNormalization: bit-exact.
  f32 GEMM / Conv (tcgen05 kind::tf32, single pass): |got - exact| <= 2^-9 * sum_k |a_k b_k| + 1e-6
  (both operands lose at most 2^-10 relative each to TF32 rounding; fp32 accumulation in TMEM).
"""
import numpy as np

TF32_REL = 2.0 ** -9


def new_ctx(rt, tf32=True):
    """The library defaults to the fp32-grade 3xTF32 mode; the kernel-variant checks below opt in to the single TF32 pass
    explicitly (their bound is the TF32 one) unless they test the 3x mode."""
    ctx = rt.Context(0)
    ctx.set_f32_mode(not tf32)
    return ctx


def assert_same_greedy_token(got, ref, tol, what):
    """Greedy decoding picks arg-max: with a stated logit tolerance two near-tied candidates may swap, so the reference's
    token must be within that tolerance of our maximum (and vice versa), not necessarily the same index."""
    scale = float(np.abs(ref).max())
    rows = np.arange(got.shape[0])
    gap_ours = got.max(1) - got[rows, ref.argmax(1)]
    gap_ref = ref.max(1) - ref[rows, got.argmax(1)]
    assert (gap_ours <= tol * scale).all() and (gap_ref <= tol * scale).all(), \
        f"{what}: greedy token differs beyond the logit tolerance (gaps {float(gap_ours.max()):.3e} / {float(gap_ref.max()):.3e}, scale {scale:.3e})"


def assert_reference_rule(got, want, what):
    """The reference's own float comparison (rten-tensor/src/test_util.rs:47-92): |a - b| <= 1e-8 + 1e-5 * |b|."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    bad = np.abs(got - want) > 1e-8 + 1e-5 * np.abs(want)
    assert not bad.any(), (f"{what}: {int(bad.sum())} of {bad.size} elements outside 1e-8 + 1e-5*|ref| "
                           f"(worst rel {float((np.abs(got - want) / np.maximum(np.abs(want), 1e-30)).max()):.2e})")


def _ulp_diff(a, b):
    a = np.ascontiguousarray(a, np.float32).view(np.int32).astype(np.int64)
    b = np.ascontiguousarray(b, np.float32).view(np.int32).astype(np.int64)
    return int(np.abs(a - b).max()) if a.size else 0


def assert_bit_exact(got, exp, what):
    got = np.asarray(got)
    exp = np.asarray(exp)
    assert got.shape == exp.shape, f"{what}: shape {got.shape} != {exp.shape}"
    if np.issubdtype(exp.dtype, np.floating):
        same = (got.view(np.int32) == exp.view(np.int32)) | (np.isnan(got) & np.isnan(exp))
        assert same.all(), f"{what}: {int((~same).sum())} of {same.size} elements differ, max ulp {_ulp_diff(got, exp)}"
    else:
        assert np.array_equal(got, exp), f"{what}: {int((got != exp).sum())} of {exp.size} elements differ"


def assert_tf32_close(got, exact, absum, what, extra_abs=0.0):
    got = np.asarray(got, np.float64)
    err = np.abs(got - exact)
    bound = TF32_REL * absum + 1e-6 + extra_abs
    worst = float((err / bound).max()) if err.size else 0.0
    assert worst <= 1.0, f"{what}: error {float(err.max()):.3e} exceeds the TF32 bound (worst ratio {worst:.2f})"
    return worst


# ------------------------------------------------------------------------------------------
def check_context(rt, oracle):
    ctx = new_ctx(rt)
    x = oracle.XorShiftRng(1234).f32((3, 5, 7))
    t = ctx.to_device(x)
    assert_bit_exact(t.numpy(), x, "copy roundtrip")
    p = t.permute(2, 0, 1)
    assert_bit_exact(p.numpy(), x.transpose(2, 0, 1), "strided D2H copy")
    assert ctx.launches > 0
    return "ok"


def check_unary(rt, oracle):
    ctx = new_ctx(rt)
    x = np.concatenate([np.arange(-6, 6, 0.001, dtype=np.float32), oracle.XorShiftRng(7).uniform((100003,), -10, 10),
                        np.array([0.0, -0.0, np.inf, -np.inf, 1e-30, -88.0, 104.0], np.float32)])
    assert_bit_exact(rt.Erf().run(ctx, x).numpy(), oracle.erf(x), "Erf")
    assert_bit_exact(rt.Gelu().run(ctx, x).numpy(), oracle.gelu(x), "Gelu")
    assert_bit_exact(rt.Gelu(approximate=True).run(ctx, x).numpy(), oracle.gelu(x, True), "ApproxGelu")
    assert_bit_exact(rt.Relu().run(ctx, x).numpy(), oracle.relu(x), "Relu")
    d = ctx.to_device(x[:4099])
    y = rt.Gelu().run(ctx, d, in_place=True)
    assert y is d
    assert_bit_exact(d.numpy(), oracle.gelu(x[:4099]), "Gelu in place")
    x2 = oracle.XorShiftRng(9).uniform((4, 6, 10))
    assert_bit_exact(rt.Erf().run(ctx, x2.transpose(2, 0, 1)).numpy(), oracle.erf(x2.transpose(2, 0, 1)), "Erf strided")
    sp = rt.Erf().run(ctx, np.array([np.nan, 0.0, np.inf, -np.inf], np.float32)).numpy()
    assert np.isnan(sp[0]) and sp[1] == 0 and sp[2] == 1 and sp[3] == -1
    return "ok"


def check_softmax(rt, oracle):
    ctx = new_ctx(rt)
    r = oracle.XorShiftRng(1234)
    for shape, axis in [((6,), 0), ((2, 3), 1), ((2, 3), 0), ((4, 4), 1), ((5, 17), -1), ((3, 4, 130), -1),
                        ((2, 12, 128, 128), -1), ((7, 1000), 1), ((3, 5, 9), 1), ((0, 4), 1), ((2, 2050), -1)]:
        x = r.uniform(shape, -4, 4)
        got = rt.Softmax(axis=axis).run(ctx, x).numpy()
        assert_bit_exact(got, oracle.softmax(x, axis), f"Softmax{shape} axis={axis}")
    x = np.array([0.1634, 0.8647, 0.6401, 0.8265, 0.0560, 0.2304], np.float32)
    assert np.allclose(rt.Softmax(0).run(ctx, x).numpy(), [0.1172, 0.2362, 0.1887, 0.2274, 0.1052, 0.1253], atol=1e-4)
    xt = r.uniform((4, 4)).T
    assert_bit_exact(rt.Softmax(1).run(ctx, xt).numpy(), oracle.softmax(xt, 1), "Softmax transposed")
    ninf = np.full(3, -np.inf, np.float32)
    assert np.isnan(rt.Softmax(0).run(ctx, ninf).numpy()).all()
    assert rt.Softmax(0, flush_nans_to_zero=True).run(ctx, ninf).numpy().tolist() == [0, 0, 0]
    # AddSoftmax: BERT-shaped mask broadcast + commutativity + in place
    qk = r.uniform((2, 3, 16, 128), -3, 3)
    for mshape in [(2, 1, 1, 128), (1, 1, 16, 128), (128,), (2, 3, 16, 128), (2, 3, 1, 1)]:
        m = r.uniform(mshape, -2, 0)
        exp = oracle.add_softmax(qk, m)
        assert_bit_exact(rt.AddSoftmax().run(ctx, qk, m).numpy(), exp, f"AddSoftmax mask{mshape}")
        assert_bit_exact(rt.AddSoftmax().run(ctx, m, qk).numpy(), exp, f"AddSoftmax swapped mask{mshape}")
    d = ctx.to_device(qk)
    m = r.uniform((2, 1, 1, 128), -2, 0)
    y = rt.AddSoftmax().run(ctx, d, ctx.to_device(m), in_place=True)
    assert y is d
    assert_bit_exact(d.numpy(), oracle.add_softmax(qk, m), "AddSoftmax in place")
    try:
        rt.AddSoftmax().run(ctx, qk, np.zeros((3, 5), np.float32))
        raise AssertionError("expected broadcast error")
    except rt.OpError as e:
        assert e.kind == "IncompatibleInputShapes" and e.msg == "Cannot broadcast inputs", str(e)
    return "ok"


def check_layer_norm(rt, oracle):
    ctx = new_ctx(rt)
    r = oracle.XorShiftRng(1234)
    for shape, axis in [((1, 5, 2), -1), ((1, 5, 2), -2), ((7, 768), -1), ((3, 4, 100), -1), ((2, 3, 64), -1),
                        ((5, 1000), -1), ((4, 15), -1), ((2, 16, 17), 1)]:
        x = r.uniform(shape, -2, 3)
        nshape = shape[axis:] if axis < 0 else shape[axis:]
        g = r.uniform(nshape, 0.5, 1.5)
        b = r.uniform(nshape, -0.5, 0.5)
        for eps in (None, 1e-12):
            assert_bit_exact(rt.LayerNormalization(axis, eps).run(ctx, x, g, b).numpy(), oracle.layer_norm(x, g, b, axis, eps),
                             f"LayerNorm{shape} axis={axis} eps={eps}")
        assert_bit_exact(rt.LayerNormalization(axis).run(ctx, x, g).numpy(), oracle.layer_norm(x, g, None, axis),
                         f"LayerNorm{shape} no bias")
    x = np.array([[0., 1., 2., 3.]], np.float32)
    assert_bit_exact(rt.LayerNormalization().run(ctx, x, np.float32(2.0), np.float32(0.5)).numpy(),
                     oracle.layer_norm(x, np.float32(2.0), np.float32(0.5)), "LayerNorm scalar scale+bias")
    assert_bit_exact(rt.LayerNormalization().run(ctx, x, np.float32(2.0)).numpy(), oracle.layer_norm(x, np.float32(2.0)),
                     "LayerNorm scalar scale")
    for bad, msg in [((np.ones((2, 3), np.float32), np.ones((2, 3), np.float32), None),
                      "`scale` is not broadcastable to normalized axes of input"),
                     ((np.ones((2, 3), np.float32), np.ones(3, np.float32), np.ones((2, 3), np.float32)),
                      "`bias` is not broadcastable to normalized axes of input")]:
        try:
            rt.LayerNormalization(-1).run(ctx, *bad)
            raise AssertionError("expected error")
        except rt.OpError as e:
            assert e.kind == "InvalidValue" and e.msg == msg, str(e)
    return "ok"


def check_dql(rt, oracle):
    ctx = new_ctx(rt)
    r = oracle.XorShiftRng(1234)
    for shape, lo, hi in [((5, 1000), -1.2, 2.8), ((4096, 768), -3, 3), ((3, 7, 11), 0.5, 2.0), ((17,), -5, -1), ((0, 3), 0, 1),
                          ((128, 128), -7, 0.25), ((16385,), -0.5, 9.0)]:  # single-kernel path up to 16384 elements, three kernels above
        x = r.uniform(shape, lo, hi)
        y, s, z = rt.DynamicQuantizeLinear().run(ctx, x)
        ey, es, ez = oracle.dynamic_quantize_linear(x)
        assert_bit_exact(s.numpy(), np.float32(es), f"DQL scale {shape}")
        assert_bit_exact(z.numpy(), np.uint8(ez), f"DQL zero point {shape}")
        assert_bit_exact(y.numpy(), ey, f"DQL y {shape}")
    # channels-last input quantised straight into the interior of a spatially pre-padded buffer (border = 128), with the
    # range taken from a caller-provided (min, max) pair
    x = r.uniform((2, 32, 6, 5), -2, 3)
    ey, es, ez = oracle.dynamic_quantize_linear(x)
    buf = ctx.to_device(np.full((2, 8, 7, 32), 128, np.uint8))
    interior = buf.view((2, 32, 6, 5), (8 * 7 * 32, 1, 7 * 32, 32), (1 * 7 + 1) * 32)
    y, s, z = rt.DynamicQuantizeLinear().run(ctx, ctx.to_device(x, channels_last=True), out=interior)
    want = np.full((2, 8, 7, 32), 128, np.uint8)
    want[:, 1:7, 1:6, :] = ey.transpose(0, 2, 3, 1)
    assert_bit_exact(buf.numpy(), want, "DQL into a pre-padded buffer")
    assert_bit_exact(s.numpy(), np.float32(es), "DQL scale (padded destination)")
    return "ok"


def check_glue(rt, oracle):
    ctx = new_ctx(rt)
    rr = oracle.XorShiftRng(55)
    table, upd = rr.uniform((40, 12)), rr.uniform((5, 12))
    idx = np.array([3, 39, 0, 17, -2], np.int32)
    td = ctx.to_device(table)
    rt.ScatterRows().run(ctx, td, idx, upd)
    want = table.copy()
    want[idx] = upd
    assert_bit_exact(td.numpy(), want, "ScatterRows")
    r = oracle.XorShiftRng(1234)
    a, b = r.uniform((2, 3, 4, 5)), r.uniform((2, 3, 4, 5))
    assert_bit_exact(rt.Add().run(ctx, a, b).numpy(), a + b, "Add")
    c = r.uniform((3, 1, 1))
    assert_bit_exact(rt.Add().run(ctx, a, c).numpy(), a + c, "Add broadcast")
    x = r.uniform((2, 6, 13, 11))
    for cl in (False, True):
        d = ctx.to_device(x, channels_last=cl)
        assert_bit_exact(rt.MaxPool((3, 3), (1, 1, 1, 1), (2, 2)).run(ctx, d).numpy(), oracle.max_pool(x, (3, 3), [1, 1, 1, 1], (2, 2)),
                         f"MaxPool cl={cl}")
        assert_bit_exact(rt.GlobalAveragePool().run(ctx, d).numpy(), oracle.global_average_pool(x), f"GlobalAveragePool cl={cl}")
    x = r.uniform((3, 70, 7, 7))
    assert_bit_exact(rt.GlobalAveragePool().run(ctx, ctx.to_device(x, True)).numpy(), oracle.global_average_pool(x), "GAP 7x7")
    table = r.uniform((50, 12))
    idx = np.array([[0, 49, 7], [3, 3, -1]], np.int32)
    assert_bit_exact(rt.GatherRows().run(ctx, table, idx).numpy(), table[idx], "GatherRows")
    return "ok"


# ------------------------------------------------------------------------------------------
def _matmul_case(rt, oracle, ctx, ashape, bshape, bias=False, alpha=None, b_kmajor=False, prepack=False, seed=1234):
    r = oracle.XorShiftRng(seed)
    a = r.uniform(ashape)
    if b_kmajor:  # B given as a transposed view of [.., N, K] storage (what TransposeFusion hands to MatMul)
        bt = r.uniform(tuple(bshape[:-2]) + (bshape[-1], bshape[-2]))
        b = np.swapaxes(bt, -1, -2)
    else:
        b = r.uniform(bshape)
    bv = r.uniform((bshape[-1],)) if bias else None
    op = rt.FusedMatMul(alpha) if (bias or alpha is not None) else rt.MatMul()
    kw = {}
    if prepack:
        kw["packed_b"] = op.prepack(ctx, 1, b)
    got = (op.run(ctx, a, b, bv, **kw) if isinstance(op, rt.FusedMatMul) else op.run(ctx, a, b, **kw)).numpy()
    exp = oracle.matmul(a, b, bv, alpha)
    assert got.shape == exp.shape, f"matmul{ashape}x{bshape}: shape {got.shape} != {exp.shape}"
    a2 = a.reshape(-1, a.shape[-1]) if a.ndim > 1 else a[None, :]
    exact = np.matmul(a.astype(np.float64), b.astype(np.float64)) * (1.0 if alpha is None else alpha)
    absum = np.matmul(np.abs(a).astype(np.float64), np.abs(b).astype(np.float64)) * abs(1.0 if alpha is None else alpha)
    if bias:
        exact = exact + bv
    worst = assert_tf32_close(got, exact, absum, f"matmul{ashape}x{bshape}")
    # and the oracle (fp32 reference arithmetic) must sit inside the same band
    assert_tf32_close(exp, exact, absum, "oracle self-check")
    return worst


def check_matmul_small(rt, oracle):
    ctx = new_ctx(rt)
    a = np.array([[1, 2], [3, 4]], np.float32)
    b = np.array([[5, 6], [7, 8]], np.float32)
    assert_bit_exact(rt.MatMul().run(ctx, a, b).numpy(), np.array([[19, 22], [43, 50]], np.float32), "2x2 f32 (exact in tf32)")
    w = _matmul_case(rt, oracle, ctx, (128, 32), (32, 128))
    w = max(w, _matmul_case(rt, oracle, ctx, (128, 64), (64, 128), b_kmajor=True))
    return f"worst err/bound {w:.3f}"


def check_matmul_shapes(rt, oracle):
    ctx = new_ctx(rt)
    worst = 0.0
    cases = [((3, 10), (10, 8)), ((2, 3, 10), (10, 8)), ((3, 10), (2, 10, 8)), ((2, 3, 10), (2, 10, 8)),
             ((2, 1, 3, 10), (1, 4, 10, 8)), ((10,), (10, 8)), ((3, 10), (10,)), ((10,), (10,)),
             ((130, 300), (300, 257)), ((1, 768), (768, 1000)), ((255, 33), (33, 129)), ((64, 1), (1, 64)),
             ((2, 5, 12), (12, 7))]
    for ash, bsh in cases:
        worst = max(worst, _matmul_case(rt, oracle, ctx, ash, bsh))
    worst = max(worst, _matmul_case(rt, oracle, ctx, (2, 5, 12), (12, 7), bias=True, alpha=0.125))
    worst = max(worst, _matmul_case(rt, oracle, ctx, (200, 96), (96, 80), bias=True, prepack=True))
    worst = max(worst, _matmul_case(rt, oracle, ctx, (4, 3, 128, 64), (4, 3, 64, 128), alpha=0.125, b_kmajor=True))
    # many row tiles with a narrow N (pair mode), odd tile counts, N / K tails
    worst = max(worst, _matmul_case(rt, oracle, ctx, (128 * 301 + 5, 72), (72, 64), bias=True, prepack=True))
    worst = max(worst, _matmul_case(rt, oracle, ctx, (40000, 40), (40, 100), b_kmajor=True))
    worst = max(worst, _matmul_case(rt, oracle, ctx, (3, 128 * 151, 33), (33, 36)))
    # zero sized dims (src/ops/matmul.rs:1344-1361)
    for ash, bsh in [((2, 0, 10), (10, 8)), ((3, 10), (10, 0)), ((3, 0), (0, 4))]:
        got = rt.MatMul().run(ctx, np.zeros(ash, np.float32), np.zeros(bsh, np.float32)).numpy()
        exp = np.matmul(np.zeros(ash, np.float32), np.zeros(bsh, np.float32))
        assert got.shape == exp.shape and not got.any(), f"matmul zero-size {ash}x{bsh}"
    for ash, bsh, kind, msg in [((1, 2), (3, 1), "IncompatibleInputShapes", "Columns of first matrix does not match rows of second matrix"),
                                ((), (3, 1), "InvalidValue", "Inputs must have >= 1 dimensions"),
                                ((2, 2, 2), (3, 2, 2), "IncompatibleInputShapes", "Cannot broadcast shapes")]:
        try:
            rt.MatMul().run(ctx, np.zeros(ash, np.float32), np.zeros(bsh, np.float32))
            raise AssertionError("expected error")
        except rt.OpError as e:
            assert e.kind == kind and e.msg == msg, str(e)
    return f"worst err/bound {worst:.3f}"


def check_matmul_bert(rt, oracle):
    ctx = new_ctx(rt)
    w = _matmul_case(rt, oracle, ctx, (4, 128, 768), (768, 768), bias=True, prepack=True)
    w = max(w, _matmul_case(rt, oracle, ctx, (512, 768), (768, 3072), bias=True))
    w = max(w, _matmul_case(rt, oracle, ctx, (256, 3072), (3072, 768), prepack=True))
    return f"worst err/bound {w:.3f}"


def check_gemm_op(rt, oracle):
    ctx = new_ctx(rt)
    r = oracle.XorShiftRng(1234)
    worst = 0.0
    for (m, n, k), ta, tb, alpha, beta, cshape in [((3, 8, 10), False, False, 1.0, 1.0, (8,)), ((32, 1000, 2048), False, True, 1.0, 1.0, (1000,)),
                                                   ((5, 7, 9), True, True, 0.5, 2.0, (5, 7)), ((5, 7, 9), False, False, 2.0, 0.0, None),
                                                   ((6, 4, 3), False, False, 1.0, 0.5, (6, 1))]:
        a = r.uniform((k, m) if ta else (m, k))
        b = r.uniform((n, k) if tb else (k, n))
        c = r.uniform(cshape) if cshape else None
        got = rt.Gemm(alpha, beta, ta, tb).run(ctx, a, b, c).numpy()
        a2, b2 = (a.T if ta else a), (b.T if tb else b)
        exact = alpha * (a2.astype(np.float64) @ b2.astype(np.float64)) + (beta * c if c is not None else 0.0)
        absum = abs(alpha) * (np.abs(a2).astype(np.float64) @ np.abs(b2).astype(np.float64))
        worst = max(worst, assert_tf32_close(got, exact, absum, f"Gemm {m}x{n}x{k} ta={ta} tb={tb}"))
    for args, kind, msg in [((np.zeros((3, 10), np.float32), np.zeros((8, 10), np.float32)), "IncompatibleInputShapes",
                             "Columns of first matrix does not match rows of second matrix"),
                            ((np.zeros((3, 10), np.float32), np.zeros((10, 8), np.float32), np.zeros((5,), np.float32)),
                             "IncompatibleInputShapes", "Cannot broadcast c to output shape")]:
        try:
            rt.Gemm().run(ctx, *args)
            raise AssertionError("expected error")
        except rt.OpError as e:
            assert e.kind == kind and e.msg == msg, str(e)
    return f"worst err/bound {worst:.3f}"


# ------------------------------------------------------------------------------------------
def check_matmul_integer(rt, oracle):
    ctx = new_ctx(rt)
    A = np.array([[1, 2], [3, 4]], np.uint8)
    B = np.array([[5, 6], [7, 8]], np.int8)
    lit = [(A, B, None, None), (A, B, np.uint8(127), np.int8(-50)), (A, B, np.array([1, 2], np.uint8), np.array([3, 4], np.int8)),
           (np.zeros((3, 2, 2), np.uint8), B, np.array([1, 2], np.uint8), np.array([3, 4], np.int8)),
           (np.array([[1, 2, 3, 4]], np.uint8), np.array([[5, 6], [7, 8], [9, 10], [11, 12]], np.int8), np.array([1], np.uint8), np.array([3, 4], np.int8)),
           (np.array([1, 2], np.uint8), np.array([[1, 2], [3, 4]], np.int8), np.array([1], np.uint8), np.array([2, 3], np.int8)),
           (A, np.array([1, 2], np.int8), np.array([1, 2], np.uint8), np.array([3], np.int8)),
           (np.zeros((0, 2), np.uint8), np.zeros((2, 3), np.int8), None, None)]
    for a, b, az, bz in lit:
        assert_bit_exact(rt.MatMulInteger().run(ctx, a, b, az, bz).numpy(), oracle.matmul_integer(a, b, az, bz), f"MatMulInteger literal {a.shape}x{b.shape}")
    r = oracle.XorShiftRng(1234)
    for adt in (np.uint8, np.int8):
        for bdt in (np.uint8, np.int8):
            for (ash, bsh) in [((2, 5, 20), (20, 9)), ((130, 300), (300, 257)), ((1, 768), (768, 64)), ((8, 768), (768, 2304)), ((64, 1000), (1000, 17))]:
                a = r.u8(ash).view(adt)
                b = r.u8(bsh).view(bdt)
                az = r.u8((ash[-2],)).view(adt)
                bz = r.u8((bsh[-1],)).view(bdt)
                for azp, bzp in [(None, None), (az, None), (None, bz), (az, bz), (az[:1].reshape(()), bz[:1].reshape(()))]:
                    got = rt.MatMulInteger().run(ctx, a, b, azp, bzp).numpy()
                    assert_bit_exact(got, oracle.matmul_integer(a, b, azp, bzp), f"MatMulInteger {adt.__name__}x{bdt.__name__} {ash}x{bsh} zp={azp is not None},{bzp is not None}")
    # prepacked B + fused cast*scale (MatMulIntegerToFloat), per-column and scalar scales
    a = r.u8((4, 128, 768))
    b = r.i8((768, 256))
    pk = rt.MatMulInteger().prepack(ctx, 1, b)
    az, bz = np.uint8(131), r.i8((256,))
    assert_bit_exact(rt.MatMulInteger().run(ctx, a, b, az, bz, packed_b=pk).numpy(), oracle.matmul_integer(a, b, az, bz), "MatMulInteger prepacked")
    for sc in (r.uniform((256,), 0.001, 0.1), np.float32(0.02), np.array([0.5], np.float32)):
        got = rt.MatMulIntegerToFloat().run(ctx, a, b, az, bz, sc, packed_b=pk).numpy()
        assert_bit_exact(got, oracle.matmul_integer_to_float(a, b, az, bz, sc), f"MatMulIntegerToFloat scale{np.shape(sc)}")
    for args, kind, msg in [((A, B, np.array([1, 2, 4], np.uint8), np.array([3, 4], np.int8)), "InvalidValue", "Zero point has incorrect size"),
                            ((A, B, np.full((2, 2), 2, np.uint8), None), "UnsupportedValue", "Only scalar or vector zero points are supported"),
                            ((np.zeros((1, 2), np.uint8), np.zeros((3, 1), np.int8)), "IncompatibleInputShapes", "Columns of first matrix does not match rows of second matrix"),
                            ((np.zeros((2, 2, 2), np.uint8), np.zeros((3, 2, 2), np.int8)), "IncompatibleInputShapes", "Cannot broadcast shapes")]:
        try:
            rt.MatMulInteger().run(ctx, *args)
            raise AssertionError("expected error")
        except rt.OpError as e:
            assert e.kind == kind and e.msg == msg, str(e)
    try:
        rt.MatMulIntegerToFloat().run(ctx, A, B, None, None, np.array([2., 3., 4.], np.float32))
        raise AssertionError("expected error")
    except rt.OpError as e:
        assert e.msg == "Scale length does not match tensor columns", str(e)
    return "ok"


# ------------------------------------------------------------------------------------------
def check_plans(rt, oracle):
    """Every launch-plan family (pair, two K atoms, split-K with the last-arriver reduction, the single 512-column
    accumulator stage of 256 x 256 tiles) must give the same answers: forced through the debug environment knobs,
    then chosen by the autotuner."""
    import os
    ctx = new_ctx(rt)
    r = oracle.XorShiftRng(99)
    keys = ("RTEN_B200_FORCE_BN", "RTEN_B200_FORCE_PAIR", "RTEN_B200_FORCE_KATOMS", "RTEN_B200_FORCE_SPLITK", "RTEN_B200_FORCE_CTA2")
    plans = [dict(), dict(BN=64, PAIR=1, CTA2=0), dict(BN=128, PAIR=0, KATOMS=2, CTA2=0), dict(BN=256, PAIR=1, CTA2=0),
             dict(BN=128, PAIR=1, SPLITK=2, CTA2=0), dict(BN=64, PAIR=0, SPLITK=3, CTA2=0), dict(BN=256, PAIR=1, SPLITK=2, CTA2=0),
             dict(BN=96, PAIR=0, SPLITK=4, KATOMS=1, CTA2=0),
             # CTA pairs (tcgen05.mma.cta_group::2, 256-row tiles, half of B per CTA)
             dict(BN=128, PAIR=0, CTA2=1), dict(BN=256, PAIR=0, CTA2=1), dict(BN=256, PAIR=1, CTA2=1), dict(BN=64, PAIR=1, CTA2=1, KATOMS=2),
             dict(BN=128, PAIR=0, CTA2=1, SPLITK=2), dict(BN=256, PAIR=1, CTA2=1, SPLITK=2), dict(BN=96, PAIR=0, CTA2=1)]
    a8 = r.u8((300, 2048))
    b8 = r.i8((2048, 512))
    az, bz = r.u8((300,)), r.i8((512,))
    exp8 = oracle.matmul_integer(a8, b8, az, bz)
    sc = r.uniform((512,), 0.001, 0.1)
    exp8f = oracle.matmul_integer_to_float(a8, b8, az, bz, sc)
    worst = 0.0
    hits_before = 0
    never = []
    try:
        for pl in plans:
            for k in keys:
                os.environ.pop(k, None)
            for k, v in pl.items():
                os.environ["RTEN_B200_FORCE_" + k] = str(v)
            tag = f"plan {pl}"
            worst = max(worst, _matmul_case(rt, oracle, ctx, (384, 1024), (1024, 512), bias=True, prepack=True, seed=5))
            worst = max(worst, _matmul_case(rt, oracle, ctx, (3, 130, 520), (520, 300), seed=6))
            assert_bit_exact(rt.MatMulInteger().run(ctx, a8, b8, az, bz).numpy(), exp8, f"MatMulInteger {tag}")
            assert_bit_exact(rt.MatMulIntegerToFloat().run(ctx, a8, b8, az, bz, sc).numpy(), exp8f, f"MatMulIntegerToFloat {tag}")
            worst = max(worst, _conv_case(rt, oracle, ctx, (4, 256, 14, 14), (256, 256, 3, 3), pads=(1, 1, 1, 1), cl=True, prepack=True, act=1))
            worst = max(worst, _conv_case(rt, oracle, ctx, (8, 512, 7, 7), (512, 512, 3, 3), pads=(1, 1, 1, 1), cl=True, residual=True, act=1))
            worst = max(worst, _conv_case(rt, oracle, ctx, (2, 64, 20, 20), (96, 64, 1, 1), cl=False))
            worst = max(worst, _conv_case(rt, oracle, ctx, (4, 512, 14, 14), (256, 512, 1, 1), cl=True, residual=True, act=1))  # 16 K blocks: split-K / CTA-pair plans exist
            hit, miss = ctx.forced_plan_counts()
            # every split-K / CTA-pair family must actually have run somewhere in the sweep (a forced combination that no
            # launch can satisfy would make this check vacuous); the remaining combinations are reported
            if pl and hit == hits_before:
                assert "SPLITK" not in pl and not (pl.get("CTA2") == 1 and "KATOMS" not in pl), \
                    f"{tag}: no launch of this sweep ran the forced plan ({miss} fell back to the model's choice)"
                never.append(str(pl))
            hits_before = hit
    finally:
        for k in keys:
            os.environ.pop(k, None)
    # autotuned plans: first call measures, second call replays the cached plan
    ctx2 = new_ctx(rt)
    ctx2.set_autotune(True)
    for _ in range(2):
        worst = max(worst, _matmul_case(rt, oracle, ctx2, (384, 1024), (1024, 512), bias=True, prepack=True, seed=5))
        assert_bit_exact(rt.MatMulInteger().run(ctx2, a8, b8, az, bz).numpy(), exp8, "MatMulInteger autotuned")
        worst = max(worst, _conv_case(rt, oracle, ctx2, (8, 512, 7, 7), (512, 512, 3, 3), pads=(1, 1, 1, 1), cl=True, prepack=True, act=1))
        worst = max(worst, _conv_case(rt, oracle, ctx2, (8, 512, 7, 7), (512, 512, 3, 3), pads=(1, 1, 1, 1), cl=True, residual=True, act=1))
    return f"worst err/bound {worst:.3f}; forced combinations no launch could take: {never if never else 'none'}"


# ------------------------------------------------------------------------------------------
def check_graph_replay(rt, oracle):
    """A captured graph of consecutive tensor-core launches must reproduce the eager results bit for bit (same plans,
    same arithmetic) when replayed: for an 8-layer and a 45-layer conv chain with residual links, more than once, and
    for independent integer launches in one capture."""
    ctx = new_ctx(rt)
    r = oracle.XorShiftRng(321)

    def conv_layer(ci, co, k, res=None, act=1):
        w = r.uniform((co, ci, k, k), -1, 1) / np.float32(np.sqrt(ci * k * k))
        b = r.uniform((co,))
        op = rt.Conv(1, (1, 1), (k // 2,) * 4, (1, 1), activation=act)
        return dict(op=op, w=ctx.to_device(w), b=ctx.to_device(b), pk=op.prepack(ctx, 1, w), res=res)

    # a: bottleneck-like chain with residual links (index of the producing layer, -1 = the input)
    chain_a = [conv_layer(64, 128, 1), conv_layer(128, 128, 3), conv_layer(128, 128, 1, res=0), conv_layer(128, 64, 3),
               conv_layer(64, 256, 1), conv_layer(256, 64, 1), conv_layer(64, 64, 3, res=5), conv_layer(64, 512, 1, act=0)]
    # b: a 45-layer chain
    chain_b = [conv_layer(64, 64, 1, res=(i - 2 if i >= 2 and i % 3 == 0 else None)) for i in range(45)]
    x = ctx.to_device(r.uniform((4, 64, 28, 28)), channels_last=True)

    def run_chain(chain, outs):
        h, produced = x, []
        for i, l in enumerate(chain):
            res = None if l["res"] is None else (x if l["res"] < 0 else produced[l["res"]])
            y = l["op"].run(ctx, h, l["w"], l["b"], packed_w=l["pk"], residual=res, out=(outs[i] if outs else None))
            produced.append(y)
            h = y
        return produced

    worst_layers = 0
    for name, chain in (("a", chain_a), ("b", chain_b)):
        eager = run_chain(chain, None)
        want = [t.numpy() for t in eager]
        for t in eager:  # poison the buffers: the replay has to recompute everything
            t.copy_from(np.full(t.shape, np.nan, np.float32))
        l0 = ctx.launches
        ctx.graph_begin()
        run_chain(chain, eager)
        g = ctx.graph_end()
        for rep in range(3):
            if rep:
                eager[-1].copy_from(np.full(eager[-1].shape, np.nan, np.float32))
            g.launch()
            ctx.sync()
            for i, (t, w) in enumerate(zip(eager, want)):
                assert_bit_exact(t.numpy(), w, f"graph replay chain {name} layer {i} replay {rep}")
        worst_layers = max(worst_layers, len(chain))
    # integer launches in one capture (independent problems)
    a8 = [r.u8((200, 512)) for _ in range(3)]
    b8 = [r.i8((512, 160)) for _ in range(3)]
    az, bz = r.u8((200,)), r.i8((160,))
    outs = [rt.MatMulInteger().run(ctx, a, b, az, bz) for a, b in zip(a8, b8)]
    want = [oracle.matmul_integer(a, b, az, bz) for a, b in zip(a8, b8)]
    da, db, dz, dbz = [ctx.to_device(a) for a in a8], [ctx.to_device(b) for b in b8], ctx.to_device(az), ctx.to_device(bz)
    for o in outs:
        o.copy_from(np.zeros(o.shape, np.int32))
    ctx.graph_begin()
    for a, b, o in zip(da, db, outs):
        rt.MatMulInteger().run(ctx, a, b, dz, dbz, out=o)
    g = ctx.graph_end()
    g.launch()
    ctx.sync()
    for o, w in zip(outs, want):
        assert_bit_exact(o.numpy(), w, "graph replay MatMulInteger")
    return f"chains of up to {worst_layers} layers replayed bit-exactly"


# ------------------------------------------------------------------------------------------
def _conv_exact(x, w, bias, pads, groups, strides, dil):
    import torch
    import torch.nn.functional as F
    xt = F.pad(torch.from_numpy(x).double(), (pads[1], pads[3], pads[0], pads[2]))
    wt = torch.from_numpy(w).double()
    y = F.conv2d(xt, wt, None if bias is None else torch.from_numpy(bias).double(), stride=strides, dilation=dil, groups=groups)
    ya = F.conv2d(xt.abs(), wt.abs(), None, stride=strides, dilation=dil, groups=groups)
    return y.numpy(), ya.numpy()


def _conv_case(rt, oracle, ctx, xs, ws, pads=(0, 0, 0, 0), groups=1, strides=(1, 1), dil=(1, 1), bias=True, cl=False, prepack=False,
               residual=False, act=0, seed=1234):
    r = oracle.XorShiftRng(seed)
    x = r.uniform(xs)
    w = r.uniform(ws, -1, 1) / np.float32(np.sqrt(ws[1] * ws[2] * ws[3]))
    b = r.uniform((ws[0],)) if bias else None
    op = rt.Conv(groups, dil, pads, strides, activation=act)
    xd = ctx.to_device(x, channels_last=cl)
    kw = {}
    if prepack:
        kw["packed_w"] = op.prepack(ctx, 1, w)
    exact, absum = _conv_exact(x, w, b, pads, groups, strides, dil)
    if residual:
        res = r.uniform(exact.shape)
        kw["residual"] = ctx.to_device(res, channels_last=cl)
        exact = exact + res
    y = op.run(ctx, xd, w, b, **kw)
    got = y.numpy()
    if act == 1:
        exact = np.maximum(exact, 0)
    what = f"Conv x{xs} w{ws} pads={pads} g={groups} s={strides} d={dil} cl={cl}"
    assert got.shape == exact.shape, f"{what}: shape {got.shape} != {exact.shape}"
    if cl:
        assert y.strides[1] == 1, f"{what}: channels-last input must give channels-last output, got {y.strides}"
    return assert_tf32_close(got, exact, absum, what)


def check_conv_basic(rt, oracle):
    ctx = new_ctx(rt)
    # reference goldens (src/ops/conv.rs:783-839); 1-channel 3x3 goes through the explicit-im2col path
    K = np.array([0.3230, 0.7632, 0.4616, 0.8837, 0.5898, 0.3424, 0.2101, 0.7821, 0.6861], np.float32).reshape(1, 1, 3, 3)
    X = np.array([0.5946, 0.8249, 0.0448, 0.9552, 0.2041, 0.2501, 0.2693, 0.1007, 0.8862], np.float32).reshape(1, 1, 3, 3)
    same = np.array([1.5202, 1.5592, 0.9939, 1.7475, 2.6358, 1.3428, 1.0165, 1.1806, 0.8685], np.float32).reshape(1, 1, 3, 3)
    assert np.abs(rt.Conv(padding=(1, 1, 1, 1)).run(ctx, X, K).numpy() - same).max() < 2e-3
    assert np.abs(rt.Conv(padding="same").run(ctx, X, K).numpy() - same).max() < 2e-3
    assert abs(rt.Conv().run(ctx, X, K, np.array([1.0], np.float32)).numpy().item() - 3.6358) < 2e-3
    w = 0.0
    w = max(w, _conv_case(rt, oracle, ctx, (2, 32, 8, 8), (16, 32, 3, 3), pads=(1, 1, 1, 1), cl=True))     # implicit, direct NHWC
    w = max(w, _conv_case(rt, oracle, ctx, (2, 32, 8, 8), (16, 32, 3, 3), pads=(1, 1, 1, 1), cl=False))    # implicit via NHWC copy, NCHW out
    w = max(w, _conv_case(rt, oracle, ctx, (2, 64, 9, 7), (40, 64, 1, 1), cl=True))                        # pointwise
    w = max(w, _conv_case(rt, oracle, ctx, (1, 3, 16, 16), (8, 3, 7, 7), pads=(3, 3, 3, 3), strides=(2, 2)))  # explicit (C=3 stem)
    return f"worst err/bound {w:.3f}"


def check_conv_stride(rt, oracle):
    ctx = new_ctx(rt)
    w = _conv_case(rt, oracle, ctx, (2, 32, 12, 12), (24, 32, 3, 3), pads=(1, 1, 1, 1), strides=(2, 2), cl=True)
    w = max(w, _conv_case(rt, oracle, ctx, (2, 64, 14, 14), (32, 64, 1, 1), strides=(2, 2), cl=True))
    w = max(w, _conv_case(rt, oracle, ctx, (1, 32, 13, 11), (8, 32, 3, 2), pads=(0, 1, 2, 0), strides=(2, 1), cl=True))
    w = max(w, _conv_case(rt, oracle, ctx, (1, 32, 10, 10), (8, 32, 3, 3), pads=(2, 2, 2, 2), strides=(2, 3), dil=(2, 2), cl=True))
    return f"worst err/bound {w:.3f}"


def check_conv_more(rt, oracle):
    ctx = new_ctx(rt)
    w = 0.0
    w = max(w, _conv_case(rt, oracle, ctx, (2, 8, 9, 7), (6, 4, 3, 2), pads=(0, 1, 2, 0), strides=(2, 1), groups=2))           # grouped, explicit
    w = max(w, _conv_case(rt, oracle, ctx, (2, 64, 9, 7), (12, 32, 3, 3), pads=(1, 1, 1, 1), groups=2, cl=True))                # grouped, implicit
    w = max(w, _conv_case(rt, oracle, ctx, (3, 64, 7, 7), (128, 64, 3, 3), pads=(1, 1, 1, 1), cl=True, prepack=True, residual=True, act=1))
    w = max(w, _conv_case(rt, oracle, ctx, (4, 96, 14, 14), (80, 96, 3, 3), pads=(1, 1, 1, 1), cl=True, bias=False))            # C tail (96 = 3*32), odd N
    w = max(w, _conv_case(rt, oracle, ctx, (2, 40, 6, 6), (16, 40, 3, 3), pads=(1, 1, 1, 1), cl=True))                          # C=40: K tail inside a block
    w = max(w, _conv_case(rt, oracle, ctx, (2, 16, 5, 5), (8, 16, 1, 1), cl=False, residual=True, act=1))
    # small-channel path (C <= 4): stem-like shapes, both layouts, asymmetric pads, stride, vertical dilation
    w = max(w, _conv_case(rt, oracle, ctx, (2, 3, 33, 29), (16, 3, 7, 7), pads=(3, 3, 3, 3), strides=(2, 2), cl=True))
    w = max(w, _conv_case(rt, oracle, ctx, (2, 3, 33, 29), (16, 3, 7, 7), pads=(3, 3, 3, 3), strides=(2, 2), cl=False, act=1))
    w = max(w, _conv_case(rt, oracle, ctx, (1, 4, 12, 12), (8, 4, 5, 5), pads=(2, 2, 2, 2), cl=True))
    w = max(w, _conv_case(rt, oracle, ctx, (3, 2, 9, 14), (5, 2, 3, 4), pads=(0, 2, 1, 0), strides=(1, 3), dil=(2, 1)))
    w = max(w, _conv_case(rt, oracle, ctx, (2, 1, 10, 10), (6, 1, 3, 8), pads=(1, 4, 1, 3), residual=True))
    # pair mode / odd tile counts / N tails through the TMA-store epilogue
    w = max(w, _conv_case(rt, oracle, ctx, (5, 32, 20, 20), (72, 32, 3, 3), pads=(1, 1, 1, 1), cl=True))
    w = max(w, _conv_case(rt, oracle, ctx, (3, 64, 28, 28), (100, 64, 1, 1), cl=True, residual=True, act=1))
    # 1-D conv (conv.rs:142-185)
    r = oracle.XorShiftRng(5)
    x, k = r.uniform((2, 3, 11)), r.uniform((4, 3, 3))
    got = rt.Conv(1, (1,), (1, 1), (2,)).run(ctx, x, k).numpy()
    exp = oracle.conv(x, k, None, [1, 1], 1, (2,), (1,))
    assert got.shape == exp.shape and np.abs(got - exp).max() < 5e-3, "Conv 1-D"
    z = lambda *s: np.zeros(s, np.float32)
    for args, kwargs, kind, msg in [((z(1, 3, 5, 5), z(2, 2, 3, 3)), {}, "IncompatibleInputShapes", "Input channels (per group) does not match kernel input channels"),
                                    ((z(1, 2, 5, 5), z(2, 2, 3, 3)), {"groups": 0}, "InvalidValue", "Group count must be > 0"),
                                    ((z(1, 3, 5, 5), z(2, 1, 3, 3)), {"groups": 2}, "InvalidValue", "Input channel count not divisible by groups"),
                                    ((z(1, 4, 5, 5), z(3, 2, 3, 3)), {"groups": 2}, "InvalidValue", "Output channel count not divisible by groups"),
                                    ((z(1, 1, 2, 2), z(1, 1, 3, 3)), {}, "InvalidValue", "Input too small for kernel size"),
                                    ((z(1, 1, 5, 5), z(1, 1, 3, 3)), {"strides": (0, 1)}, "InvalidValue", "Strides must be > 0"),
                                    ((z(1, 1, 5, 5), z(1, 1, 3, 3)), {"strides": (1,)}, "InvalidValue", "expected 2 stride values")]:
        try:
            rt.Conv(**kwargs).run(ctx, *args)
            raise AssertionError("expected error")
        except rt.OpError as e:
            assert e.kind == kind and e.msg == msg, str(e)
    return f"worst err/bound {w:.3f}"


def check_conv_integer(rt, oracle):
    ctx = new_ctx(rt)
    rng = oracle.XorShiftRng(1234)
    krng = oracle.XorShiftRng(5678)
    mk = lambda r, s, dt: (r.u8(s).view(np.int8) if dt == np.int8 else r.u8(s))
    # the reference's case table (src/ops/conv.rs:1429-1497), all four signedness combos
    for xdt in (np.uint8, np.int8):
        for wdt in (np.uint8, np.int8):
            for xs, ws, xz, wz, g in [((1, 2, 5, 5), (1, 2, 3, 3), 12, [1], 1), ((1, 2, 5, 5), (3, 2, 3, 3), 12, [1, 2, 3], 1),
                                      ((1, 4, 5, 5), (4, 2, 3, 3), 12, [1, 2, 3, 4], 2), ((1, 2, 5, 5), (1, 2, 3, 3), None, None, 1),
                                      ((1, 2, 5, 5), (1, 2, 1, 1), 12, [1], 1), ((1, 2, 1, 1), (1, 2, 1, 1), 12, [1], 1)]:
                x, w = mk(rng, xs, xdt), mk(krng, ws, wdt)
                xzp = None if xz is None else np.array(xz, xdt)
                wzp = None if wz is None else np.array(wz, wdt)
                got = rt.ConvInteger(groups=g).run(ctx, x, w, xzp, wzp).numpy()
                assert_bit_exact(got, oracle.conv_integer(x, w, xzp, wzp, groups=g), f"ConvInteger {xdt.__name__}/{wdt.__name__} x{xs} w{ws}")
    # tensor-core path: 16-byte channel groups, padding (production path: G3), stride, zero points, channels-last
    for xdt in (np.uint8, np.int8):
        for xs, ws, pads, st, cl in [((2, 32, 9, 9), (24, 32, 3, 3), (1, 1, 1, 1), (1, 1), True), ((2, 64, 12, 10), (16, 64, 3, 3), (1, 1, 1, 1), (2, 2), True),
                                     ((2, 128, 7, 7), (40, 128, 1, 1), (0, 0, 0, 0), (1, 1), True), ((1, 16, 8, 8), (8, 16, 3, 3), (1, 0, 1, 0), (1, 1), False),
                                     # small-channel 8-bit path (quantised RGB stem): padded 16-byte pixels, one K block per filter row
                                     ((2, 3, 32, 32), (16, 3, 7, 7), (3, 3, 3, 3), (2, 2), True), ((3, 1, 12, 13), (8, 1, 3, 3), (1, 1, 1, 1), (1, 1), False),
                                     ((2, 4, 9, 9), (32, 4, 5, 5), (2, 1, 0, 2), (1, 2), True)]:
            x, w = mk(rng, xs, xdt), krng.i8(ws)
            xzp, wzp = np.array(77 if xdt == np.uint8 else -3, xdt), krng.i8((ws[0],))
            for zx, zw in [(xzp, wzp), (xzp, None), (None, wzp), (None, None)]:
                op = rt.ConvInteger(padding=pads, strides=st)
                got = op.run(ctx, ctx.to_device(x, channels_last=cl), w, zx, zw).numpy()
                assert_bit_exact(got, oracle.conv_integer(x, w, zx, zw, padding=list(pads), strides=st),
                                 f"ConvInteger tc {xdt.__name__} x{xs} w{ws} pads={pads} s={st} zp={zx is not None},{zw is not None}")
    x, w = rng.u8((2, 32, 9, 9)), krng.i8((24, 32, 3, 3))
    op = rt.ConvIntegerToFloat(padding=(1, 1, 1, 1))
    pk = op.prepack(ctx, 1, w)
    got = op.run(ctx, ctx.to_device(x, True), w, np.uint8(12), None, np.float32(0.1), packed_w=pk).numpy()
    assert_bit_exact(got, oracle.conv_integer_to_float(x, w, np.uint8(12), None, np.float32(0.1), padding=[1, 1, 1, 1]), "ConvIntegerToFloat")
    try:
        op.run(ctx, x, w, np.uint8(12), None, np.array([0.1, 0.2, 0.3], np.float32))
        raise AssertionError("expected error")
    except rt.OpError as e:
        assert e.msg == "scale should be a scalar", str(e)
    return "ok"


def check_conv_integer_fused(rt, oracle):
    """ConvIntegerToFloat with the following Add(bias) / Add(identity) / Relu folded into the epilogue must be
    bit-identical to the separate operators (exact f32 mul, add, add, max), channels-last and NCHW, all plan kinds."""
    ctx = new_ctx(rt)
    r = oracle.XorShiftRng(77)
    worst = 0
    for (xs, ws, pads, strides, cl) in [((2, 64, 14, 14), (128, 64, 1, 1), (0, 0, 0, 0), (1, 1), True),
                                        ((2, 64, 14, 14), (64, 64, 3, 3), (1, 1, 1, 1), (1, 1), True),
                                        ((3, 32, 9, 9), (48, 32, 3, 3), (1, 1, 1, 1), (2, 2), False),
                                        ((2, 128, 7, 7), (96, 128, 1, 1), (0, 0, 0, 0), (1, 1), True)]:
        x = r.u8(xs)
        w = r.i8(ws)
        xz = np.uint8(121)
        scale = np.float32(0.0173)
        bias = r.uniform((ws[0],))
        op = rt.ConvIntegerToFloat(1, (1, 1), pads, strides)
        base = oracle.conv_integer_to_float(x, w, xz, None, scale, padding=list(pads), groups=1, strides=strides, dilations=(1, 1))
        res = r.uniform(base.shape)
        xd = ctx.to_device(x, channels_last=cl)
        for use_res in (False, True):
            for act in (0, 1):
                want = oracle.add(base, bias.reshape(1, -1, 1, 1))
                if use_res:
                    want = oracle.add(want, res)
                if act:
                    want = oracle.relu(want)
                op.activation = act
                got = op.run(ctx, xd, w, xz, None, scale, bias=bias, residual=(ctx.to_device(res, channels_last=cl) if use_res else None)).numpy()
                assert_bit_exact(got, want, f"ConvIntegerToFloat fused x{xs} w{ws} res={use_res} act={act} cl={cl}")
                worst += 1
    # the Mul(x_scale, w_scale) node folded into the epilogue (scale_b) and an 8-bit scalar zero point read in place
    x, w = r.u8((2, 64, 12, 12)), r.i8((96, 64, 3, 3))
    xs_, ws_, xz = np.float32(0.0371), np.float32(0.0042), np.uint8(97)
    op = rt.ConvIntegerToFloat(1, (1, 1), (1, 1, 1, 1), (1, 1))
    want = oracle.conv_integer_to_float(x, w, xz, None, np.float32(xs_ * ws_), padding=[1, 1, 1, 1], groups=1, strides=(1, 1), dilations=(1, 1))
    got = op.run(ctx, ctx.to_device(x, channels_last=True), w, xz, None, ws_, scale_b=xs_).numpy()
    assert_bit_exact(got, want, "ConvIntegerToFloat with folded scale product")
    a8, b8 = r.u8((70, 256)), r.i8((256, 96))
    wsv = r.uniform((96,), 0.001, 0.01)
    want = oracle.matmul_integer_to_float(a8, b8, xz, None, (xs_ * wsv).astype(np.float32))
    got = rt.MatMulIntegerToFloat().run(ctx, a8, b8, xz, None, wsv, scale_b=xs_).numpy()
    assert_bit_exact(got, want, "MatMulIntegerToFloat with folded scale product")
    # Mul (used for x_scale * w_scale)
    a, b = r.uniform((5, 1, 7)), r.uniform((3, 1))
    assert_bit_exact(rt.Mul().run(ctx, a, b).numpy(), (a * b).astype(np.float32), "Mul broadcast")
    return f"{worst} fused cases bit-exact"


def check_resnet50_int8_model(rt, oracle):
    """configs[3]: dynamically quantised ResNet-50 (DynamicQuantizeLinear -> ConvIntegerToFloat -> Add -> Relu ...), full
    224x224 images.  Every operator up to the pooled features is exact integer or exactly rounded f32 arithmetic, so
    those features must be BIT-IDENTICAL to the CPU oracle's -- fused or not, with the exported per-channel zero weight
    zero points or with that constant dropped; the f32 classifier on top carries the TF32 tolerance."""
    from rten_b200 import graphs
    import model_ref
    ctx = new_ctx(rt)
    rng = oracle.XorShiftRng(5678)
    spec = graphs.make_resnet50(lambda s: rng.uniform(s))
    q = graphs.quantize_resnet50(spec)
    x = oracle.XorShiftRng(4321).uniform((2, 3, 224, 224))
    ref, ref_feat = model_ref.resnet50_int8_oracle(oracle, q, x)
    worst = 0.0
    for fuse, wz in ((True, False), (True, True), (False, True)):
        logits, feat = graphs.ResNet50Int8Runner(ctx, q, fuse=fuse, w_zero_points=wz).run(ctx.to_device(x, channels_last=True), True)
        assert_bit_exact(feat.numpy(), ref_feat, f"ResNet-50 int8 pooled features (fuse={fuse}, w_zp={wz})")
        rel = float(np.abs(logits.numpy() - ref).max() / np.abs(ref).max())
        assert rel <= 2e-3, f"ResNet-50 int8 logits (f32 classifier, TF32): rel err {rel:.3e}"
        worst = max(worst, rel)
    f32 = model_ref.resnet50_oracle(oracle, spec, x)
    drift = float(np.abs(ref - f32).max() / np.abs(f32).max())
    return f"features bit-exact; classifier rel err {worst:.1e}; int8 vs fp32 model drift {drift:.3f} of max |logit|"


def check_gpt2_int8_kvcache(rt, oracle):
    """configs[4]: dynamically quantised GPT-2 blocks (full width 768 / 12 heads / FFN 3072), prefill then decode steps
    against a device-resident KV cache.  Linear layers are exact (int8 + exactly rounded f32 epilogue); the two attention
    products run single-pass TF32, and a last-bit change there can move a dynamically quantised activation by one
    step, so logits are compared with a stated tolerance: max |d| <= 2e-2 * max |ref|.  Fused and unfused epilogues
    must agree with each other bit for bit."""
    from rten_b200 import graphs
    import model_ref
    ctx = new_ctx(rt)
    rng = oracle.XorShiftRng(5678)
    spec = graphs.make_gpt2_int8(lambda s: rng.uniform(s), layers=3, vocab=5000, max_pos=128)
    B, T0 = 2, 40
    ids = (oracle.XorShiftRng(1).u64(B * (T0 + 3)) % 5000).astype(np.int32).reshape(B, T0 + 3)
    steps = [ids[:, :T0]] + [ids[:, T0 + i:T0 + i + 1] for i in range(3)]
    ref = model_ref.gpt2_int8_oracle(oracle, spec, steps)
    outs = {}
    for fuse in (True, False):
        runner = graphs.GPT2Int8Runner(ctx, spec, B, 64, fuse=fuse)
        outs[fuse] = [runner.forward(st).numpy() for st in steps]
    worst = 0.0
    for i, (a, b, r) in enumerate(zip(outs[True], outs[False], ref)):
        assert_bit_exact(a, b, f"GPT-2 int8 step {i}: fused vs unfused epilogues")
        rel = float(np.abs(a - r).max() / np.abs(r).max())
        assert a.shape == r.shape and rel <= 2e-2, f"GPT-2 int8 step {i}: rel err {rel:.3e}"
        assert (a.argmax(1) == r.argmax(1)).all(), f"GPT-2 int8 step {i}: greedy token differs"
        worst = max(worst, rel)
    # decode steps replayed as ONE CUDA graph: the fused path (quantised-linear skinny kernels + single-query attention
    # with the cache append inside) and the separate operators (ScatterRows append, fixed-length masked attention)
    for fused in (True, False):
        runner = graphs.GPT2Int8Runner(ctx, spec, B, 64, fuse=True)
        g_out = [runner.forward(steps[0]).numpy()]
        runner.build_decode_graph(fused=fused)
        g_out += [runner.decode_step(st).numpy().copy() for st in steps[1:]]
        for i, (a, r) in enumerate(zip(g_out, ref)):
            rel = float(np.abs(a - r).max() / np.abs(r).max())
            assert rel <= 2e-2 and (a.argmax(1) == r.argmax(1)).all(), f"GPT-2 int8 graph decode (fused={fused}) step {i}: rel err {rel:.3e}"
            worst = max(worst, rel)
    return f"prefill {T0} + 3 decode steps (eager, graph-replayed fused and unfused), worst rel err {worst:.2e}"


def check_tf32x3(rt, oracle):
    """RTEN_F32_TF32X3: three TF32 passes over split operands (hi*hi + hi*lo + lo*hi).  Stated tolerance:
    |got - exact| <= 2^-18 * sum_k |a_k b_k| + 1e-6 -- 500x tighter than the single-pass bound and of the order of the
    reference's own f32 accumulation error; whole ResNet-50 logits within 1e-4 of max |ref| (single pass: ~1e-3)."""
    global TF32_REL
    from rten_b200 import graphs
    import model_ref
    ctx = new_ctx(rt, tf32=False)
    saved = TF32_REL
    TF32_REL = 2.0 ** -18
    try:
        w = _matmul_case(rt, oracle, ctx, (128, 64), (64, 128))
        w = max(w, _matmul_case(rt, oracle, ctx, (3, 130, 520), (520, 300), seed=6))
        w = max(w, _matmul_case(rt, oracle, ctx, (2, 4, 64, 33), (2, 4, 33, 70), seed=9))            # batched B, K % 4 != 0
        w = max(w, _matmul_case(rt, oracle, ctx, (384, 1024), (1024, 512), bias=True, prepack=True, seed=5))
        w = max(w, _conv_case(rt, oracle, ctx, (2, 64, 20, 20), (96, 64, 1, 1), cl=True))
        w = max(w, _conv_case(rt, oracle, ctx, (2, 32, 14, 14), (64, 32, 3, 3), pads=(1, 1, 1, 1), cl=True, residual=True, act=1))
        w = max(w, _conv_case(rt, oracle, ctx, (2, 16, 9, 9), (32, 8, 3, 3), pads=(1, 1, 1, 1), groups=2, strides=(2, 2), cl=False))
        w = max(w, _conv_case(rt, oracle, ctx, (2, 3, 32, 32), (16, 3, 7, 7), pads=(3, 3, 3, 3), strides=(2, 2), cl=True))   # stem-like
    finally:
        TF32_REL = saved
    # The two-plane form (A = original tensor for both `hi` segments + a low-part plane; prepacked B split once and
    # cached) must be BIT-IDENTICAL to the three-segment copies built per call: kind::tf32 ignores the 13 low
    # mantissa bits, so feeding the raw f32 values is the same as feeding their truncations.
    import os
    r = oracle.XorShiftRng(99)
    n_same = 0
    for (xs, ws, pads, strides) in [((4, 64, 14, 14), (128, 64, 3, 3), (1, 1, 1, 1), (1, 1)), ((3, 256, 9, 9), (64, 256, 1, 1), (0, 0, 0, 0), (1, 1)),
                                    ((2, 96, 12, 12), (32, 96, 3, 3), (1, 1, 1, 1), (2, 2))]:
        x = ctx.to_device(r.f32(xs), channels_last=True)
        wt = ctx.to_device(r.f32(ws))
        op = rt.Conv(1, (1, 1), pads, strides, activation=rt.ACT_RELU)
        pk = op.prepack(ctx, 1, wt)
        two = op.run(ctx, x, wt, packed_w=pk).numpy()
        os.environ["RTEN_B200_X3_THREE_PLANES"] = "1"
        os.environ["RTEN_B200_X3_NO_CACHE"] = "1"
        try:
            three = op.run(ctx, x, wt, packed_w=pk).numpy()
        finally:
            os.environ.pop("RTEN_B200_X3_THREE_PLANES")
            os.environ.pop("RTEN_B200_X3_NO_CACHE")
        assert_bit_exact(two, three, f"3xTF32 conv {xs}x{ws}: two-plane vs three-segment operands")
        n_same += 1
    a, b = r.f32((300, 768)), r.f32((768, 320))
    db = ctx.to_device(b)
    pk = rt.MatMul().prepack(ctx, 1, db)
    two = rt.MatMul().run(ctx, ctx.to_device(a), db, packed_b=pk).numpy()
    os.environ["RTEN_B200_X3_THREE_PLANES"] = "1"
    os.environ["RTEN_B200_X3_NO_CACHE"] = "1"
    try:
        three = rt.MatMul().run(ctx, ctx.to_device(a), db, packed_b=pk).numpy()
    finally:
        os.environ.pop("RTEN_B200_X3_THREE_PLANES")
        os.environ.pop("RTEN_B200_X3_NO_CACHE")
    assert_bit_exact(two, three, "3xTF32 MatMul 300x768x320: two-plane vs three-segment operands")
    assert_reference_rule(two, oracle.matmul(a, b), "3xTF32 MatMul 300x768x320 (two-plane)")
    rng = oracle.XorShiftRng(5678)
    spec = graphs.make_resnet50(lambda s: rng.uniform(s))
    x = oracle.XorShiftRng(1234).uniform((2, 3, 224, 224))
    ref = model_ref.resnet50_oracle(oracle, spec, x)
    got = graphs.ResNet50Runner(ctx, spec, fuse=True).run(ctx.to_device(x, channels_last=True)).numpy()
    rel = float(np.abs(got - ref).max() / np.abs(ref).max())
    assert rel <= 1e-4, f"ResNet-50 logits in 3xTF32 mode: rel err {rel:.3e}"
    return f"worst err/bound {w:.3f} (bound 2^-18); {n_same + 1} two-plane launches bit-identical to three-segment ones; ResNet-50 logits rel err {rel:.2e}"


def check_mnist_model(rt, oracle):
    """configs[0]: the reference's MNIST test model with its real weights (tests/golden/mnist.npz): 1-channel stem through
    the small-C path, 72-channel pointwise conv, 2x2 max pooling, ReduceMean, Gemm.  Single-pass TF32 within 1e-2 of
    max |logit| (the whole-model bound used for ResNet-50 too), 3xTF32 within 5e-5; fused and unfused epilogues; batch 1 (the reference's test input) and batch 5."""
    import os
    from rten_b200 import graphs
    import model_ref
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "mnist.npz")
    w = graphs.load_mnist_weights(path)
    x1 = np.full((1, 1, 28, 28), 0.5, np.float32)
    x5 = np.concatenate([x1, oracle.XorShiftRng(8).uniform((4, 1, 28, 28))], 0)
    out = []
    for x in (x1, x5):
        ref = model_ref.mnist_oracle(oracle, w, x)
        for x3, tol in ((False, 1e-2), (True, 5e-5)):
            ctx = new_ctx(rt, tf32=not x3)
            for fuse in (True, False):
                got = graphs.MnistRunner(ctx, w, fuse=fuse).run(ctx.to_device(x)).numpy()
                rel = float(np.abs(got - ref).max() / np.abs(ref).max())
                assert got.shape == ref.shape and rel <= tol, f"MNIST logits (batch {x.shape[0]}, x3={x3}, fuse={fuse}): rel err {rel:.3e}"
                assert (got.argmax(1) == ref.argmax(1)).all()
                out.append(rel)
    return f"rel err tf32 {max(out[0::4] + out[1::4]):.1e}, 3xtf32 {max(out[2::4] + out[3::4]):.1e}"


def check_resnet50_model(rt, oracle):
    """Whole-model parity (ResNet-50 fp32, full 224x224 images, batch 2): every conv runs single-pass TF32,
    so the logits carry ~53 layers of 2^-11-relative operand rounding.  Stated tolerance: max |d| <= 1e-2 * max |ref|."""
    from rten_b200 import graphs
    import model_ref
    ctx = new_ctx(rt)
    rng = oracle.XorShiftRng(5678)
    spec = graphs.make_resnet50(lambda s: rng.uniform(s))
    x = oracle.XorShiftRng(1234).uniform((2, 3, 224, 224))
    ref = model_ref.resnet50_oracle(oracle, spec, x)
    outs = {}
    for fuse in (True, False):
        runner = graphs.ResNet50Runner(ctx, spec, fuse=fuse)
        outs[fuse] = runner.run(ctx.to_device(x, channels_last=True)).numpy()
        rel = float(np.abs(outs[fuse] - ref).max() / np.abs(ref).max())
        assert outs[fuse].shape == ref.shape and rel <= 1e-2, f"ResNet-50 logits (fuse={fuse}): rel err {rel:.3e}"
        assert (outs[fuse].argmax(1) == ref.argmax(1)).all()
    # NCHW-contiguous input (the reference's native layout) must give the same answer as channels-last
    y_nchw = graphs.ResNet50Runner(ctx, spec, fuse=True).run(ctx.to_device(x)).numpy()
    rel2 = float(np.abs(y_nchw - ref).max() / np.abs(ref).max())
    assert rel2 <= 1e-2, f"ResNet-50 NCHW input rel err {rel2:.3e}"
    return f"rel err fused {float(np.abs(outs[True] - ref).max() / np.abs(ref).max()):.2e} unfused {float(np.abs(outs[False] - ref).max() / np.abs(ref).max()):.2e} nchw {rel2:.2e}"


def check_bert_model(rt, oracle):
    """BERT-base encoder, 3 layers, batch 2 x seq 128 (full width 768/3072).  Tolerance: max |d| <= 1e-2 (LayerNorm
    keeps activations O(1))."""
    from rten_b200 import graphs
    import model_ref
    ctx = new_ctx(rt)
    rng = oracle.XorShiftRng(5678)
    spec = graphs.make_bert(lambda s: rng.uniform(s), layers=3)
    ids = (oracle.XorShiftRng(1234).u64(2 * 128) % 30522).astype(np.int32).reshape(2, 128)
    tt = np.zeros((2, 128), np.int32)
    tt[:, 64:] = 1
    mask = np.zeros((2, 1, 1, 128), np.float32)
    mask[1, :, :, 100:] = -10000.0
    ref = model_ref.bert_oracle(oracle, spec, ids, tt, mask)
    res = []
    for fuse in (True, False):
        runner = graphs.BertRunner(ctx, spec, fuse=fuse)
        got = runner.run(ctx.to_device(ids), ctx.to_device(tt), ctx.to_device(mask)).numpy()
        err = float(np.abs(got - ref).max())
        assert got.shape == ref.shape and err <= 1e-2, f"BERT hidden states (fuse={fuse}): max abs err {err:.3e}"
        res.append(err)
    return f"max abs err fused {res[0]:.2e} unfused {res[1]:.2e} (|ref| max {float(np.abs(ref).max()):.2f})"


# ------------------------------------------------------------------------------------------
# The reference's own float rule on the reference's own kind of test data
# ------------------------------------------------------------------------------------------
def check_reference_rule_f32(rt, oracle):
    """Library default (3xTF32): MatMul / Gemm / Conv outputs obey the reference's comparison rule
    |got - oracle| <= 1e-8 + 1e-5 * |oracle| (rten-tensor/src/test_util.rs:47-92) element by element, on the kind of
    data the reference's tests draw -- XorShiftRng f32 in [0, 1) (rten-gemm/src/tests.rs:336-362, src/ops/conv.rs:1131-1319) --
    at the reference's sweep sizes and at the BASELINE layer sizes.  (Signed data with cancellation is covered by the
    sum |a b| bounds of check_tf32x3: no two f32 summation orders agree to 1e-5 of a result that cancels to ~0.)"""
    ctx = rt.Context(0)  # untouched default mode
    r = oracle.XorShiftRng(1234)
    n = 0
    for (m, k, nn) in [(1, 1, 1), (2, 2, 2), (5, 7, 10), (17, 33, 9), (64, 64, 64), (130, 520, 300), (2048, 768, 768), (32, 2048, 1000)]:
        a, b = r.f32((m, k)), r.f32((k, nn))
        assert_reference_rule(rt.MatMul().run(ctx, a, b).numpy(), oracle.matmul(a, b), f"MatMul {m}x{k}x{nn} (reference rule)")
        n += 1
    a, b, c = r.f32((40, 96)), r.f32((50, 96)), r.f32((50,))
    assert_reference_rule(rt.Gemm(0.5, 2.0, False, True).run(ctx, a, b, c).numpy(), oracle.gemm_op(a, b, c, 0.5, 2.0, False, True),
                          "Gemm alpha/beta/transB (reference rule)")
    q, kt = r.f32((2, 12, 128, 64)), r.f32((2, 12, 64, 128))
    assert_reference_rule(rt.FusedMatMul(0.125).run(ctx, q, kt).numpy(), oracle.matmul(q, kt, None, 0.125), "batched QK^T (reference rule)")
    for xs, ws, pads, st in [((2, 3, 20, 20), (8, 3, 3, 3), (1, 1, 1, 1), (1, 1)), ((2, 64, 56, 56), (64, 64, 3, 3), (1, 1, 1, 1), (1, 1)),
                             ((2, 256, 14, 14), (1024, 256, 1, 1), (0, 0, 0, 0), (1, 1)), ((2, 128, 28, 28), (128, 128, 3, 3), (1, 1, 1, 1), (2, 2)),
                             ((1, 3, 64, 64), (16, 3, 7, 7), (3, 3, 3, 3), (2, 2))]:
        x, w, b = r.f32(xs), r.f32(ws), r.f32((ws[0],))
        want = oracle.conv(x, w, b, list(pads), 1, st, (1, 1))
        for cl in (False, True):
            got = rt.Conv(1, (1, 1), pads, st).run(ctx, ctx.to_device(x, channels_last=cl), w, b).numpy()
            assert_reference_rule(got, want, f"Conv {xs} * {ws} cl={cl} (reference rule)")
            n += 1
    return f"{n} MatMul / Conv cases inside 1e-8 + 1e-5*|ref|"


# ------------------------------------------------------------------------------------------
# Parity at the exact BASELINE sizes, on the graphs bench.py times (autotuned plans, CUDA-graph replay)
# ------------------------------------------------------------------------------------------
def _replayed(ctx, fn):
    """Eager pass (autotunes, warms the pool), then capture + replay: the output of the REPLAY is what is compared."""
    ctx.set_autotune(True)
    first = fn()
    ctx.sync()
    ctx.set_autotune(False)
    del first
    ctx.graph_begin()
    out = fn()
    g = ctx.graph_end()
    if out.dtype == np.float32:
        out.copy_from(np.full(out.shape, np.nan, np.float32))
    g.launch()
    ctx.sync()
    return out, g


def check_resnet50_b32_baseline(rt, oracle):
    """configs[1] exactly as benched: ResNet-50 fp32, batch 32, autotuned launch plans (split-K, CTA pairs ...), the step
    replayed from a CUDA graph.  TF32 single pass: logits within 1e-2 * max |ref|; 3xTF32 (library default): within
    1e-4 * max |ref| and the same arg-max on every image."""
    from rten_b200 import graphs
    import model_ref
    rng = oracle.XorShiftRng(5678)
    spec = graphs.make_resnet50(lambda s: rng.uniform(s))
    x = oracle.XorShiftRng(1234).uniform((32, 3, 224, 224))
    oracle.use_all_cores()
    ref = model_ref.resnet50_oracle(oracle, spec, x)
    res = {}
    for name, tf32, tol in (("tf32", True, 1e-2), ("tf32x3", False, 1e-4)):
        ctx = new_ctx(rt, tf32=tf32)
        runner = graphs.ResNet50Runner(ctx, spec, fuse=True)
        xd = ctx.to_device(x, channels_last=True)
        out, g = _replayed(ctx, lambda: runner.run(xd))
        got = out.numpy()
        rel = float(np.abs(got - ref).max() / np.abs(ref).max())
        assert got.shape == ref.shape and rel <= tol, f"ResNet-50 b32 ({name}): rel err {rel:.3e} > {tol}"
        assert (got.argmax(1) == ref.argmax(1)).all(), f"ResNet-50 b32 ({name}): arg-max differs"
        res[name] = rel
        del g
    return f"b32 graph replay: rel err tf32 {res['tf32']:.2e}, tf32x3 {res['tf32x3']:.2e}"


def check_bert_b16_baseline(rt, oracle):
    """configs[2] exactly as benched: BERT-base, 12 layers, batch 16 x seq 128, graph replay.  TF32: hidden states within
    3e-2 absolute (12 layers of 2^-11-relative operand rounding; LayerNorm keeps activations O(1)); 3xTF32: within 2e-4."""
    from rten_b200 import graphs
    import model_ref
    rng = oracle.XorShiftRng(5678)
    spec = graphs.make_bert(lambda s: rng.uniform(s))
    ids = (oracle.XorShiftRng(1234).u64(16 * 128) % 30522).astype(np.int32).reshape(16, 128)
    tt = np.zeros((16, 128), np.int32)
    mask = np.zeros((16, 1, 1, 128), np.float32)
    oracle.use_all_cores()
    ref = model_ref.bert_oracle(oracle, spec, ids, tt, mask)
    res = {}
    for name, tf32, tol in (("tf32", True, 3e-2), ("tf32x3", False, 2e-4)):
        ctx = new_ctx(rt, tf32=tf32)
        runner = graphs.BertRunner(ctx, spec, fuse=True)
        di, dt, dm = ctx.to_device(ids), ctx.to_device(tt), ctx.to_device(mask)
        out, g = _replayed(ctx, lambda: runner.run(di, dt, dm))
        got = out.numpy()
        err = float(np.abs(got - ref).max())
        assert got.shape == ref.shape and err <= tol, f"BERT-base b16 x s128 ({name}): max abs err {err:.3e} > {tol}"
        res[name] = err
        del g
    return f"12 layers b16 x s128 graph replay: max abs err tf32 {res['tf32']:.2e}, tf32x3 {res['tf32x3']:.2e}"


def check_resnet50_int8_b64_baseline(rt, oracle):
    """configs[3] exactly as benched: dynamically quantised ResNet-50, batch 64, fused epilogues, graph replay: pooled
    features BIT-IDENTICAL to the oracle."""
    from rten_b200 import graphs
    import model_ref
    rng = oracle.XorShiftRng(5678)
    spec = graphs.make_resnet50(lambda s: rng.uniform(s))
    q = graphs.quantize_resnet50(spec)
    x = oracle.XorShiftRng(1234).uniform((64, 3, 224, 224))
    oracle.use_all_cores()
    ref, ref_feat = model_ref.resnet50_int8_oracle(oracle, q, x)
    ctx = new_ctx(rt)
    runner = graphs.ResNet50Int8Runner(ctx, q, fuse=True)
    xd = ctx.to_device(x, channels_last=True)
    ctx.set_autotune(True)
    runner.run(xd, True)
    ctx.sync()
    ctx.set_autotune(False)
    ctx.graph_begin()
    logits, feat = runner.run(xd, True)
    g = ctx.graph_end()
    feat.copy_from(np.zeros(feat.shape, np.float32))
    g.launch()
    ctx.sync()
    assert_bit_exact(feat.numpy(), ref_feat, "ResNet-50 int8 b64 pooled features (graph replay)")
    rel = float(np.abs(logits.numpy() - ref).max() / np.abs(ref).max())
    assert rel <= 2e-3, f"ResNet-50 int8 b64 logits: rel err {rel:.3e}"
    return f"b64 features bit-exact; classifier rel err {rel:.1e}"


def check_gpt2_b8_baseline(rt, oracle):
    """configs[4] exactly as benched: GPT-2 small int8, 12 layers, vocabulary 50257, batch 8: prefill of 512 tokens, then
    8 decode steps replayed from ONE CUDA graph against the 576-position KV cache.  Last-position logits within
    2e-2 * max |ref| of the oracle's at every step, greedy tokens equal; the graph-replayed prefill bit-identical to the eager one."""
    from rten_b200 import graphs
    import model_ref
    rng = oracle.XorShiftRng(5678)
    spec = graphs.make_gpt2_int8(lambda s: rng.uniform(s))
    B, T0, nd = 8, 512, 8
    ids = (oracle.XorShiftRng(1).u64(B * (T0 + nd)) % 50257).astype(np.int32).reshape(B, T0 + nd)
    steps = [ids[:, :T0]] + [ids[:, T0 + i:T0 + i + 1] for i in range(nd)]
    oracle.use_all_cores()
    ref = model_ref.gpt2_int8_oracle(oracle, spec, steps)
    ctx = new_ctx(rt, tf32=False)  # the f32 attention products of the prefill at fp32 grade (library default)
    ctx.set_autotune(True)
    runner = graphs.GPT2Int8Runner(ctx, spec, B, 576, fuse=True)
    outs = [runner.forward(steps[0]).numpy()]
    # the prefill as ONE replayed CUDA graph (what bench.py times) must reproduce the eager prefill bit for bit: logits
    # AND the KV cache it leaves behind
    ctx.set_autotune(False)
    k_eager, v_eager = runner.layers[-1]["k"].numpy().copy(), runner.layers[-1]["vt"].numpy().copy()
    runner.reset()
    runner.build_prefill_graph(T0)
    runner.reset()
    for d in runner.layers:
        d["k"].copy_from(np.zeros(d["k"].shape, np.float32))
        d["vt"].copy_from(np.zeros(d["vt"].shape, np.float32))
    assert_bit_exact(runner.prefill(steps[0]).numpy(), outs[0], "GPT-2 int8 b8: graph-replayed prefill vs eager prefill")
    assert_bit_exact(runner.layers[-1]["k"].numpy(), k_eager, "key cache after the graph-replayed prefill")
    assert_bit_exact(runner.layers[-1]["vt"].numpy(), v_eager, "value cache after the graph-replayed prefill")
    ctx.set_autotune(True)
    runner.build_decode_graph()
    ctx.set_autotune(False)
    outs += [runner.decode_step(st).numpy().copy() for st in steps[1:]]
    worst = 0.0
    for i, (a, r) in enumerate(zip(outs, ref)):
        rel = float(np.abs(a - r).max() / np.abs(r).max())
        assert a.shape == r.shape and rel <= 2e-2, f"GPT-2 int8 b8 step {i}: rel err {rel:.3e}"
        assert_same_greedy_token(a, r, 2e-2, f"GPT-2 int8 b8 step {i}")
        worst = max(worst, rel)
    return f"prefill 512 + {nd} graph-replayed decode steps, worst rel err {worst:.2e}"


def check_graph_pool_isolation(rt, oracle):
    """Buffers a captured graph references (temporaries, intermediate outputs freed after capture) never return to the
    pool while the graph exists: allocations made AFTER graph_end cannot alias them, so replays stay correct."""
    ctx = new_ctx(rt)
    r = oracle.XorShiftRng(77)
    a, b = r.uniform((256, 384)), r.uniform((384, 320))
    bias = r.uniform((320,))
    da, db, dbias = ctx.to_device(a), ctx.to_device(b.T.copy()).permute(1, 0), ctx.to_device(bias)
    eager = rt.Gelu().run(ctx, rt.FusedMatMul(None).run(ctx, da, db, dbias)).numpy()
    ctx.graph_begin()
    mid = rt.FusedMatMul(None).run(ctx, da, db, dbias)   # intermediate: freed right after the capture
    out = rt.Gelu().run(ctx, mid)
    g = ctx.graph_end()
    del mid
    # grab (and scribble over) everything the pool would hand out in the sizes the graph uses
    junk = [ctx.to_device(np.full((256, 320), np.nan, np.float32)) for _ in range(6)]
    junk += [ctx.to_device(np.full((n,), 255, np.uint8)) for n in (512, 4096, 65536, 1 << 20)]
    for rep in range(2):
        g.launch()
        ctx.sync()
        assert_bit_exact(out.numpy(), eager, f"graph replay {rep} after post-capture allocations")
        for j in junk[:6]:
            assert np.isnan(j.numpy()).all(), "a post-capture allocation aliases a buffer the graph writes"
    return "replays unaffected by post-capture allocations"


# ------------------------------------------------------------------------------------------
# Decode path: fused quantised linear layer, single-query attention, skinny f32 products
# ------------------------------------------------------------------------------------------
def _qlinear_oracle(oracle, x, ln, wq, wz, ws, bias, residual, act, eps):
    f32 = np.float32
    h = oracle.layer_norm(x, ln[0], ln[1], -1, eps) if ln is not None else x
    xq, xs, xz = oracle.dynamic_quantize_linear(h)
    scale = (f32(xs) * np.asarray(ws, f32)).astype(f32)
    y = oracle.matmul_integer_to_float(xq.reshape(-1, xq.shape[-1]), wq, xz, wz, scale if scale.ndim else scale.reshape(()))
    if bias is not None:
        y = oracle.add(y, bias)
    if residual is not None:
        y = oracle.add(y, residual.reshape(y.shape))
    if act == 3:
        y = oracle.gelu(y, True)
    elif act == 2:
        y = oracle.gelu(y)
    elif act == 1:
        y = oracle.relu(y)
    return y.reshape(x.shape[:-1] + (wq.shape[1],))


def check_quantized_linear(rt, oracle):
    """rten_b200_quantized_linear = [LayerNormalization] -> DynamicQuantizeLinear -> Mul -> MatMulIntegerToFloat -> Add -> Add
    -> activation.  The skinny-M kernel (M <= 16) and the composed path (larger M) must both be BIT-IDENTICAL to the
    oracle's operator chain: GPT-2 decode shapes, per-column and scalar scales, weight zero points, u8 weights."""
    ctx = new_ctx(rt)
    r = oracle.XorShiftRng(4242)
    n = 0
    cases = [  # (x shape, N, layer norm, bias, residual, activation, weight zero points, weight dtype, scalar scale)
        ((8, 768), 2304, True, True, False, 0, None, np.int8, False), ((8, 768), 768, False, True, True, 0, None, np.int8, False),
        ((8, 768), 3072, True, True, False, 3, None, np.int8, False), ((8, 3072), 768, False, True, True, 0, None, np.int8, False),
        ((8, 768), 5003, True, False, False, 0, None, np.int8, False), ((1, 768), 777, True, True, True, 2, "vec", np.int8, False),
        ((3, 5, 256), 130, False, True, False, 1, "vec", np.uint8, True), ((16, 1024), 4100, True, False, True, 0, "scalar", np.int8, False),
        ((13, 128), 64, True, True, False, 0, None, np.uint8, False), ((40, 768), 300, True, True, True, 3, None, np.int8, False),
        ((2, 9, 160), 96, False, False, False, 0, "vec", np.int8, True), ((8, 48), 40, False, True, False, 0, None, np.int8, False)]
    for xs, N, has_ln, has_bias, has_res, act, wzp, wdt, scalar_scale in cases:
        K = xs[-1]
        x = r.uniform(xs, -2, 3)
        ln = (r.uniform((K,), 0.5, 1.5), r.uniform((K,), -0.5, 0.5)) if has_ln else None
        wq = r.i8((K, N)) if wdt == np.int8 else r.u8((K, N))
        ws = r.uniform((), 0.001, 0.05) if scalar_scale else r.uniform((N,), 0.001, 0.05)
        bias = r.uniform((N,)) if has_bias else None
        M = int(np.prod(xs[:-1]))
        res = r.uniform(xs[:-1] + (N,)) if has_res else None
        wz = None
        if wzp == "vec":
            wz = r.i8((N,)) if wdt == np.int8 else r.u8((N,))
        elif wzp == "scalar":
            wz = np.array(r.i8((1,))[0] if wdt == np.int8 else r.u8((1,))[0])
        want = _qlinear_oracle(oracle, x, ln, wq, wz, ws, bias, res, act, 1e-5)
        dw = ctx.to_device(wq)
        op = rt.QuantizedLinear(act, 1e-5)
        pk = rt.MatMulInteger().prepack(ctx, 1, dw)
        dev = lambda a: None if a is None else ctx.to_device(a)
        got = op.run(ctx, dev(x), dw, dev(ws), packed_w=pk, w_zero_point=dev(wz), bias=dev(bias), residual=dev(res),
                     ln_scale=dev(ln[0]) if ln else None, ln_bias=dev(ln[1]) if ln else None).numpy()
        assert_bit_exact(got, want, f"QuantizedLinear x{xs} N={N} ln={has_ln} act={act} wzp={wzp} {np.dtype(wdt).name}")
        # host tensors / no prepack -> the composed operator chain: same bits
        got2 = op.run(ctx, x, wq, ws, w_zero_point=wz, bias=bias, residual=res, ln_scale=ln[0] if ln else None,
                      ln_bias=ln[1] if ln else None).numpy()
        assert_bit_exact(got2, want, f"QuantizedLinear (composed) x{xs} N={N}")
        n += 1
    return f"{n} cases bit-exact (fused kernel and composed chain)"


def _attention_ref(q, k, v, lens, mask, scale):
    """float64 reference of softmax(scale q k^T + mask) v over the first lens[b] positions."""
    B, qh, _, dh = q.shape
    kvh = k.shape[1]
    out = np.zeros((B, qh, 1, dh))
    for b in range(B):
        L = int(lens[b])
        for h in range(qh):
            hk = h // (qh // kvh)
            if L == 0:
                continue
            s = scale * (k[b, hk, :L].astype(np.float64) @ q[b, h, 0].astype(np.float64))
            if mask is not None:
                s = s + np.broadcast_to(mask, (B, qh, 1, k.shape[2]))[b, h, 0, :L]
            s = s - s.max()
            p = np.exp(s)
            out[b, h, 0] = (p / p.sum()) @ v[b, hk, :L].astype(np.float64)
    return out


def check_attention_decode(rt, oracle):
    """rten_b200_attention with q_seq = 1 against a float64 restatement of sdpa_head (src/ops/attention.rs:518-560) over an
    externally managed, right-padded cache (nonpad_kv_seqlen): natural and transposed value caches, grouped-query heads,
    additive masks, head sizes 64 / 128, cache lengths that split over several CTAs, the fused cache append, and the
    composed path for q_seq > 1.  f32 arithmetic: |d| <= 2e-5 * max |ref| (stated)."""
    ctx = new_ctx(rt, tf32=False)
    r = oracle.XorShiftRng(777)
    worst, n = 0.0, 0
    for B, qh, kvh, dh, cap, lens, use_mask, vt in [(3, 4, 4, 64, 200, [1, 77, 200], False, False), (8, 12, 12, 64, 576, [513] * 8, False, True),
                                                    (2, 8, 2, 64, 1000, [1000, 333], True, True), (2, 4, 4, 128, 96, [96, 5], True, False),
                                                    (1, 2, 1, 64, 5000, [4999], False, False), (2, 3, 3, 64, 64, [0, 64], False, True)]:
        q = r.uniform((B, qh, 1, dh))
        k = r.uniform((B, kvh, cap, dh))
        v = r.uniform((B, kvh, cap, dh))
        mask = r.uniform((B, 1, 1, cap), -2, 0) if use_mask else None
        lens_a = np.array(lens, np.int32)
        scale = 1.0 / np.sqrt(dh)
        ref = _attention_ref(q, k, v, lens_a, mask, scale)
        dk = ctx.to_device(k)
        if vt:  # value cache stored [.., dh, cap]; the operator sees the [.., cap, dh] view
            dvt = ctx.to_device(np.ascontiguousarray(v.transpose(0, 1, 3, 2)))
            dv = dvt.view((B, kvh, cap, dh), (kvh * dh * cap, dh * cap, 1, cap))
        else:
            dv = ctx.to_device(v)
        op = rt.Attention(is_causal=True, q_num_heads=qh, kv_num_heads=kvh)
        got = op.run(ctx, ctx.to_device(q), dk, dv, attn_mask=None if mask is None else ctx.to_device(mask),
                     nonpad_kv_seqlen=ctx.to_device(lens_a)).numpy()
        err = float(np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-30))
        assert got.shape == ref.shape and err <= 2e-5, f"Attention decode B={B} heads={qh}/{kvh} dh={dh} cap={cap} lens={lens}: rel err {err:.2e}"
        worst = max(worst, err)
        n += 1
    # fused cache append: the new key / value land at position len - 1 and take part in the attention
    B, nh, dh, cap = 4, 6, 64, 160
    lens_a = np.array([1, 50, 160, 97], np.int32)
    q, kn, vn = r.uniform((B, nh, 1, dh)), r.uniform((B, nh, 1, dh)), r.uniform((B, nh, 1, dh))
    k, v = r.uniform((B, nh, cap, dh)), r.uniform((B, nh, cap, dh))
    k2, v2 = k.copy(), v.copy()
    for b in range(B):
        k2[b, :, lens_a[b] - 1] = kn[b, :, 0]
        v2[b, :, lens_a[b] - 1] = vn[b, :, 0]
    ref = _attention_ref(q, k2, v2, lens_a, None, 0.125)
    for vt in (False, True):
        dk = ctx.to_device(k)
        if vt:
            dvt = ctx.to_device(np.ascontiguousarray(v.transpose(0, 1, 3, 2)))
            dv = dvt.view((B, nh, cap, dh), (nh * dh * cap, dh * cap, 1, cap))
        else:
            dv = ctx.to_device(v)
        got = rt.Attention(is_causal=True, scale=0.125).run(ctx, ctx.to_device(q), dk, dv, nonpad_kv_seqlen=ctx.to_device(lens_a),
                                                            new_key=ctx.to_device(kn), new_value=ctx.to_device(vn)).numpy()
        err = float(np.abs(got - ref).max() / np.abs(ref).max())
        assert err <= 2e-5, f"Attention with fused append (vt={vt}): rel err {err:.2e}"
        assert_bit_exact(dk.numpy(), k2, "key cache after the fused append")
        assert_bit_exact(dv.numpy(), v2, "value cache after the fused append")
        worst = max(worst, err)
    # q_seq > 1 (composed MatMul / Softmax / MatMul, 3xTF32): BERT-shaped, float mask
    q, k, v = r.uniform((2, 4, 32, 64)), r.uniform((2, 4, 48, 64)), r.uniform((2, 4, 48, 64))
    mask = r.uniform((2, 1, 1, 48), -2, 0)
    got = rt.Attention().run(ctx, q, k, v, attn_mask=mask).numpy()
    s = 0.125 * np.einsum("bhqd,bhkd->bhqk", q.astype(np.float64), k.astype(np.float64)) + mask
    p = np.exp(s - s.max(-1, keepdims=True))
    ref = np.einsum("bhqk,bhkd->bhqd", p / p.sum(-1, keepdims=True), v.astype(np.float64))
    err = float(np.abs(got - ref).max() / np.abs(ref).max())
    assert err <= 1e-4, f"Attention q_seq=32 (composed): rel err {err:.2e}"
    try:
        rt.Attention().run(ctx, r.uniform((2, 4, 1, 64)), r.uniform((2, 3, 9, 64)), r.uniform((2, 3, 9, 64)))
        raise AssertionError("expected an error")
    except rt.OpError as e:
        assert e.kind == "IncompatibleInputShapes" and e.msg == "q_num_heads must be a positive multiple of kv_num_heads", str(e)
    return f"{n + 2} decode cases, worst rel err {worst:.1e}; composed q_seq=32 rel err {err:.1e}"


def check_attention_encoder(rt, oracle):
    """rten_b200_attention on encoder shapes (128 keys, head size 64, q_seq a multiple of 128) in the single-pass TF32 mode:
    the one-kernel tcgen05 path (QK^T -> masked softmax -> PV inside the SM) against a float64 restatement of
    src/ops/attention.rs:645-905, for every value layout the kernel takes -- contiguous [B,nh,S,dh], strided views of a
    merged Q|K|V projection ([B,S,3H] memory, the layout BertRunner feeds it), and a transposed value tensor --
    with and without an additive [B,1,1,S] mask, output written through a strided [B,S,H] view.  TF32 operands
    (10-bit mantissas) in both products: |d| <= 4e-3 * max |ref| (stated); the composed 3xTF32 path must agree with the
    float64 reference within 1e-4 on the same inputs."""
    r = oracle.XorShiftRng(4242)
    worst = 0.0
    n = 0
    for B, nh, S, use_mask in [(3, 5, 128, True), (2, 12, 128, False), (2, 3, 256, True)]:
        dh, H = 64, nh * 64
        kv = 128
        qkv = r.uniform((B, max(S, kv), 3 * H), -1, 1)
        q = qkv[:, :S, 0:H].reshape(B, S, nh, dh).transpose(0, 2, 1, 3)
        k = qkv[:, :kv, H:2 * H].reshape(B, kv, nh, dh).transpose(0, 2, 1, 3)
        v = qkv[:, :kv, 2 * H:].reshape(B, kv, nh, dh).transpose(0, 2, 1, 3)
        mask = r.uniform((B, 1, 1, kv), -3, 0) if use_mask else None
        s = 0.125 * np.einsum("bhqd,bhkd->bhqk", q.astype(np.float64), k.astype(np.float64))
        if mask is not None:
            s = s + mask
        pr = np.exp(s - s.max(-1, keepdims=True))
        ref = np.einsum("bhqk,bhkd->bhqd", pr / pr.sum(-1, keepdims=True), v.astype(np.float64))
        for tf32 in (True, False):
            ctx = new_ctx(rt, tf32=tf32)
            dm = None if mask is None else ctx.to_device(mask)
            Sm = qkv.shape[1]
            dqkv = ctx.to_device(qkv)
            part = lambda i, rows: dqkv.view((B, nh, rows, dh), (Sm * 3 * H, dh, 3 * H, 1), i * H)
            layouts = {
                "merged qkv views": (part(0, S), part(1, kv), part(2, kv)),
                "contiguous": (ctx.to_device(np.ascontiguousarray(q)), ctx.to_device(np.ascontiguousarray(k)), ctx.to_device(np.ascontiguousarray(v))),
            }
            dvt = ctx.to_device(np.ascontiguousarray(v.transpose(0, 1, 3, 2)))
            layouts["transposed value"] = (layouts["contiguous"][0], layouts["contiguous"][1], dvt.view((B, nh, kv, dh), (nh * dh * kv, dh * kv, 1, kv)))
            for name, (dq, dk, dv) in layouts.items():
                att = ctx.empty((B, S, H))
                rt.Attention(scale=0.125).run(ctx, dq, dk, dv, attn_mask=dm, out=att.view((B, nh, S, dh), (S * H, dh, H, 1)))
                got = att.numpy().reshape(B, S, nh, dh).transpose(0, 2, 1, 3)
                err = float(np.abs(got - ref).max() / np.abs(ref).max())
                tol = 4e-3 if tf32 else 1e-4
                assert err <= tol, f"encoder Attention B={B} nh={nh} S={S} mask={use_mask} tf32={tf32} ({name}): rel err {err:.2e} > {tol}"
                if tf32:
                    worst = max(worst, err)
                n += 1
    return f"{n} cases (3 value layouts x 2 modes x 3 shapes), one-kernel TF32 path worst rel err {worst:.1e}"


def check_gelu_epilogue(rt, oracle):
    """The GEMM epilogue's Gelu (two lanes per packed f32x2 instruction, math.cuh gelu_ref_x2) must be BIT-IDENTICAL to
    the Gelu operator (the reference's scalar recipe, bit-exact against the oracle in check_unary) applied to the same
    product: FusedMatMul(bias, Gelu) vs FusedMatMul(bias) -> Gelu with the launch plan pinned (same accumulation order),
    for erf-Gelu and the tanh form, values spanning the exp cut-off, zeros and large magnitudes."""
    import os
    ctx = new_ctx(rt, tf32=True)
    r = oracle.XorShiftRng(2718)
    forced = {"RTEN_B200_FORCE_BN": "128", "RTEN_B200_FORCE_PAIR": "0", "RTEN_B200_FORCE_KATOMS": "1", "RTEN_B200_FORCE_SPLITK": "1", "RTEN_B200_FORCE_CTA2": "0"}
    os.environ.update(forced)
    try:
        n = 0
        for (m, k, nn), amp in [((384, 64, 256), 1.0), ((256, 128, 384), 6.0), ((128, 32, 128), 40.0)]:
            a = (r.uniform((m, k), -1, 1) * amp).astype(np.float32)
            a[:4] = 0.0  # rows of exact zeros: Gelu(bias) alone
            b = r.uniform((k, nn), -1, 1)
            bias = r.uniform((nn,), -1, 1)
            bias[:3] = 0.0
            da, db, dbias = ctx.to_device(a), ctx.to_device(b), ctx.to_device(bias)
            for act, approx in ((rt.ACT_GELU, False), (rt.ACT_GELU_TANH, True)):
                fused = rt.FusedMatMul(None, activation=act).run(ctx, da, db, dbias).numpy()
                plain = rt.FusedMatMul(None).run(ctx, da, db, dbias)
                two = rt.Gelu(approximate=approx).run(ctx, plain).numpy()
                assert_bit_exact(fused, two, f"Gelu epilogue (approximate={approx}) {m}x{k}x{nn} amp {amp}")
                n += 1
    finally:
        for kname in forced:
            os.environ.pop(kname, None)
    return f"{n} fused-vs-operator comparisons bit-identical"


def check_skinny_f32(rt, oracle):
    """MatMul / Gemm / FusedMatMul with M <= 32 rows run the HBM-streaming skinny kernel in exact f32 FMA arithmetic
    (rten-gemm's gemv path): the reference's float rule against the oracle, in BOTH f32 modes (the mode does not
    matter here), incl. the ResNet-50 classifier shape, bias, alpha, beta * C and the vector forms."""
    worst = 0
    for tf32 in (True, False):
        ctx = new_ctx(rt, tf32=tf32)
        r = oracle.XorShiftRng(31)
        for (m, k, n) in [(32, 2048, 1000), (8, 768, 3072), (1, 768, 50), (16, 3072, 768), (5, 100, 7), (31, 64, 33)]:
            a, b, bias = r.f32((m, k)), r.f32((k, n)), r.f32((n,))
            assert_reference_rule(rt.FusedMatMul(0.5).run(ctx, a, b, bias).numpy(), oracle.matmul(a, b, bias, 0.5), f"skinny FusedMatMul {m}x{k}x{n}")
            worst += 1
        a, b, c = r.f32((32, 2048)), r.f32((1000, 2048)), r.f32((1000,))
        assert_reference_rule(rt.Gemm(1.0, 1.0, False, True).run(ctx, a, b, c).numpy(), oracle.gemm_op(a, b, c, 1.0, 1.0, False, True), "skinny Gemm transB + C")
        v, mtx = r.f32((768,)), r.f32((768, 1000))
        assert_reference_rule(rt.MatMul().run(ctx, v, mtx).numpy(), oracle.matmul(v, mtx), "skinny vector x matrix")
    return f"{worst} cases inside 1e-8 + 1e-5*|ref| in both modes"


def check_halo_conv(rt, oracle):
    """Stride-1 windows on the halo-reuse kernel (one activation patch per channel block in shared memory, the filter taps
    as shifted matrix descriptors): ResNet-50's 3x3 layer shapes at several batch sizes (row strips, whole images, several
    images per unit, batch tails), 5x5 / 1x3 / 3x1 windows, asymmetric padding, both f32 modes; against float64 within the
    TF32 bound, and the generic implicit-GEMM kernel must agree within the same bound."""
    import os
    os.environ["RTEN_B200_HALO"] = "1"  # the kernel is opt-in (DESIGN.md 4.2)
    try:
        return _check_halo_conv(rt, oracle)
    finally:
        os.environ.pop("RTEN_B200_HALO", None)


def _check_halo_conv(rt, oracle):
    import os
    worst, n = 0.0, 0
    cases = [((2, 64, 56, 56), (64, 64, 3, 3), (1, 1, 1, 1)), ((3, 128, 28, 28), (128, 128, 3, 3), (1, 1, 1, 1)),
             ((5, 256, 14, 14), (256, 256, 3, 3), (1, 1, 1, 1)), ((7, 512, 7, 7), (512, 512, 3, 3), (1, 1, 1, 1)),
             ((2, 32, 20, 17), (96, 32, 5, 5), (2, 2, 2, 2)), ((2, 64, 9, 30), (32, 64, 1, 3), (0, 1, 0, 1)),
             ((1, 32, 30, 9), (64, 32, 3, 1), (1, 0, 1, 0)), ((2, 96, 12, 12), (160, 96, 3, 3), (0, 0, 0, 0)),
             ((2, 64, 16, 16), (64, 64, 3, 3), (2, 0, 0, 2)), ((33, 64, 8, 8), (32, 64, 3, 3), (1, 1, 1, 1))]
    for tf32 in (True, False):
        ctx = new_ctx(rt, tf32=tf32)
        global TF32_REL
        saved = TF32_REL
        TF32_REL = 2.0 ** -9 if tf32 else 2.0 ** -18
        try:
            for xs, ws, pads in cases:
                for act in (0, 1):
                    worst = max(worst, _conv_case(rt, oracle, ctx, xs, ws, pads=pads, cl=True, prepack=True, act=act))
                    n += 1
        finally:
            TF32_REL = saved
    # the two kernels on the same problem
    ctx = new_ctx(rt)
    r = oracle.XorShiftRng(17)
    x, w, b = r.uniform((4, 128, 28, 28)), r.uniform((128, 128, 3, 3)) / np.float32(34.0), r.uniform((128,))
    xd = ctx.to_device(x, channels_last=True)
    op = rt.Conv(1, (1, 1), (1, 1, 1, 1), (1, 1), activation=1)
    halo = op.run(ctx, xd, w, b).numpy()
    os.environ["RTEN_B200_NO_HALO"] = "1"
    try:
        generic = op.run(ctx, xd, w, b).numpy()
    finally:
        os.environ.pop("RTEN_B200_NO_HALO", None)
    exact, absum = _conv_exact(x, w, b, (1, 1, 1, 1), 1, (1, 1), (1, 1))
    assert_tf32_close(halo, np.maximum(exact, 0), absum, "halo kernel")
    assert_tf32_close(generic, np.maximum(exact, 0), absum, "generic kernel")
    return f"{n} cases, worst err/bound {worst:.3f}; halo vs generic max |d| {float(np.abs(halo - generic).max()):.2e}"


# ------------------------------------------------------------------------------------------
# ONNX reader + graph executor (rten_b200_model_*)
# ------------------------------------------------------------------------------------------
def _onnx_interpret(oracle, nodes, consts, feeds, want):
    """Test-side interpreter of the small ONNX graphs built below: every node through the CPU oracle's operator of the
    same name, unfused -- what rten's executor would compute."""
    vals = dict(consts)
    vals.update(feeds)
    f32 = np.float32
    for op, ins, outs, attrs in nodes:
        x = [vals[i] if i else None for i in ins]
        if op == "MatMul":
            y = oracle.matmul(x[0], x[1])
        elif op == "Add":
            y = oracle.add(x[0], x[1])
        elif op == "Mul":
            y = (x[0] * x[1]).astype(f32)
        elif op == "Softmax":
            y = oracle.softmax(x[0], attrs.get("axis", -1))
        elif op == "LayerNormalization":
            y = oracle.layer_norm(x[0], x[1], x[2] if len(x) > 2 else None, attrs.get("axis", -1), attrs.get("epsilon", 1e-5))
        elif op == "Gelu":
            y = oracle.gelu(x[0], attrs.get("approximate") == "tanh")
        elif op == "Erf":
            y = oracle.erf(x[0])
        elif op == "Relu":
            y = oracle.relu(x[0])
        elif op == "Reshape":
            shape = [int(x[0].shape[i]) if d == 0 else int(d) for i, d in enumerate(np.asarray(x[1]).reshape(-1))]
            y = np.ascontiguousarray(x[0]).reshape(shape)
        elif op == "Transpose":
            y = x[0].transpose(attrs["perm"])
        elif op == "Gather":
            y = x[0][x[1]]
        elif op == "DynamicQuantizeLinear":
            q, sc, zp = oracle.dynamic_quantize_linear(x[0])
            vals[outs[0]], vals[outs[1]], vals[outs[2]] = q, np.asarray(sc, f32).reshape(()), np.asarray(zp, np.uint8).reshape(())
            continue
        elif op == "MatMulInteger":
            y = oracle.matmul_integer(x[0], x[1], x[2] if len(x) > 2 else None, x[3] if len(x) > 3 else None)
        elif op == "Cast":
            y = x[0].astype(f32)
        else:
            raise AssertionError(f"interpreter: {op}")
        vals[outs[0]] = y
    return [vals[w] for w in want]


def _bert_layer_onnx(oracle, W, B, S, H, nh, ffn, seed):
    """One BERT encoder layer as an exporter writes it (opset 20: LayerNormalization and Gelu are single nodes): MatMul + Add
    for every linear layer, Reshape / Transpose head split, Mul by 1/sqrt(d), additive mask, Softmax."""
    r = oracle.XorShiftRng(seed)
    dh = H // nh
    lin = lambda i, o: ((r.uniform((i, o)) / np.float32(np.sqrt(i))).astype(np.float32), (r.uniform((o,)) * np.float32(0.1)).astype(np.float32))
    consts = {}
    for name, (i, o) in {"q": (H, H), "k": (H, H), "v": (H, H), "o": (H, H), "f1": (H, ffn), "f2": (ffn, H)}.items():
        consts["w" + name], consts["b" + name] = lin(i, o)
    for n in ("ln1", "ln2"):
        consts[n + "g"] = (1 + 0.1 * r.uniform((H,))).astype(np.float32)
        consts[n + "b"] = (0.1 * r.uniform((H,))).astype(np.float32)
    consts["shape_heads"] = np.array([0, 0, nh, dh], np.int64)
    consts["shape_merge"] = np.array([0, 0, H], np.int64)
    consts["scale"] = np.array(1.0 / np.sqrt(dh), np.float32)
    nodes = []
    N = lambda op, ins, outs, **a: nodes.append((op, ins, outs, a))
    for t in "qkv":
        N("MatMul", ["x", "w" + t], [t + "0"])
        N("Add", [t + "0", "b" + t], [t + "1"])
        N("Reshape", [t + "1", "shape_heads"], [t + "2"])
        N("Transpose", [t + "2"], [t + "h"], perm=[0, 2, 3, 1] if t == "k" else [0, 2, 1, 3])
    N("MatMul", ["qh", "kh"], ["s0"])
    N("Mul", ["s0", "scale"], ["s1"])
    N("Add", ["s1", "mask"], ["s2"])
    N("Softmax", ["s2"], ["p"], axis=-1)
    N("MatMul", ["p", "vh"], ["c0"])
    N("Transpose", ["c0"], ["c1"], perm=[0, 2, 1, 3])
    N("Reshape", ["c1", "shape_merge"], ["c2"])
    N("MatMul", ["c2", "wo"], ["a0"])
    N("Add", ["a0", "bo"], ["a1"])
    N("Add", ["a1", "x"], ["a2"])
    N("LayerNormalization", ["a2", "ln1g", "ln1b"], ["h"], axis=-1, epsilon=1e-12)
    N("MatMul", ["h", "wf1"], ["f0"])
    N("Add", ["f0", "bf1"], ["f1"])
    N("Gelu", ["f1"], ["f2"])
    N("MatMul", ["f2", "wf2"], ["g0"])
    N("Add", ["g0", "bf2"], ["g1"])
    N("Add", ["g1", "h"], ["g2"])
    N("LayerNormalization", ["g2", "ln2g", "ln2b"], ["out"], axis=-1, epsilon=1e-12)
    data = W.model([W.node(op, ins, outs, **a) for op, ins, outs, a in nodes], [W.tensor(k, v) for k, v in consts.items()],
                   [W.value_info("x", W.FLOAT, [B, S, H]), W.value_info("mask", W.FLOAT, [B, 1, 1, S])], [W.value_info("out", W.FLOAT, [B, S, H])], opset=20)
    return data, nodes, consts


def check_model_executor(rt, oracle):
    """rten_b200_model_load / _run: the ONNX reader and the native graph executor.  (1) The reference's MNIST test model
    (re-encoded from the golden fixture) gives the oracle's logits, with Conv + Relu fused at load and intermediate values
    requestable by name.  (2) A BERT encoder layer in exporter form (MatMul + Add, Reshape / Transpose views, Softmax,
    LayerNormalization, Gelu) matches the oracle interpreting the same graph, in both f32 modes.  (3) A dynamically
    quantised linear layer (DynamicQuantizeLinear -> MatMulInteger -> Cast -> Mul -> Add) is bit-exact.  (4) Error paths."""
    import os
    import onnx_writer as W
    from rten_b200 import graphs
    from rten_b200.model import Model
    import model_ref
    here = os.path.dirname(os.path.abspath(__file__))
    # ---- (1) MNIST
    data = W.mnist_from_fixture(os.path.join(here, "golden", "mnist.npz"))
    wts = graphs.load_mnist_weights(os.path.join(here, "golden", "mnist.npz"))
    x1 = np.full((1, 1, 28, 28), 0.5, np.float32)
    ref = model_ref.mnist_oracle(oracle, wts, x1)
    res = {}
    for tf32, tol in ((True, 1e-2), (False, 5e-5)):
        ctx = new_ctx(rt, tf32=tf32)
        m = Model(ctx, data)
        assert m.input_names == ["input"] and m.output_names == ["logits"]
        assert m.node_ops == ["Conv", "MaxPool", "Conv", "MaxPool", "Conv", "ReduceMean", "Reshape", "Gemm"], m.node_ops  # Relu fused
        for xin in (x1, ctx.to_device(x1)):  # host tensor staged by the executor, and a resident tensor
            (logits,) = m.run({"input": xin})
            got = logits.numpy()
            rel = float(np.abs(got - ref).max() / np.abs(ref).max())
            assert got.shape == ref.shape and rel <= tol, f"MNIST through the executor (tf32={tf32}): rel err {rel:.3e}"
        res[tf32] = rel
        # any value of the graph can be requested: the pooled activation after the first block, and the logits with it
        pooled, logits2 = m.run({"input": x1}, ["max_pool2d", "logits"])
        want = oracle.max_pool(oracle.relu(oracle.conv(x1, wts["conv1.weight"], wts["conv1.bias"], [1, 1, 1, 1], 1, (1, 1), (1, 1))), (2, 2), [0, 0, 0, 0], (2, 2))
        assert pooled.shape == want.shape and float(np.abs(pooled.numpy() - want).max()) <= (3e-2 if tf32 else 1e-4)
        assert_bit_exact(logits2.numpy(), got, "same logits when an intermediate is requested too")
        try:
            m.run({"input": np.zeros((2, 1, 28, 28), np.float32)})  # the model's Reshape is to [1, 64]
            raise AssertionError("expected a Reshape error")
        except rt.OpError as e:
            assert e.kind == "InvalidValue" and "total elements" in e.msg, str(e)
        (again,) = m.run({"input": x1})  # the failed run released everything it held
        assert_bit_exact(again.numpy(), got, "run after a failed run")
    # ---- (2) transformer layer
    B, S, H, nh, ffn = 2, 16, 64, 4, 128
    data, nodes, consts = _bert_layer_onnx(oracle, W, B, S, H, nh, ffn, 2024)
    r = oracle.XorShiftRng(9)
    x = r.uniform((B, S, H))
    mask = np.zeros((B, 1, 1, S), np.float32)
    mask[1, ..., 11:] = -10000.0
    (want,) = _onnx_interpret(oracle, nodes, consts, {"x": x, "mask": mask}, ["out"])
    errs = []
    for tf32, tol in ((True, 2e-2), (False, 2e-4)):
        ctx = new_ctx(rt, tf32=tf32)
        m = Model(ctx, data)
        assert m.node_ops.count("Add") == 3 and m.node_ops.count("MatMul") == 8, m.node_ops  # six MatMul + Add(bias) pairs fused, residual / mask adds kept
        (out,) = m.run({"x": ctx.to_device(x), "mask": mask})
        err = float(np.abs(out.numpy() - want).max())
        assert out.shape == want.shape and err <= tol, f"BERT layer through the executor (tf32={tf32}): max abs err {err:.3e}"
        errs.append(err)
    # ---- (3) dynamically quantised linear layer, unfused exporter form
    K, N = 96, 80
    wq, wz = r.i8((K, N)), r.i8((N,))
    ws, bias = r.uniform((N,), 0.001, 0.05), r.uniform((N,))
    qnodes = [("DynamicQuantizeLinear", ["x"], ["xq", "xs", "xz"], {}), ("MatMulInteger", ["xq", "w", "xz", "wz"], ["acc"], {}),
              ("Cast", ["acc"], ["accf"], {"to": 1}), ("Mul", ["xs", "ws"], ["sc"], {}), ("Mul", ["accf", "sc"], ["y0"], {}), ("Add", ["y0", "b"], ["y"], {})]
    qconsts = {"w": wq, "wz": wz, "ws": ws, "b": bias}
    qdata = W.model([W.node(op, ins, outs, **a) for op, ins, outs, a in qnodes], [W.tensor(k, v) for k, v in qconsts.items()],
                    [W.value_info("x", W.FLOAT, [5, K])], [W.value_info("y", W.FLOAT, [5, N])], opset=18)
    xq = r.uniform((5, K), -2, 3)
    (want_q,) = _onnx_interpret(oracle, qnodes, qconsts, {"x": xq}, ["y"])
    ctx = new_ctx(rt)
    (got_q,) = Model(ctx, qdata).run({"x": xq})
    assert_bit_exact(got_q.numpy(), want_q, "quantised linear layer through the executor")
    # ---- (4) errors
    bad = W.model([W.node("NonMaxSuppression", ["x"], ["y"])], [], [W.value_info("x", W.FLOAT, [1])], [W.value_info("y", W.FLOAT, [1])])
    try:
        Model(ctx, bad)
        raise AssertionError("expected an unsupported-operator error")
    except rt.OpError as e:
        assert e.kind == "UnsupportedValue" and e.msg == "unsupported operator NonMaxSuppression", str(e)
    m = Model(ctx, qdata)
    for kwargs, kind in (({"inputs": {"nope": xq}}, "InvalidValue"), ({"inputs": {}}, "MissingInputs"), ({"inputs": {"x": xq}, "outputs": ["zzz"]}, "InvalidValue")):
        try:
            m.run(**kwargs)
            raise AssertionError("expected an error")
        except rt.OpError as e:
            assert e.kind == kind, str(e)
    return f"MNIST rel err tf32 {res[True]:.1e} / 3xtf32 {res[False]:.1e}; BERT layer max abs err {errs[0]:.1e} / {errs[1]:.1e}; int8 layer bit-exact"


def check_generator(rt, oracle):
    """rten-generate's loop (generator.rs:481-1000) over the HBM-resident GPT-2: the model is driven ONLY through the
    Optimum names (input_ids / attention_mask / position_ids / past_key_values.N.* in, logits / present.N.* out), the
    present.* handles of one step are the past_key_values.* of the next, and the cache doubles its capacity when full
    (:878-884) -- here from 16 to 32 positions in the middle of the run, which also re-captures the decode graph.  Every
    step's logits are compared with the oracle decoding the same tokens (2e-2 of max |logit|, greedy token within it)."""
    from rten_b200 import graphs
    from rten_b200.generate import GPT2DecoderModel, Generator, TopKSampler
    import model_ref
    ctx = new_ctx(rt, tf32=False)
    rng = oracle.XorShiftRng(5678)
    spec = graphs.make_gpt2_int8(lambda s: rng.uniform(s), layers=3, vocab=5000, max_pos=128)
    B, T0, nsteps = 2, 12, 9
    prompt = (oracle.XorShiftRng(3).u64(B * T0) % 5000).astype(np.int32).reshape(B, T0)
    model = GPT2DecoderModel(ctx, spec, B, initial_capacity=16)
    gen = Generator.from_model(model).with_prompt(prompt)
    assert len(gen.kv_pairs) == 2 * 3 and gen.kv_cache_len() is None
    dec = None
    worst = 0.0
    caps = []
    for step in range(nsteps):
        tok = next(gen)
        if dec is None:
            dec = model_ref.gpt2_int8_decoder(oracle, spec, prompt)
            ref = dec.logits
        else:
            ref = dec.step(prev[:, None])
        rel = float(np.abs(gen.last_logits - ref).max() / np.abs(ref).max())
        assert gen.last_logits.shape == ref.shape and rel <= 2e-2, f"generator step {step}: rel err {rel:.3e}"
        assert_same_greedy_token(gen.last_logits, ref, 2e-2, f"generator step {step}")
        assert (tok == gen.last_logits.argmax(1)).all()
        worst = max(worst, rel)
        prev = tok  # teacher forcing: the oracle decodes the tokens the generator actually produced
        assert gen.kv_cache_len() == T0 + step
        caps.append(gen.kv_cache["past_key_values.0.key"].capacity)
    assert caps[0] == 16 and caps[-1] == 32, caps
    assert gen.prev_tokens().shape == (B, nsteps)
    # a seeded TopK sampler runs through the same loop
    g2 = Generator.from_model(GPT2DecoderModel(ctx, spec, B, initial_capacity=32)).with_prompt(prompt).with_sampler(TopKSampler(5, 0.8, seed=1))
    toks = [next(g2) for _ in range(3)]
    assert all(t.shape == (B,) for t in toks)
    return f"{nsteps} steps, cache capacity 16 -> 32, worst rel err {worst:.2e}"


ALL_CHECKS = [
    ("context", check_context), ("unary", check_unary), ("softmax", check_softmax), ("layer_norm", check_layer_norm),
    ("dql", check_dql), ("glue", check_glue), ("matmul_small", check_matmul_small), ("matmul_shapes", check_matmul_shapes),
    ("matmul_bert", check_matmul_bert), ("gemm_op", check_gemm_op), ("matmul_integer", check_matmul_integer),
    ("conv_basic", check_conv_basic), ("conv_stride", check_conv_stride), ("conv_more", check_conv_more),
    ("conv_integer", check_conv_integer), ("plans", check_plans), ("tf32x3", check_tf32x3), ("graph_replay", check_graph_replay), ("conv_integer_fused", check_conv_integer_fused),
    ("resnet50_int8_model", check_resnet50_int8_model), ("gpt2_int8_kvcache", check_gpt2_int8_kvcache), ("mnist_model", check_mnist_model), ("resnet50_model", check_resnet50_model), ("bert_model", check_bert_model),
    ("model_executor", check_model_executor), ("generator", check_generator), ("halo_conv", check_halo_conv), ("quantized_linear", check_quantized_linear), ("attention_decode", check_attention_decode), ("attention_encoder", check_attention_encoder), ("gelu_epilogue", check_gelu_epilogue), ("skinny_f32", check_skinny_f32),
    ("reference_rule_f32", check_reference_rule_f32), ("graph_pool_isolation", check_graph_pool_isolation),
    ("resnet50_b32_baseline", check_resnet50_b32_baseline), ("bert_b16_baseline", check_bert_b16_baseline),
    ("resnet50_int8_b64_baseline", check_resnet50_int8_b64_baseline), ("gpt2_b8_baseline", check_gpt2_b8_baseline),
]
