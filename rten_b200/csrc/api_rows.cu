// Operator entry points of the C ABI, row / elementwise operators (Softmax, LayerNormalization, Erf / Gelu / Relu, Add / Mul,
// DynamicQuantizeLinear, Gather / Scatter rows): shape / argument validation with the reference's error strings,
// operand normalisation (K-major, TMA-addressable), kernel dispatch.  Mirrors, per function, the
// reference operator named in include/rten_b200.h.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "api_shared.h"
#include "comm_device.cuh"
#include "api_util.h"
#include "rowops.h"
#include "skinny.h"
#include "umma_gemm.h"

using namespace rtb;
using namespace rtb::api;

extern "C" {

// ---- Softmax / AddSoftmax -------------------------------------------------------------------
rten_status rten_b200_softmax(rten_ctx* ctx, const rten_tensor* x, const rten_tensor* mask, int axis, int flush_nans,
                              rten_tensor* out) {
    RTB_TRY(check_ctx(ctx));
    if (!x || !out) return fail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
    if (x->dtype != RTEN_F32 || (mask && mask->dtype != RTEN_F32)) return fail(ctx, RTEN_ERR_UNSUPPORTED_TYPE, "unsupported type");
    const int nd = x->ndim;
    if (nd == 0 || axis < -nd || axis >= nd) return fail(ctx, RTEN_ERR_INVALID_VALUE, "Axis is invalid");
    const int ax = axis < 0 ? axis + nd : axis;
    OpScope sc(ctx);
    rten_tensor xv, mv, ov;
    rten_status st = sc.in(x, &xv);
    if (st == RTEN_OK && mask) st = sc.in(mask, &mv);
    if (st == RTEN_OK) st = sc.out(out, RTEN_F32, nd, xv.shape, &ov, nullptr);
    if (st == RTEN_OK && numel(&xv) > 0) {
        // view with `ax` moved last
        int perm[RTEN_MAX_DIMS], k = 0;
        for (int i = 0; i < nd; i++)
            if (i != ax) perm[k++] = i;
        perm[nd - 1] = ax;
        rten_tensor xp = xv, op = ov;
        for (int i = 0; i < nd; i++) {
            xp.shape[i] = xv.shape[perm[i]];
            xp.strides[i] = xv.strides[perm[i]];
            op.shape[i] = ov.shape[perm[i]];
            op.strides[i] = ov.strides[perm[i]];
        }
        rten_tensor xc;
        st = sc.contiguous(&xp, &xc);
        // run in place on the output when it is lane-contiguous in the permuted view, else via temp
        rten_tensor yc = op;
        const bool out_direct = is_contiguous(&op);
        if (st == RTEN_OK && !out_direct) {
            set_contiguous(&yc);
            void* t = nullptr;
            st = temp_alloc(ctx, (size_t)numel(&xv) * 4, &t);
            yc.data = t;
        }
        if (st == RTEN_OK) {
            const int n = (int)xp.shape[nd - 1];
            const long long rows = numel(&xv) / n;
            const float* mp = nullptr;
            long long lead[4] = {1, 1, 1, 1}, ms[4] = {0, 0, 0, 0}, ms_last = 0;
            int nlead = 0;
            if (mask) {
                // broadcast mask to x's shape (numpy rules), in the permuted dim order
                if (mv.ndim > nd) {
                    st = fail(ctx, RTEN_ERR_INCOMPATIBLE_SHAPES, "Cannot broadcast inputs");
                } else {
                    long long mstr[RTEN_MAX_DIMS];
                    for (int i = 0; i < nd && st == RTEN_OK; i++) {
                        const int mi = i - (nd - mv.ndim);
                        if (mi < 0 || mv.shape[mi] == 1)
                            mstr[i] = 0;
                        else if (mv.shape[mi] == xv.shape[i])
                            mstr[i] = mv.strides[mi];
                        else
                            st = fail(ctx, RTEN_ERR_INCOMPATIBLE_SHAPES, "Cannot broadcast inputs");
                    }
                    if (st == RTEN_OK) {
                        // leading dims in permuted order, collapsed where the mask advances uniformly
                        std::vector<long long> ls, lst;
                        for (int i = 0; i < nd - 1; i++) {
                            const long long s = xp.shape[i], stv = mstr[perm[i]];
                            if (s == 1) continue;
                            if (!ls.empty() && lst.back() == stv * s) {
                                ls.back() *= s;
                                lst.back() = stv;
                            } else {
                                ls.push_back(s);
                                lst.push_back(stv);
                            }
                        }
                        if (ls.size() > 4) {
                            st = fail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "mask broadcast pattern needs more than 4 strided dims");
                        } else {
                            nlead = (int)ls.size();
                            for (int i = 0; i < nlead; i++) {
                                lead[i] = ls[i];
                                ms[i] = lst[i];
                            }
                            ms_last = mstr[ax];
                            mp = (const float*)mv.data;
                        }
                    }
                }
            }
            if (st == RTEN_OK)
                st = launch_softmax(ctx, (const float*)xc.data, (float*)yc.data, rows, n, flush_nans, mp, nlead, lead, ms,
                                    ms_last);
            if (st == RTEN_OK && !out_direct) {
                long long shape[RTEN_MAX_DIMS], ss[RTEN_MAX_DIMS], ds[RTEN_MAX_DIMS];
                for (int i = 0; i < nd; i++) {
                    shape[i] = yc.shape[i];
                    ss[i] = yc.strides[i];
                    ds[i] = op.strides[i];
                }
                st = launch_nd_copy(ctx, 4, yc.data, op.data, nd, shape, ss, ds);
            }
        }
    }
    return sc.finish(st);
}

// ---- LayerNormalization -------------------------------------------------------------------------
rten_status rten_b200_layer_norm(rten_ctx* ctx, const rten_tensor* x, const rten_tensor* scale, const rten_tensor* bias,
                                 int axis, float epsilon, rten_tensor* out) {
    RTB_TRY(check_ctx(ctx));
    if (!x || !scale || !out) return fail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
    if (x->dtype != RTEN_F32 || scale->dtype != RTEN_F32 || (bias && bias->dtype != RTEN_F32))
        return fail(ctx, RTEN_ERR_UNSUPPORTED_TYPE, "unsupported type");
    const int nd = x->ndim;
    if (axis < -nd || axis >= std::max(nd, 1)) return fail(ctx, RTEN_ERR_INVALID_VALUE, "Axis is invalid");
    const int ax = axis < 0 ? axis + nd : axis;
    const float eps = epsilon < 0.0f ? 1e-5f : epsilon;
    OpScope sc(ctx);
    rten_tensor xv, xc, sv, bv, ov;
    rten_status st = sc.in(x, &xv);
    if (st == RTEN_OK) st = sc.in(scale, &sv);
    if (st == RTEN_OK && bias) st = sc.in(bias, &bv);
    const int nn = nd - ax;  // normalized dims
    // broadcast a parameter to the normalized shape, materialised contiguous; scalars stay scalar
    auto param = [&](const rten_tensor& pv, const char* err, const float** ptr, float* scalar, bool* is_scalar) -> rten_status {
        if (numel(&pv) == 1) {
            // scale.item(): read on device later -> use a 1-element broadcast with stride 0
            *is_scalar = true;
            *ptr = (const float*)pv.data;
            (void)scalar;
            return RTEN_OK;
        }
        *is_scalar = false;
        if (pv.ndim > nn) return fail(ctx, RTEN_ERR_INVALID_VALUE, err);
        rten_tensor b = pv;
        b.ndim = nn;
        for (int i = 0; i < nn; i++) {
            const int pi = i - (nn - pv.ndim);
            const int64_t want = xv.shape[ax + i];
            b.shape[i] = want;
            if (pi < 0 || pv.shape[pi] == 1)
                b.strides[i] = 0;
            else if (pv.shape[pi] == want)
                b.strides[i] = pv.strides[pi];
            else
                return fail(ctx, RTEN_ERR_INVALID_VALUE, err);
        }
        rten_tensor c;
        RTB_TRY(sc.contiguous(&b, &c));
        *ptr = (const float*)c.data;
        return RTEN_OK;
    };
    const float *gp = nullptr, *bp = nullptr;
    float gs = 1.0f, bs = 0.0f;
    bool g_scalar = false, b_scalar = false;
    if (st == RTEN_OK) st = param(sv, "`scale` is not broadcastable to normalized axes of input", &gp, &gs, &g_scalar);
    if (st == RTEN_OK && bias) st = param(bv, "`bias` is not broadcastable to normalized axes of input", &bp, &bs, &b_scalar);
    if (st == RTEN_OK) st = sc.contiguous(&xv, &xc);
    if (st == RTEN_OK) st = sc.out(out, RTEN_F32, nd, xv.shape, &ov, nullptr);
    if (st == RTEN_OK && numel(&xv) > 0) {
        long long n = 1;
        for (int i = ax; i < nd; i++) n *= xv.shape[i];
        const long long rows = numel(&xv) / n;
        // scalar gamma / beta stay on the device and are read by the kernel (the reference's scalar-scale arm computes
        // rstd = scale / sqrt(var + eps), src/ops/norm.rs:456-529): no host read, no synchronisation, capturable
        const float *gsp = nullptr, *bsp = nullptr;
        if (g_scalar) {
            gsp = gp;
            gp = nullptr;
        }
        if (bias && b_scalar) {
            bsp = bp;
            bp = nullptr;
        }
        rten_tensor yc = ov;
        const bool direct = is_contiguous(&ov);
        if (!direct) {
            set_contiguous(&yc);
            void* t = nullptr;
            st = temp_alloc(ctx, (size_t)numel(&xv) * 4, &t);
            yc.data = t;
        }
        if (st == RTEN_OK)
            st = launch_layer_norm(ctx, (const float*)xc.data, (float*)yc.data, rows, (int)n, gp, gs, bp, bs, eps, gsp, bsp);
        if (st == RTEN_OK && !direct) {
            long long shape[RTEN_MAX_DIMS], ss[RTEN_MAX_DIMS], ds[RTEN_MAX_DIMS];
            for (int i = 0; i < nd; i++) {
                shape[i] = yc.shape[i];
                ss[i] = yc.strides[i];
                ds[i] = ov.strides[i];
            }
            st = launch_nd_copy(ctx, 4, yc.data, ov.data, nd, shape, ss, ds);
        }
    }
    return sc.finish(st);
}

// ---- unary elementwise ----------------------------------------------------------------------------
static rten_status unary_op(rten_ctx* ctx, int op, const rten_tensor* x, rten_tensor* out) {
    RTB_TRY(check_ctx(ctx));
    if (!x || !out) return fail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
    if (x->dtype != RTEN_F32) return fail(ctx, RTEN_ERR_UNSUPPORTED_TYPE, "unsupported type");
    OpScope sc(ctx);
    rten_tensor xv, ov;
    rten_status st = sc.in(x, &xv);
    // dense (any dim order) tensors are processed in memory order: output takes the input's strides
    bool dense = false;
    if (st == RTEN_OK) dense = span_elems(&xv) == numel(&xv);
    if (st == RTEN_OK) st = sc.out(out, RTEN_F32, xv.ndim, xv.shape, &ov, (out->data == nullptr && dense) ? xv.strides : nullptr);
    if (st == RTEN_OK && numel(&xv) > 0) {
        bool same_layout = dense;
        for (int i = 0; i < xv.ndim && same_layout; i++)
            if (xv.shape[i] != 1 && xv.strides[i] != ov.strides[i]) same_layout = false;
        if (same_layout) {
            st = launch_unary(ctx, op, (const float*)xv.data, (float*)ov.data, numel(&xv));
        } else {
            rten_tensor xc;
            st = sc.contiguous(&xv, &xc);
            if (st == RTEN_OK && is_contiguous(&ov)) {
                st = launch_unary(ctx, op, (const float*)xc.data, (float*)ov.data, numel(&xv));
            } else if (st == RTEN_OK) {
                void* t = nullptr;
                st = temp_alloc(ctx, (size_t)numel(&xv) * 4, &t);
                if (st == RTEN_OK) st = launch_unary(ctx, op, (const float*)xc.data, (float*)t, numel(&xv));
                if (st == RTEN_OK) {
                    long long shape[RTEN_MAX_DIMS], ss[RTEN_MAX_DIMS], ds[RTEN_MAX_DIMS];
                    for (int i = 0; i < xv.ndim; i++) {
                        shape[i] = xc.shape[i];
                        ss[i] = xc.strides[i];
                        ds[i] = ov.strides[i];
                    }
                    st = launch_nd_copy(ctx, 4, t, ov.data, xv.ndim, shape, ss, ds);
                }
            }
        }
    }
    return sc.finish(st);
}

rten_status rten_b200_erf(rten_ctx* ctx, const rten_tensor* x, rten_tensor* out) { return unary_op(ctx, UNARY_ERF, x, out); }
rten_status rten_b200_gelu(rten_ctx* ctx, const rten_tensor* x, int approximate, rten_tensor* out) {
    return unary_op(ctx, approximate ? UNARY_APPROX_GELU : UNARY_GELU, x, out);
}
rten_status rten_b200_relu(rten_ctx* ctx, const rten_tensor* x, rten_tensor* out) { return unary_op(ctx, UNARY_RELU, x, out); }

// ---- Add ----------------------------------------------------------------------------------------------
// Add / Mul with numpy broadcasting (src/ops/binary_elementwise.rs); flags: 0 = Add, 2 = Mul
static rten_status binary_f32(rten_ctx* ctx, const rten_tensor* a, const rten_tensor* b, rten_tensor* out, int flags) {
    RTB_TRY(check_ctx(ctx));
    if (!a || !b || !out) return fail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
    if (a->dtype != RTEN_F32 || b->dtype != RTEN_F32) return fail(ctx, RTEN_ERR_UNSUPPORTED_TYPE, "unsupported type");
    OpScope sc(ctx);
    rten_tensor av, bv, ov;
    rten_status st = sc.in(a, &av);
    if (st == RTEN_OK) st = sc.in(b, &bv);
    int nd = std::max(a->ndim, b->ndim);
    int64_t shape[RTEN_MAX_DIMS];
    long long sa[RTEN_MAX_DIMS], sb[RTEN_MAX_DIMS];
    for (int i = 0; i < nd && st == RTEN_OK; i++) {
        const int ia = i - (nd - av.ndim), ib = i - (nd - bv.ndim);
        const int64_t da = ia >= 0 ? av.shape[ia] : 1, db = ib >= 0 ? bv.shape[ib] : 1;
        if (da != db && da != 1 && db != 1) st = fail(ctx, RTEN_ERR_INCOMPATIBLE_SHAPES, "Cannot broadcast inputs");
        shape[i] = (da == 0 || db == 0) ? 0 : std::max(da, db);
        sa[i] = (ia >= 0 && da != 1) ? av.strides[ia] : 0;
        sb[i] = (ib >= 0 && db != 1) ? bv.strides[ib] : 0;
    }
    // same-shape dense operands: keep a's layout for the output
    bool same = st == RTEN_OK && av.ndim == bv.ndim && span_elems(&av) == numel(&av);
    for (int i = 0; i < nd && same; i++)
        if (av.shape[i] != bv.shape[i] || (av.shape[i] != 1 && av.strides[i] != bv.strides[i])) same = false;
    if (st == RTEN_OK) st = sc.out(out, RTEN_F32, nd, shape, &ov, (out->data == nullptr && same) ? av.strides : nullptr);
    if (st == RTEN_OK && numel(&ov) > 0) {
        bool flat = same;
        for (int i = 0; i < nd && flat; i++)
            if (ov.shape[i] != 1 && ov.strides[i] != av.strides[i]) flat = false;
        if (flat) {
            st = launch_add_flat(ctx, (const float*)av.data, (const float*)bv.data, (float*)ov.data, numel(&ov), flags);
        } else {
            long long shp[RTEN_MAX_DIMS], sd[RTEN_MAX_DIMS];
            for (int i = 0; i < nd; i++) {
                shp[i] = shape[i];
                sd[i] = ov.strides[i];
            }
            st = launch_nd_add(ctx, (const float*)av.data, (const float*)bv.data, (float*)ov.data, nd, shp, sa, sb, sd, flags);
        }
    }
    return sc.finish(st);
}

rten_status rten_b200_add(rten_ctx* ctx, const rten_tensor* a, const rten_tensor* b, rten_tensor* out) {
    return binary_f32(ctx, a, b, out, 0);
}
rten_status rten_b200_mul(rten_ctx* ctx, const rten_tensor* a, const rten_tensor* b, rten_tensor* out) {
    return binary_f32(ctx, a, b, out, 2);
}

// ---- DynamicQuantizeLinear ---------------------------------------------------------------------------
rten_status rten_b200_range_reset(rten_ctx* ctx, rten_tensor* ranges) {
    RTB_TRY(check_ctx(ctx));
    if (!ranges) return fail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
    if (ranges->dtype != RTEN_I32 || ranges->device < 0 || !is_contiguous(ranges) || numel(ranges) % 2)
        return fail(ctx, RTEN_ERR_INVALID_VALUE, "ranges must be a contiguous device-resident i32[n, 2]");
    cudaSetDevice(ctx->device);
    return launch_range_reset(ctx, (int*)ranges->data, (int)(numel(ranges) / 2));
}

rten_status rten_b200_dynamic_quantize_linear(rten_ctx* ctx, const rten_tensor* x, rten_tensor* y, rten_tensor* scale,
                                              rten_tensor* zero_point, void* nccl_comm) {
    return rten_b200_dynamic_quantize_linear_ranged(ctx, x, nullptr, y, scale, zero_point, nccl_comm);
}

rten_status rten_b200_dynamic_quantize_linear_ranged(rten_ctx* ctx, const rten_tensor* x, const rten_tensor* range,
                                                     rten_tensor* y, rten_tensor* scale, rten_tensor* zero_point,
                                                     void* nccl_comm) {
    RTB_TRY(check_ctx(ctx));
    if (!x || !y || !scale || !zero_point) return fail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
    if (x->dtype != RTEN_F32) return fail(ctx, RTEN_ERR_UNSUPPORTED_TYPE, "unsupported type");
    if (range && (range->dtype != RTEN_I32 || numel(range) != 2 || range->device < 0 || !is_contiguous(range)))
        return fail(ctx, RTEN_ERR_INVALID_VALUE, "the range must be a device-resident i32[2]");
    OpScope sc(ctx);
    rten_tensor xv, xc, yv, sv, zv;
    rten_status st = sc.in(x, &xv);
    // The op is elementwise plus an order-independent min / max: a DENSE input in any dim order (e.g. channels-last
    // activations) is processed in memory order and the quantised output keeps the input's strides.
    bool dense = st == RTEN_OK && span_elems(&xv) == numel(&xv) && y->data == nullptr;
    for (int i = 0; i < xv.ndim && dense; i++)
        if (xv.strides[i] <= 0 && xv.shape[i] > 1) dense = false;
    const bool x_cl_dense = st == RTEN_OK && xv.ndim == 4 && xv.strides[1] == 1 && xv.strides[3] == xv.shape[1] &&
                            xv.strides[2] == xv.shape[3] * xv.shape[1] && xv.strides[0] == xv.shape[2] * xv.shape[3] * xv.shape[1];
    if (dense || (x_cl_dense && y->data && y->ndim == 4 && y->strides[1] == 1)) {
        xc = xv;
    } else if (st == RTEN_OK) {
        st = sc.contiguous(&xv, &xc);
    }
    // A caller-provided channels-last output whose rows (b, h) sit at arbitrary pitches -- the interior of a spatially
    // pre-padded buffer, so that the consuming ConvInteger needs no padded copy -- is written row by row.
    bool rows_out = false;
    if (st == RTEN_OK && y->data && xv.ndim == 4 && y->ndim == 4 && y->device >= 0) {
        const int64_t Cc = xv.shape[1], Hh = xv.shape[2], Ww = xv.shape[3];
        rows_out = xv.strides[1] == 1 && xv.strides[3] == Cc && xv.strides[2] == Ww * Cc && xv.strides[0] == Hh * Ww * Cc &&
                   y->strides[1] == 1 && y->strides[3] == Cc && !is_contiguous(y) &&
                   !(y->strides[2] == Ww * Cc && y->strides[0] == Hh * Ww * Cc);
        if (rows_out) xc = xv;
    }
    if (st == RTEN_OK) st = sc.out(y, RTEN_U8, xv.ndim, xv.shape, &yv, dense ? xv.strides : nullptr);
    if (st == RTEN_OK) st = sc.out(scale, RTEN_F32, 0, nullptr, &sv, nullptr);
    if (st == RTEN_OK) st = sc.out(zero_point, RTEN_U8, 0, nullptr, &zv, nullptr);
    if (st == RTEN_OK && !dense && !rows_out && !is_contiguous(&yv)) st = fail(ctx, RTEN_ERR_UNSUPPORTED_OUTPUT, "quantized output must be contiguous");
    if (st == RTEN_OK) {
        const long long n = numel(&xv);
        if (n == 0) {
            // quantize.rs:378-386: scale 1, zero point 0
            const float one = 1.0f;
            RTB_CUDA(ctx, cudaMemcpyAsync(sv.data, &one, 4, cudaMemcpyHostToDevice, ctx->stream));
            RTB_CUDA(ctx, cudaMemsetAsync(zv.data, 0, 1, ctx->stream));
        } else if (!nccl_comm && !range && !rows_out && n <= 16384) {
            st = launch_dql_small(ctx, (const float*)xc.data, (uint8_t*)yv.data, (int)n, (float*)sv.data, (uint8_t*)zv.data);
        } else {
            // `range`: the producer of x already accumulated (min, max) in its epilogue -- no pass over x for it
            int* mm = range ? (int*)range->data : nullptr;
            if (!mm) {
                st = temp_alloc(ctx, 8, (void**)&mm);
                if (st == RTEN_OK) st = launch_minmax(ctx, (const float*)xc.data, n, mm);
            }
            // batch-sharded run: the range is the range of the whole (unsharded) tensor -- exchanged over NVLink peer
            // mailboxes by the quantise kernel's own prologue, or by two ncclAllReduce calls in front of it
            RangeExchange xch;
            const bool fused_xch = nccl_comm && comm_range_exchange(reinterpret_cast<rten_comm*>(nccl_comm), &xch);
            if (st == RTEN_OK && nccl_comm && !fused_xch) st = comm_allreduce_minmax(ctx, reinterpret_cast<rten_comm*>(nccl_comm), mm);
            if (st == RTEN_OK && rows_out)
                st = launch_dql_quantize_rows(ctx, (const float*)xc.data, (uint8_t*)yv.data, xv.shape[0] * xv.shape[2],
                                              (int)(xv.shape[3] * xv.shape[1]), (int)xv.shape[2], yv.strides[2], yv.strides[0], mm,
                                              (float*)sv.data, (uint8_t*)zv.data, fused_xch ? &xch : nullptr);
            else if (st == RTEN_OK)
                st = launch_dql_quantize(ctx, (const float*)xc.data, (uint8_t*)yv.data, n, mm, (float*)sv.data, (uint8_t*)zv.data,
                                         fused_xch ? &xch : nullptr);
        }
    }
    return sc.finish(st);
}

// ---- gather / scatter ------------------------------------------------------------------------------
rten_status rten_b200_gather_rows(rten_ctx* ctx, const rten_tensor* table, const rten_tensor* idx, rten_tensor* out) {
    RTB_TRY(check_ctx(ctx));
    if (!table || !idx || !out) return fail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
    if (table->dtype != RTEN_F32 || idx->dtype != RTEN_I32) return fail(ctx, RTEN_ERR_UNSUPPORTED_TYPE, "unsupported type");
    if (table->ndim != 2) return fail(ctx, RTEN_ERR_INVALID_VALUE, "gather_rows expects a 2-D table");
    OpScope sc(ctx);
    rten_tensor tv, iv, ic, ov;
    rten_status st = sc.in(table, &tv);
    if (st == RTEN_OK) st = sc.in(idx, &iv);
    if (st == RTEN_OK) st = sc.contiguous(&iv, &ic);
    if (st == RTEN_OK) {
        int64_t oshape[RTEN_MAX_DIMS];
        if (iv.ndim + 1 > RTEN_MAX_DIMS) return sc.finish(fail(ctx, RTEN_ERR_INVALID_VALUE, "tensor rank out of range"));
        for (int i = 0; i < iv.ndim; i++) oshape[i] = iv.shape[i];
        oshape[iv.ndim] = tv.shape[1];
        st = sc.out(out, RTEN_F32, iv.ndim + 1, oshape, &ov, nullptr);
        if (st == RTEN_OK && !is_contiguous(&ov)) st = fail(ctx, RTEN_ERR_UNSUPPORTED_OUTPUT, "gather output must be contiguous");
        if (st == RTEN_OK)
            st = launch_gather_rows(ctx, (const float*)tv.data, (const int*)ic.data, (float*)ov.data, numel(&iv),
                                    (int)tv.shape[1], tv.strides[0], tv.strides[1], tv.shape[0]);
    }
    return sc.finish(st);
}

rten_status rten_b200_scatter_rows(rten_ctx* ctx, rten_tensor* table, const rten_tensor* idx, const rten_tensor* src) {
    RTB_TRY(check_ctx(ctx));
    if (!table || !idx || !src) return fail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
    if (table->dtype != RTEN_F32 || src->dtype != RTEN_F32 || idx->dtype != RTEN_I32)
        return fail(ctx, RTEN_ERR_UNSUPPORTED_TYPE, "unsupported type");
    if (table->ndim != 2 || src->ndim != 2 || idx->ndim != 1) return fail(ctx, RTEN_ERR_INVALID_VALUE, "scatter_rows expects 2-D table / updates and 1-D indices");
    if (src->shape[0] != idx->shape[0] || src->shape[1] != table->shape[1])
        return fail(ctx, RTEN_ERR_INCOMPATIBLE_SHAPES, "updates do not match the indices / table width");
    if (table->device < 0) return fail(ctx, RTEN_ERR_UNSUPPORTED_OUTPUT, "the table must be device resident (updated in place)");
    OpScope sc(ctx);
    rten_tensor iv, ic, sv;
    rten_status st = sc.in(idx, &iv);
    if (st == RTEN_OK) st = sc.contiguous(&iv, &ic);
    if (st == RTEN_OK) st = sc.in(src, &sv);
    if (st == RTEN_OK)
        st = launch_scatter_rows(ctx, (float*)table->data, (const int*)ic.data, (const float*)sv.data, iv.shape[0],
                                 (int)table->shape[1], table->strides[0], table->strides[1], sv.strides[0], sv.strides[1],
                                 table->shape[0]);
    return sc.finish(st);
}

}  // extern "C"
