// Operator entry points of the C ABI, MatMul family (Gemm, MatMul / FusedMatMul, MatMulInteger(ToFloat), prepack):
// shape / argument validation with the reference's error strings,
// operand normalisation (K-major, TMA-addressable), kernel dispatch.  Mirrors, per function, the
// reference operator named in include/rten_b200.h.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "api_shared.h"
#include "api_util.h"
#include "rowops.h"
#include "skinny.h"
#include "umma_gemm.h"

using namespace rtb;
using namespace rtb::api;

namespace {

// ---------------------------------------------------------------------------------------
// K-major 2-level operand: rows x K with element strides.  Packs into an aligned workspace when
// TMA cannot address the original (k stride != 1, misaligned base / pitch).
// ---------------------------------------------------------------------------------------
struct Mat {
    const void* base;
    int64_t rows, K;
    int64_t rs, ks;       // element strides
    int64_t z0 = 1, z1 = 1;  // batch dims (z0 inner)
    int64_t zs0 = 0, zs1 = 0;
};

rten_status to_kmajor(rten_ctx* ctx, int esize, const Mat& m, OperandDesc* od) {
    OperandDesc d;
    d.base = m.base;
    d.dims[0] = m.K;
    d.dims[1] = m.rows;
    // broadcast batch dims (stride 0) become size-1 dims: the kernel then always passes coordinate 0
    d.dims[2] = (m.z0 > 1 && m.zs0 != 0) ? m.z0 : 1;
    d.dims[3] = (m.z1 > 1 && m.zs1 != 0) ? m.z1 : 1;
    d.strides[0] = m.ks;
    d.strides[1] = m.rs;
    d.strides[2] = d.dims[2] > 1 ? m.zs0 : 0;
    d.strides[3] = d.dims[3] > 1 ? m.zs1 : 0;
    if (m.K == 1) d.strides[0] = 1;  // a single k element is trivially contiguous
    if (tma_compatible(d, esize, 4)) {
        *od = d;
        return RTEN_OK;
    }
    // pack: [z1', z0', rows, Kpad]; broadcast batch dims (stride 0) are NOT expanded
    const int64_t kpad = round_up(m.K, 16 / esize);
    const int64_t e0 = (m.z0 > 1 && m.zs0 == 0) ? 1 : m.z0;
    const int64_t e1 = (m.z1 > 1 && m.zs1 == 0) ? 1 : m.z1;
    void* buf = nullptr;
    RTB_TRY(temp_alloc(ctx, (size_t)(e1 * e0 * m.rows * kpad) * esize, &buf));
    long long shape[4] = {e1, e0, m.rows, m.K};
    long long ss[4] = {m.zs1, m.zs0, m.rs, m.ks};
    long long ds[4] = {e0 * m.rows * kpad, m.rows * kpad, kpad, 1};
    RTB_TRY(launch_nd_copy(ctx, esize, m.base, buf, 4, shape, ss, ds));
    d.base = buf;
    d.dims[2] = e0;
    d.dims[3] = e1;
    d.strides[0] = 1;
    d.strides[1] = kpad;
    d.strides[2] = e0 > 1 ? m.rows * kpad : 0;
    d.strides[3] = e1 > 1 ? e0 * m.rows * kpad : 0;
    *od = d;
    return RTEN_OK;
}

// Collapse broadcast prefix dims of a matmul into at most 2 batch dims (z0 inner, z1 outer).  Dims are merged
// only when A, B and the output all advance uniformly across them.
struct BatchDims {
    int64_t z0 = 1, z1 = 1;
    int64_t a0 = 0, a1 = 0, b0 = 0, b1 = 0, o0 = 0, o1 = 0;
    bool ok = true;
};

BatchDims collapse_batch(const std::vector<int64_t>& size, const std::vector<int64_t>& as, const std::vector<int64_t>& bs,
                         const std::vector<int64_t>& os) {
    std::vector<int64_t> s, a, b, o;
    for (size_t i = 0; i < size.size(); i++) {
        if (size[i] == 1) continue;
        if (!s.empty() && a.back() == as[i] * size[i] && b.back() == bs[i] * size[i] && o.back() == os[i] * size[i]) {
            s.back() *= size[i];
            a.back() = as[i];
            b.back() = bs[i];
            o.back() = os[i];
            continue;
        }
        s.push_back(size[i]);
        a.push_back(as[i]);
        b.push_back(bs[i]);
        o.push_back(os[i]);
    }
    BatchDims r;
    if (s.size() > 2) {
        r.ok = false;
        return r;
    }
    if (s.size() == 1) {
        r.z0 = s[0];
        r.a0 = a[0];
        r.b0 = b[0];
        r.o0 = o[0];
    } else if (s.size() == 2) {
        r.z1 = s[0];
        r.a1 = a[0];
        r.b1 = b[0];
        r.o1 = o[0];
        r.z0 = s[1];
        r.a0 = a[1];
        r.b0 = b[1];
        r.o0 = o[1];
    }
    return r;
}

struct MatMulArgs {
    int kind;  // 0 f32, 1 int8
    const rten_tensor* a;
    const rten_tensor* b;
    const rten_packed* pb;
    EpilogueDesc epi;  // d / strides filled by matmul_core
    int out_dtype;
    // int8 extras
    const rten_tensor* a_zp = nullptr;
    const rten_tensor* b_zp = nullptr;
    // residual (same shape as out) for matmul_ex
    const rten_tensor* residual = nullptr;
};

// numpy-matmul shape logic of src/ops/matmul.rs:208-385 + kernel dispatch
rten_status matmul_core(OpScope& sc, MatMulArgs& A, rten_tensor* out) {
    rten_ctx* ctx = sc.ctx;
    rten_tensor a = *A.a, b = *A.b;
    if (a.ndim < 1 || b.ndim < 1) return fail(ctx, RTEN_ERR_INVALID_VALUE, "Inputs must have >= 1 dimensions");
    const bool a_vec = a.ndim == 1, b_vec = b.ndim == 1;
    if (a_vec) {  // [K] -> [1, K]
        a.ndim = 2;
        a.shape[1] = a.shape[0];
        a.strides[1] = a.strides[0];
        a.shape[0] = 1;
        a.strides[0] = 0;
    }
    if (b_vec) {  // [K] -> [K, 1]
        b.ndim = 2;
        b.shape[1] = 1;
        b.strides[1] = 0;
    }
    const int64_t M = a.shape[a.ndim - 2], K = a.shape[a.ndim - 1];
    const int64_t Kb = b.shape[b.ndim - 2], N = b.shape[b.ndim - 1];
    if (K != Kb)
        return fail(ctx, RTEN_ERR_INCOMPATIBLE_SHAPES, "Columns of first matrix does not match rows of second matrix");
    // broadcast prefixes
    const int pa = a.ndim - 2, pb = b.ndim - 2, pn = std::max(pa, pb);
    std::vector<int64_t> psize(pn), pas(pn), pbs(pn);
    for (int i = 0; i < pn; i++) {
        const int ia = i - (pn - pa), ib = i - (pn - pb);
        const int64_t sa = ia >= 0 ? a.shape[ia] : 1, sb = ib >= 0 ? b.shape[ib] : 1;
        if (sa != sb && sa != 1 && sb != 1) return fail(ctx, RTEN_ERR_INCOMPATIBLE_SHAPES, "Cannot broadcast shapes");
        psize[i] = std::max(sa, sb);
        if (sa == 0 || sb == 0) psize[i] = 0;
        pas[i] = (ia >= 0 && sa != 1) ? a.strides[ia] : 0;
        pbs[i] = (ib >= 0 && sb != 1) ? b.strides[ib] : 0;
    }
    // output shape
    int64_t oshape[RTEN_MAX_DIMS];
    int on = 0;
    for (int i = 0; i < pn; i++) oshape[on++] = psize[i];
    if (!a_vec) oshape[on++] = M;
    if (!b_vec) oshape[on++] = N;
    if (on > RTEN_MAX_DIMS) return fail(ctx, RTEN_ERR_INVALID_VALUE, "tensor rank out of range");
    rten_tensor ov;
    RTB_TRY(sc.out(out, A.out_dtype, on, oshape, &ov, nullptr));
    int64_t total = 1;
    for (int i = 0; i < on; i++) total *= oshape[i];
    if (total == 0) return RTEN_OK;
    // output strides of the prefix dims / row / col in the (vector-expanded) [prefix.., M, N] view
    std::vector<int64_t> pos(pn, 0);
    int64_t o_rs = 0, o_cs = 0;
    {
        int k = 0;
        for (int i = 0; i < pn; i++) pos[i] = ov.strides[k++];
        if (!a_vec) o_rs = ov.strides[k++];
        if (!b_vec) o_cs = ov.strides[k++];
    }
    rten_tensor dv = ov;
    bool copy_out = false;
    const int esize = A.kind == 0 ? 4 : 1;
    int64_t nbatch = 1;
    for (int i = 0; i < pn; i++) nbatch *= psize[i];
    int64_t nb_mats = 1;
    for (int i = 0; i < pb; i++) nb_mats *= b.shape[i];

    GemmLaunch L;
    L.kind = A.kind;
    L.a_signed = A.a->dtype == RTEN_I8;
    L.b_signed = (A.pb ? A.pb->dtype : A.b->dtype) == RTEN_I8;
    L.N = (int)N;
    L.K = (int)K;
    L.epi = A.epi;
    L.epi.d_is_i32 = A.out_dtype == RTEN_I32;

    if (K == 0) {
        // lib.rs:843-873: product term vanishes; out = bias (f32) / 0 (int).  Reuse Add machinery: fill.
        if (!is_contiguous(&ov)) {
            set_contiguous(&dv);
            void* t = nullptr;
            RTB_TRY(temp_alloc(ctx, (size_t)total * 4, &t));
            dv.data = t;
            copy_out = true;
        }
        RTB_CUDA(ctx, cudaMemsetAsync(dv.data, 0, (size_t)total * 4, ctx->stream));
        if (A.kind == 0 && L.epi.bias) {
            long long shp[2] = {total / N, N}, s0[2] = {N, 1}, sb[2] = {0, 1};
            RTB_TRY(launch_nd_add(ctx, (const float*)dv.data, L.epi.bias, (float*)dv.data, 2, shp, s0, sb, s0, 0));
        }
    } else {
        // B operand
        Mat mb;
        if (A.pb) {
            if (A.pb->kind != 0 || A.pb->K != K || A.pb->N != N)
                return fail(ctx, RTEN_ERR_INVALID_VALUE, "prepacked B does not match the matmul shape");
            mb.base = A.pb->data;
            mb.rows = N;
            mb.K = K;
            mb.rs = A.pb->ld;
            mb.ks = 1;
            nb_mats = 1;
        } else {
            mb.base = b.data;
            mb.rows = N;
            mb.K = K;
            mb.rs = b.strides[b.ndim - 1];
            mb.ks = b.strides[b.ndim - 2];
        }
        Mat ma;
        ma.base = a.data;
        ma.K = K;
        ma.ks = a.strides[a.ndim - 1];
        ma.rs = a.strides[a.ndim - 2];
        ma.rows = M;

        // Flatten [A.., M, K] x [K, N] into one [A*M, K] GEMM (matmul.rs:266-297) when A's rows are
        // uniformly strided; otherwise keep (up to two) batch dims.
        bool flat = false;
        BatchDims bd;
        const std::vector<int64_t> b_eff = A.pb ? std::vector<int64_t>(pn, 0) : pbs;
        for (int attempt = 0; attempt < 2; attempt++) {
            // attempt 0: write straight into the caller's (possibly strided) output; attempt 1: contiguous temp
            if (attempt == 1) {
                set_contiguous(&dv);
                void* t = nullptr;
                RTB_TRY(temp_alloc(ctx, (size_t)total * 4, &t));
                dv.data = t;
                copy_out = true;
                int k = 0;
                for (int i = 0; i < pn; i++) pos[i] = dv.strides[k++];
                if (!a_vec) o_rs = dv.strides[k++];
                if (!b_vec) o_cs = dv.strides[k++];
            }
            flat = false;
            if (nb_mats == 1) {
                std::vector<int64_t> sz = psize, as = pas, zs(pn, 0), os = pos;
                sz.push_back(M);
                as.push_back(ma.rs);
                zs.push_back(0);
                os.push_back(o_rs);
                BatchDims c = collapse_batch(sz, as, zs, os);
                if (c.ok && c.z1 == 1) {
                    flat = true;
                    ma.rows = c.z0;
                    if (c.z0 > 1) {
                        ma.rs = c.a0;
                        o_rs = c.o0;
                    }
                    break;
                }
            }
            bd = collapse_batch(psize, pas, b_eff, pos);
            if (bd.ok) break;
            if (attempt == 1)
                return fail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "matmul batch dims do not collapse to 2 strided dims");
        }
        L.epi.d = dv.data;
        L.epi.s_row = o_rs;
        L.epi.s_col = b_vec ? 1 : o_cs;
        if (flat) {
            L.M = (int)ma.rows;
            L.z0 = L.z1 = 1;
        } else {
            L.M = (int)M;
            L.z0 = (int)bd.z0;
            L.z1 = (int)bd.z1;
            ma.z0 = bd.z0;
            ma.z1 = bd.z1;
            ma.zs0 = bd.a0;
            ma.zs1 = bd.a1;
            mb.z0 = bd.z0;
            mb.z1 = bd.z1;
            mb.zs0 = bd.b0;
            mb.zs1 = bd.b1;
            L.epi.s_z0 = bd.o0;
            L.epi.s_z1 = bd.o1;
        }
        if (A.kind == 1 && !flat && (A.a_zp || A.b_zp) && nbatch > 1)
            return fail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "MatMulInteger with a batched RHS and zero points is not supported");
        RTB_TRY(to_kmajor(ctx, esize, ma, &L.a));
        if (mb.z0 > 1 && mb.zs0 == 0) {}  // broadcast handled by stride 0
        RTB_TRY(to_kmajor(ctx, esize, mb, &L.b));
        if (A.pb && A.kind == 0 && L.b.base == A.pb->data) L.b_x3_slot = &const_cast<rten_packed*>(A.pb)->x3;

        // residual (same shape as out, any strides) -> only contiguous or row-strided supported directly
        if (A.residual) {
            rten_tensor rv;
            RTB_TRY(sc.in(A.residual, &rv));
            if (rv.ndim != on) return fail(ctx, RTEN_ERR_INCOMPATIBLE_SHAPES, "residual shape does not match output");
            for (int i = 0; i < on; i++)
                if (rv.shape[i] != oshape[i]) return fail(ctx, RTEN_ERR_INCOMPATIBLE_SHAPES, "residual shape does not match output");
            rten_tensor rc;
            RTB_TRY(sc.contiguous(&rv, &rc));
            L.epi.r = (const float*)rc.data;
            L.epi.r_scale = 1.0f;
            L.epi.r_col = 1;
            L.epi.r_row = N;
            L.epi.r_z0 = flat ? 0 : M * N;
            L.epi.r_z1 = flat ? 0 : bd.z0 * M * N;
        }

        // integer zero points
        if (A.kind == 1) {
            const int64_t rows_total = flat ? ma.rows : M;
            if (A.a_zp) {
                rten_tensor z;
                RTB_TRY(sc.in(A.a_zp, &z));
                const int len = z.ndim == 0 ? 1 : (int)z.shape[0];
                if (len == 1) {  // scalar (DynamicQuantizeLinear's zero point): read in place by the epilogue
                    L.epi.za8 = (const uint8_t*)z.data;
                    L.epi.za8_signed = z.dtype == RTEN_I8;
                } else {
                    int32_t* za = nullptr;
                    RTB_TRY(temp_alloc(ctx, (size_t)len * 4, (void**)&za));
                    RTB_TRY(launch_zp_to_i32(ctx, z.data, z.dtype == RTEN_I8, len, z.ndim == 0 ? 0 : z.strides[0], za));
                    L.epi.za = za;
                    L.epi.za_len = len;
                }
                if (A.pb && A.pb->colsum) {
                    L.epi.colsum = A.pb->colsum;
                } else {
                    int32_t* cs = nullptr;
                    RTB_TRY(temp_alloc(ctx, (size_t)N * 4, (void**)&cs));
                    RTB_TRY(launch_rowsum8(ctx, L.b.base, L.b_signed, N, (int)K, L.b.strides[1], cs));
                    L.epi.colsum = cs;
                }
            }
            if (A.b_zp) {
                rten_tensor z;
                RTB_TRY(sc.in(A.b_zp, &z));
                const int len = z.ndim == 0 ? 1 : (int)z.shape[0];
                int32_t* zb = nullptr;
                RTB_TRY(temp_alloc(ctx, (size_t)len * 4, (void**)&zb));
                RTB_TRY(launch_zp_to_i32(ctx, z.data, z.dtype == RTEN_I8, len, z.ndim == 0 ? 0 : z.strides[0], zb));
                L.epi.zb = zb;
                L.epi.zb_len = len;
                int32_t* rs = nullptr;
                RTB_TRY(temp_alloc(ctx, (size_t)rows_total * 4, (void**)&rs));
                RTB_TRY(launch_rowsum8(ctx, L.a.base, L.a_signed, rows_total, (int)K, L.a.strides[1], rs));
                L.epi.rowsum = rs;
            }
        }
        // M <= 32 f32 rows: the HBM-streaming skinny kernel (exact f32 FMA arithmetic) instead of a 128-row MMA tile
        // (rten-gemm's gemv path, rten-gemm/src/lib.rs:668-747)
        if (A.kind == 0 && L.z0 == 1 && L.z1 == 1 && L.M <= 32 && L.epi.s_col == 1 && L.epi.bias_kind != 2 &&
            (!L.epi.r || L.epi.r_col == 1) && !L.epi.range && L.a.strides[0] == 1 && L.b.strides[0] == 1) {
            SkinnyF32Launch S;
            S.a = (const float*)L.a.base;
            S.as = L.a.strides[1];
            S.b = (const float*)L.b.base;
            S.bs = L.b.strides[1];
            S.M = L.M;
            S.N = L.N;
            S.K = L.K;
            S.alpha = L.epi.alpha;
            S.bias = L.epi.bias_kind == 1 ? L.epi.bias : nullptr;
            S.residual = L.epi.r;
            S.rs = L.epi.r_row;
            S.r_scale = L.epi.r_scale;
            S.act = L.epi.act;
            S.out = (float*)L.epi.d;
            S.os = L.epi.s_row;
            if (skinny_f32_supported(S)) {
                RTB_TRY(launch_skinny_f32(ctx, S));
                goto launched;
            }
        }
        {
        rten_status st = launch_umma_gemm(ctx, L);
        if (st == RTEN_ERR_UNSUPPORTED_VALUE) return fail(ctx, st, "GEMM operands are not addressable by TMA after packing");
        RTB_TRY(st);
        }
    launched:;
    }
    if (copy_out) {
        long long shape[RTEN_MAX_DIMS], ss[RTEN_MAX_DIMS], ds[RTEN_MAX_DIMS];
        for (int i = 0; i < on; i++) {
            shape[i] = oshape[i];
            ss[i] = dv.strides[i];
            ds[i] = ov.strides[i];
        }
        RTB_TRY(launch_nd_copy(ctx, 4, dv.data, ov.data, on, shape, ss, ds));
    }
    return RTEN_OK;
}

// src/ops/matmul.rs:513-533 zero_point_to_vec validation
}  // namespace

extern "C" {

rten_status rten_b200_prepack_b(rten_ctx* ctx, const rten_tensor* b, rten_packed** out) {
    RTB_TRY(check_ctx(ctx));
    if (!b || !out) return RTEN_ERR_INVALID_VALUE;
    *out = nullptr;
    if (b->ndim != 2) return fail(ctx, RTEN_ERR_INVALID_VALUE, "prepack expects a matrix");  // matmul_prepack_b: try_into Matrix
    if (b->dtype == RTEN_I32) return fail(ctx, RTEN_ERR_UNSUPPORTED_TYPE, "unsupported type");
    OpScope sc(ctx);
    rten_tensor bv;
    rten_status st = sc.in(b, &bv);
    rten_packed* p = nullptr;
    if (st == RTEN_OK) {
        const int es = dtype_size(b->dtype);
        p = new rten_packed();
        p->kind = 0;
        p->dtype = b->dtype;
        p->K = bv.shape[0];
        p->N = bv.shape[1];
        p->ld = round_up(std::max<int64_t>(p->K, 1), 16 / es);
        st = pool_alloc(ctx, (size_t)std::max<int64_t>(p->N * p->ld, 1) * es, &p->data);
        if (st == RTEN_OK) {
            RTB_CUDA(ctx, cudaMemsetAsync(p->data, 0, (size_t)std::max<int64_t>(p->N * p->ld, 1) * es, ctx->stream));
            long long shape[2] = {p->N, p->K}, ss[2] = {bv.strides[1], bv.strides[0]}, ds[2] = {p->ld, 1};
            st = launch_nd_copy(ctx, es, bv.data, p->data, 2, shape, ss, ds);
        }
        if (st == RTEN_OK && es == 1 && p->N > 0) {
            st = pool_alloc(ctx, (size_t)p->N * 4, (void**)&p->colsum);
            if (st == RTEN_OK) st = launch_rowsum8(ctx, p->data, p->dtype == RTEN_I8, p->N, (int)p->K, p->ld, p->colsum);
        }
    }
    st = sc.finish(st);
    if (st != RTEN_OK) {
        if (p) rten_b200_packed_free(ctx, p);
        return st;
    }
    *out = p;
    return RTEN_OK;
}

void rten_b200_packed_free(rten_ctx* ctx, rten_packed* p) {
    if (!p) return;
    if (ctx) {
        pool_free(ctx, p->data);
        pool_free(ctx, p->colsum);
    }
    if (p->x3) cudaFree(p->x3);
    delete p;
}

// ---- Gemm ---------------------------------------------------------------------------------
rten_status rten_b200_gemm(rten_ctx* ctx, const rten_tensor* a, const rten_tensor* b, const rten_tensor* c, float alpha,
                           float beta, int trans_a, int trans_b, rten_tensor* out) {
    RTB_TRY(check_ctx(ctx));
    if (!a || !b || !out) return fail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
    if (a->dtype != RTEN_F32 || b->dtype != RTEN_F32 || (c && c->dtype != RTEN_F32))
        return fail(ctx, RTEN_ERR_UNSUPPORTED_TYPE, "unsupported type");
    if (a->ndim != 2 || b->ndim != 2) return fail(ctx, RTEN_ERR_INVALID_VALUE, "input must have 2 dims");
    OpScope sc(ctx);
    rten_tensor av, bv, cv;
    rten_status st = sc.in(a, &av);
    if (st == RTEN_OK) st = sc.in(b, &bv);
    if (st == RTEN_OK && c) st = sc.in(c, &cv);
    if (st == RTEN_OK) {
        auto transpose = [](rten_tensor& t) {
            std::swap(t.shape[0], t.shape[1]);
            std::swap(t.strides[0], t.strides[1]);
        };
        if (trans_a) transpose(av);
        if (trans_b) transpose(bv);
        if (av.shape[1] != bv.shape[0]) {
            st = fail(ctx, RTEN_ERR_INCOMPATIBLE_SHAPES, "Columns of first matrix does not match rows of second matrix");
        } else {
            MatMulArgs A{};
            A.kind = 0;
            A.a = &av;
            A.b = &bv;
            A.pb = nullptr;
            A.out_dtype = RTEN_F32;
            A.epi.alpha = alpha;
            const int64_t M = av.shape[0], N = bv.shape[1];
            if (c && beta != 0.0f) {
                // broadcast c to [M, N] (matmul.rs:63-67)
                int64_t cs[2] = {0, 0};
                bool ok = cv.ndim <= 2;
                if (ok) {
                    for (int i = 0; i < cv.ndim; i++) {
                        const int od = 2 - cv.ndim + i;
                        const int64_t want = od == 0 ? M : N;
                        if (cv.shape[i] == want)
                            cs[od] = cv.strides[i];
                        else if (cv.shape[i] == 1)
                            cs[od] = 0;
                        else
                            ok = false;
                    }
                }
                if (!ok) {
                    st = fail(ctx, RTEN_ERR_INCOMPATIBLE_SHAPES, "Cannot broadcast c to output shape");
                } else {
                    A.epi.r = (const float*)cv.data;
                    A.epi.r_scale = beta;
                    A.epi.r_row = cs[0];
                    A.epi.r_col = cs[1];
                }
            }
            if (st == RTEN_OK) {
                // matmul_core's residual plumbing is for same-shape tensors; C is already set in epi.
                st = matmul_core(sc, A, out);
            }
        }
    }
    return sc.finish(st);
}

// ---- MatMul / FusedMatMul -----------------------------------------------------------------
rten_status rten_b200_matmul_ex(rten_ctx* ctx, const rten_tensor* a, const rten_tensor* b, const rten_packed* pb,
                                const rten_tensor* bias, float alpha, const rten_tensor* residual, int activation,
                                rten_tensor* out) {
    RTB_TRY(check_ctx(ctx));
    if (!a || !b || !out) return fail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
    if (a->dtype != RTEN_F32 || b->dtype != RTEN_F32 || (pb && pb->dtype != RTEN_F32))
        return fail(ctx, RTEN_ERR_UNSUPPORTED_TYPE, "unsupported type");
    OpScope sc(ctx);
    rten_tensor av, bv, biasv, biasc;
    rten_status st = sc.in(a, &av);
    if (st == RTEN_OK) {
        if (pb) {
            bv = *b;  // only the shape is consulted
            bv.data = nullptr;
        } else {
            st = sc.in(b, &bv);
        }
    }
    MatMulArgs A{};
    A.kind = 0;
    A.a = &av;
    A.b = &bv;
    A.pb = pb;
    A.out_dtype = RTEN_F32;
    A.epi.alpha = alpha;
    A.epi.act = activation;
    A.residual = residual;
    if (st == RTEN_OK && bias) {
        if (bias->dtype != RTEN_F32 || bias->ndim != 1) {
            st = fail(ctx, RTEN_ERR_CAST_FAILED, "bias must be a float vector");
        } else {
            st = sc.in(bias, &biasv);
            if (st == RTEN_OK) st = sc.contiguous(&biasv, &biasc);
            const int64_t N = bv.ndim >= 2 ? bv.shape[bv.ndim - 1] : 1;
            if (st == RTEN_OK && biasc.shape[0] != N) st = fail(ctx, RTEN_ERR_INVALID_VALUE, "WrongBiasSize");
            A.epi.bias = (const float*)biasc.data;
            A.epi.bias_kind = 1;
        }
    }
    if (st == RTEN_OK) st = matmul_core(sc, A, out);
    return sc.finish(st);
}

rten_status rten_b200_matmul(rten_ctx* ctx, const rten_tensor* a, const rten_tensor* b, const rten_packed* pb,
                             const rten_tensor* bias, float alpha, rten_tensor* out) {
    return rten_b200_matmul_ex(ctx, a, b, pb, bias, alpha, nullptr, 0, out);
}

// ---- MatMulInteger / MatMulIntegerToFloat ------------------------------------------------------
rten_status rten_b200_matmul_integer(rten_ctx* ctx, const rten_tensor* a, const rten_tensor* b, const rten_packed* pb,
                                     const rten_tensor* a_zp, const rten_tensor* b_zp, const rten_tensor* scale,
                                     rten_tensor* out) {
    return rten_b200_matmul_integer_ex(ctx, a, b, pb, a_zp, b_zp, scale, nullptr, nullptr, nullptr, 0, nullptr, out);
}

rten_status rten_b200_matmul_integer_ex(rten_ctx* ctx, const rten_tensor* a, const rten_tensor* b, const rten_packed* pb,
                                        const rten_tensor* a_zp, const rten_tensor* b_zp, const rten_tensor* scale,
                                        const rten_tensor* scale_b, const rten_tensor* bias, const rten_tensor* residual,
                                        int activation, rten_tensor* out_range, rten_tensor* out) {
    RTB_TRY(check_ctx(ctx));
    if (!a || !b || !out) return fail(ctx, RTEN_ERR_MISSING_INPUTS, "missing inputs");
    if ((bias || residual || activation || scale_b) && !scale)
        return fail(ctx, RTEN_ERR_INVALID_VALUE, "bias / residual / activation follow the float conversion: a scale is required");
    if (activation < 0 || activation > 3) return fail(ctx, RTEN_ERR_INVALID_VALUE, "unknown activation");
    auto is8 = [](int dt) { return dt == RTEN_U8 || dt == RTEN_I8; };
    if (!is8(a->dtype) || !is8(b->dtype)) return fail(ctx, RTEN_ERR_UNSUPPORTED_TYPE, "unsupported type");
    const int64_t a_rows = a->ndim > 1 ? a->shape[a->ndim - 2] : 1;
    const int64_t b_cols = b->ndim > 1 ? b->shape[b->ndim - 1] : 1;
    RTB_TRY(check_zero_point(ctx, a_zp, a_rows, a->dtype));
    RTB_TRY(check_zero_point(ctx, b_zp, b_cols, b->dtype));
    OpScope sc(ctx);
    rten_tensor av, bv, sv, svc;
    rten_status st = sc.in(a, &av);
    if (st == RTEN_OK) {
        if (pb && pb->dtype == b->dtype) {
            bv = *b;
            bv.data = nullptr;
        } else {
            pb = nullptr;
            st = sc.in(b, &bv);
        }
    }
    MatMulArgs A{};
    A.kind = 1;
    A.a = &av;
    A.b = &bv;
    A.pb = pb;
    A.a_zp = a_zp;
    A.b_zp = b_zp;
    A.out_dtype = scale ? RTEN_F32 : RTEN_I32;
    if (st == RTEN_OK && scale) {
        // OutputScale::from_view (matmul.rs:712-721)
        if (scale->dtype != RTEN_F32) {
            st = fail(ctx, RTEN_ERR_CAST_FAILED, "scale must be float");
        } else if (scale->ndim > 1) {
            st = fail(ctx, RTEN_ERR_INVALID_VALUE, "scale should have rank 0 or 1");
        } else {
            st = sc.in(scale, &sv);
            if (st == RTEN_OK) st = sc.contiguous(&sv, &svc);
            const int64_t len = svc.ndim == 0 ? 1 : svc.shape[0];
            if (st == RTEN_OK && len != 1 && len != b_cols)
                st = fail(ctx, RTEN_ERR_INCOMPATIBLE_SHAPES, "Scale length does not match tensor columns");
            A.epi.scale = (const float*)svc.data;
            A.epi.scale_len = (int)len;
        }
    }
    rten_tensor biasv, biasc, s2v;
    if (st == RTEN_OK && scale_b) {
        if (scale_b->dtype != RTEN_F32 || numel(scale_b) != 1) {
            st = fail(ctx, RTEN_ERR_INVALID_VALUE, "the second scale factor must be a float scalar");
        } else {
            st = sc.in(scale_b, &s2v);
            A.epi.scale2 = (const float*)s2v.data;
        }
    }
    if (st == RTEN_OK && bias) {
        if (bias->dtype != RTEN_F32 || bias->ndim != 1) {
            st = fail(ctx, RTEN_ERR_CAST_FAILED, "bias must be a float vector");
        } else {
            st = sc.in(bias, &biasv);
            if (st == RTEN_OK) st = sc.contiguous(&biasv, &biasc);
            if (st == RTEN_OK && biasc.shape[0] != b_cols) st = fail(ctx, RTEN_ERR_INVALID_VALUE, "WrongBiasSize");
            A.epi.bias = (const float*)biasc.data;
            A.epi.bias_kind = 1;
        }
    }
    A.epi.act = activation;
    A.residual = residual;
    if (st == RTEN_OK && out_range) {
        if (!scale || out_range->dtype != RTEN_I32 || numel(out_range) != 2 || out_range->device < 0 || !is_contiguous(out_range))
            st = fail(ctx, RTEN_ERR_INVALID_VALUE, "the output range must be a device-resident i32[2] (float outputs only)");
        else
            A.epi.range = (int*)out_range->data;
    }
    if (st == RTEN_OK) st = matmul_core(sc, A, out);
    return sc.finish(st);
}

}  // extern "C"
