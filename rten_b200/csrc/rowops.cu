// HBM-bound kernels of the hot path: Softmax / AddSoftmax, LayerNormalization, Erf / Gelu,
// DynamicQuantizeLinear, plus the layout / glue kernels that keep whole models resident.
//
// Accumulation ORDER follows the reference's AVX-512 path (16 f32 lanes, fold_unroll<4>), so
// Softmax and LayerNormalization results are bit-identical to it, not merely close:
//   softmax lane sums  : rten-vecmath/src/softmax.rs:192-228 (per-SIMD-lane partial sums, lanes summed in order)
//   Sum / SumSquareSub : rten-vecmath/src/sum.rs:22-35,111-130 + rten-simd/src/iter.rs:70-120
//   Normalize          : rten-vecmath/src/normalize.rs:101-169
#include <cuda_runtime.h>

#include <cfloat>
#include <cstdint>
#include <cstdlib>

#include "common.h"
#include "math.cuh"
#include "rowmath.cuh"
#include "rowops.h"
#include "comm_device.cuh"

namespace rtb {

constexpr int VL = 16;  // AVX-512 f32 lanes of the reference path

// =========================================================================================
// Softmax: one warp per row of n contiguous floats.
// =========================================================================================
struct SoftmaxParams {
    const float* x;
    float* y;
    long long rows;
    int n;
    int flush_nan;
    // optional mask, broadcast over up to 4 leading dims of x (row index decomposed over lead[])
    const float* mask;
    int nlead;
    long long lead[4];
    long long mstride[4];
    long long mstride_last;
};

__global__ void __launch_bounds__(256) softmax_kernel(const SoftmaxParams p) {
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= p.rows) return;
    const float* x = p.x + row * p.n;
    float* y = p.y + row * p.n;
    const float* m = nullptr;
    if (p.mask) {
        long long off = 0;
        if (p.rows < 0x7fffffffLL) {  // 32-bit division: a 64-bit one costs ~10x the instructions, per row
            unsigned rem = (unsigned)row;
            for (int d = p.nlead - 1; d >= 0; d--) {
                const unsigned ld = (unsigned)p.lead[d];
                const unsigned q = rem / ld;
                off += (long long)(rem - q * ld) * p.mstride[d];
                rem = q;
            }
        } else {
            long long rem = row;
            for (int d = p.nlead - 1; d >= 0; d--) {
                const long long idx = rem % p.lead[d];
                rem /= p.lead[d];
                off += idx * p.mstride[d];
            }
        }
        m = p.mask + off;
    }
    const int n = p.n;
    // pass 1: z = x (+ mask), max  (softmax.rs:176-190; max is order independent)
    float mx = -FLT_MAX;
    for (int i = lane; i < n; i += 32) {
        float v = x[i];
        if (m) v = __fadd_rn(v, m[(long long)i * p.mstride_last]);
        mx = fmaxf(mx, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    // pass 2: e = ReducedRangeExp(z - max); partial[l] accumulates elements i == l (mod 16) in
    // ascending i -- thread l (< 16) adds its own element, then the one held by thread l + 16.
    float partial = 0.0f;
    for (int i0 = 0; i0 < n; i0 += 32) {
        const int i = i0 + lane;
        float e = 0.0f;
        if (i < n) {
            float v = x[i];
            if (m) v = __fadd_rn(v, m[(long long)i * p.mstride_last]);
            e = reduced_range_exp(__fsub_rn(v, mx));
            y[i] = e;
        }
        const float e_hi = __shfl_down_sync(0xffffffffu, e, 16);
        if (lane < VL) {
            if (i < n) partial = __fadd_rn(partial, e);
            if (i + 16 < n) partial = __fadd_rn(partial, e_hi);
        }
    }
    float s = 0.0f;
#pragma unroll
    for (int l = 0; l < VL; l++) s = __fadd_rn(s, __shfl_sync(0xffffffffu, partial, l));
    const float inv = __fdiv_rn(1.0f, s);
    __syncwarp();
    // pass 3: y = e * (1/sum), optional NaN flush
    for (int i = lane; i < n; i += 32) {
        float v = __fmul_rn(y[i], inv);
        if (p.flush_nan && v != v) v = 0.0f;
        y[i] = v;
    }
}

// -----------------------------------------------------------------------------------------
// Vectorised softmax: the row lives in registers, ONE pass over global memory (128-bit loads and stores).
// The reference accumulates the exponentials in 16 SIMD-lane partial sums, lane l owning the elements i = l (mod 16)
// in ascending i (rten-vecmath/src/softmax.rs:192-228).  A float4 at float4-index f holds lanes 4 (f mod 4) .. + 3, so
// thread (t0 = f mod 4) owns FOUR of the sixteen chains outright: a row is handled by 4 * S threads, thread (t0, s)
// holding the float4s f = t0 + 4 (s F + k), k < F -- its own contiguous-in-i piece of its four chains.  Adds inside a
// thread are sequential in i; segment s starts from segment s - 1's sums (shuffle), which keeps the exact order.
// Requires n % (16 S) == 0, F = n / (16 S) <= 16, 16-byte aligned rows.
// -----------------------------------------------------------------------------------------
template <int S, int FMAX>
__global__ void __launch_bounds__(128) softmax_vec_kernel(const SoftmaxParams p) {
    constexpr int LPR = 4 * S;        // threads per row
    constexpr int RPW = 32 / LPR;     // rows per warp
    const int lane = threadIdx.x & 31;
    const int t0 = lane & 3, seg = (lane >> 2) & (S - 1), rw = lane / LPR;
    const long long warp_id = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const long long row = warp_id * RPW + rw;
    const bool live = row < p.rows;
    const int n = p.n;
    const int F = n / (16 * S);
    const long long rr = live ? row : 0;
    const float4* x4 = reinterpret_cast<const float4*>(p.x + rr * n);
    float4* y4 = reinterpret_cast<float4*>(p.y + rr * n);
    const float* m = nullptr;
    if (p.mask) {
        long long off = 0;
        unsigned rem = (unsigned)rr;  // (the launcher keeps rows < 2^31 on this path)
#pragma unroll
        for (int d = 3; d >= 0; d--) {  // (static indices: the parameter arrays stay in the constant bank)
            if (d < p.nlead) {
                const unsigned ld = (unsigned)p.lead[d];
                const unsigned q = rem / ld;
                off += (long long)(rem - q * ld) * p.mstride[d];
                rem = q;
            }
        }
        m = p.mask + off;
    }
    float4 v[FMAX];
    float mx = -FLT_MAX;
#pragma unroll
    for (int k = 0; k < FMAX; k++) {
        if (k < F) {
            const int f = t0 + 4 * (seg * F + k);
            float4 a = live ? __ldg(x4 + f) : make_float4(0.f, 0.f, 0.f, 0.f);
            if (m) {
                float4 b;
                if (p.mstride_last == 1) {
                    b = __ldg(reinterpret_cast<const float4*>(m) + f);
                } else {
                    const long long ms = p.mstride_last;
                    b = make_float4(__ldg(m + (4LL * f) * ms), __ldg(m + (4LL * f + 1) * ms), __ldg(m + (4LL * f + 2) * ms),
                                    __ldg(m + (4LL * f + 3) * ms));
                }
                a.x = __fadd_rn(a.x, b.x);
                a.y = __fadd_rn(a.y, b.y);
                a.z = __fadd_rn(a.z, b.z);
                a.w = __fadd_rn(a.w, b.w);
            }
            v[k] = a;
            mx = fmaxf(mx, fmaxf(fmaxf(a.x, a.y), fmaxf(a.z, a.w)));
        }
    }
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
#pragma unroll
    for (int k = 0; k < FMAX; k++) {
        if (k < F) {
            v[k].x = reduced_range_exp(__fsub_rn(v[k].x, mx));
            v[k].y = reduced_range_exp(__fsub_rn(v[k].y, mx));
            v[k].z = reduced_range_exp(__fsub_rn(v[k].z, mx));
            v[k].w = reduced_range_exp(__fsub_rn(v[k].w, mx));
        }
    }
    // the four chains of this thread, segment after segment
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int sg = 0; sg < S; sg++) {
        if (sg > 0) {  // continue from the previous segment's running sums
            const float4 in = make_float4(__shfl_up_sync(0xffffffffu, acc.x, 4), __shfl_up_sync(0xffffffffu, acc.y, 4),
                                          __shfl_up_sync(0xffffffffu, acc.z, 4), __shfl_up_sync(0xffffffffu, acc.w, 4));
            if (seg == sg) acc = in;
        }
        if (seg == sg) {
#pragma unroll
            for (int k = 0; k < FMAX; k++) {
                if (k < F) {
                    acc.x = __fadd_rn(acc.x, v[k].x);
                    acc.y = __fadd_rn(acc.y, v[k].y);
                    acc.z = __fadd_rn(acc.z, v[k].z);
                    acc.w = __fadd_rn(acc.w, v[k].w);
                }
            }
        }
    }
    // lanes summed in order l = 0 .. 15: thread t0 of the LAST segment holds l = 4 t0 .. 4 t0 + 3
    float s = 0.0f;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const float in = __shfl_up_sync(0xffffffffu, s, 1);
        if (t0 == q) {
            if (q > 0) s = in;
            s = __fadd_rn(__fadd_rn(__fadd_rn(__fadd_rn(s, acc.x), acc.y), acc.z), acc.w);
        }
    }
    s = __shfl_sync(0xffffffffu, s, rw * LPR + (S - 1) * 4 + 3);
    const float inv = __fdiv_rn(1.0f, s);
    if (!live) return;
#pragma unroll
    for (int k = 0; k < FMAX; k++) {
        if (k < F) {
            float4 o = make_float4(__fmul_rn(v[k].x, inv), __fmul_rn(v[k].y, inv), __fmul_rn(v[k].z, inv), __fmul_rn(v[k].w, inv));
            if (p.flush_nan) {
                if (o.x != o.x) o.x = 0.0f;
                if (o.y != o.y) o.y = 0.0f;
                if (o.z != o.z) o.z = 0.0f;
                if (o.w != o.w) o.w = 0.0f;
            }
            y4[t0 + 4 * (seg * F + k)] = o;
        }
    }
}

rten_status launch_softmax(rten_ctx* ctx, const float* x, float* y, long long rows, int n, int flush_nan,
                           const float* mask, int nlead, const long long* lead, const long long* mstride,
                           long long mstride_last) {
    if (rows == 0 || n == 0) return RTEN_OK;
    SoftmaxParams p;
    p.x = x;
    p.y = y;
    p.rows = rows;
    p.n = n;
    p.flush_nan = flush_nan;
    p.mask = mask;
    p.nlead = nlead;
    for (int i = 0; i < 4; i++) {
        p.lead[i] = i < nlead ? lead[i] : 1;
        p.mstride[i] = i < nlead ? mstride[i] : 0;
    }
    p.mstride_last = mstride_last;
    const int wpb = 8;
    // register-resident rows, 128-bit accesses: n a multiple of 16 S with F = n / (16 S) <= 16 float4s per thread.
    // More segments (threads per row) when the rows alone would not give every SM enough warps to hide the latency
    // of its one burst of loads.
    int S = 0;
    for (int c = 1; c <= 8; c *= 2) {
        if (n % (16 * c) != 0 || n / (16 * c) > 16) continue;
        S = c;
        const long long warps = (rows * 4 * c + 31) / 32;
        if (warps >= 32LL * ctx->num_sms || n / (16 * c) <= 2) break;
    }
    const bool aligned = (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 &&
                         (!mask || mstride_last != 1 || (reinterpret_cast<uintptr_t>(mask) & 15) == 0);
    bool mask_vec_ok = true;  // vector mask loads need every row's mask base 16-byte aligned
    if (mask && mstride_last == 1)
        for (int i = 0; i < nlead; i++)
            if (mstride[i] % 4) mask_vec_ok = false;
    if (S && aligned && mask_vec_ok && rows < 0x7fffffffLL && !getenv("RTEN_B200_NO_VEC_ROWS")) {
        const int rpw = 32 / (4 * S);
        const int vwpb = 4;
        const long long warps = (rows + rpw - 1) / rpw;
        const unsigned blocks = (unsigned)((warps + vwpb - 1) / vwpb);
        const int F = n / (16 * S);
        const int fm = F <= 2 ? 2 : (F <= 4 ? 4 : (F <= 8 ? 8 : 16));
        cudaStream_t st = ctx->stream;
#define RTB_SOFTMAX_CASE(SS, FF) \
    case SS * 100 + FF: softmax_vec_kernel<SS, FF><<<blocks, vwpb * 32, 0, st>>>(p); break;
        switch (S * 100 + fm) {
            RTB_SOFTMAX_CASE(1, 2) RTB_SOFTMAX_CASE(1, 4) RTB_SOFTMAX_CASE(1, 8) RTB_SOFTMAX_CASE(1, 16)
            RTB_SOFTMAX_CASE(2, 2) RTB_SOFTMAX_CASE(2, 4) RTB_SOFTMAX_CASE(2, 8) RTB_SOFTMAX_CASE(2, 16)
            RTB_SOFTMAX_CASE(4, 2) RTB_SOFTMAX_CASE(4, 4) RTB_SOFTMAX_CASE(4, 8) RTB_SOFTMAX_CASE(4, 16)
            RTB_SOFTMAX_CASE(8, 2) RTB_SOFTMAX_CASE(8, 4) RTB_SOFTMAX_CASE(8, 8) RTB_SOFTMAX_CASE(8, 16)
        }
#undef RTB_SOFTMAX_CASE
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail_cuda(ctx, e, "softmax launch");
        count_launch(ctx);
        return RTEN_OK;
    }
    const long long blocks = (rows + wpb - 1) / wpb;
    softmax_kernel<<<(unsigned)blocks, wpb * 32, 0, ctx->stream>>>(p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "softmax launch");
    count_launch(ctx);
    return RTEN_OK;
}

// =========================================================================================
// LayerNormalization: one warp per row.
// fold_unroll<4> with V=16: position p = i % 64 owns accumulator (u = p / 16, l = p % 16) for the
// full 64-element chunks; thread t owns p = t and p = t + 32.
// =========================================================================================
template <bool SQSUB>
__device__ __forceinline__ float simd_fold_unroll4(const float* x, int n, float off, int lane) {
    float a0 = 0.0f, a1 = 0.0f;
    const int nfull = n / 64;
    for (int c = 0; c < nfull; c++) {
        a0 = fold_step<SQSUB>(a0, x[c * 64 + lane], off);
        a1 = fold_step<SQSUB>(a1, x[c * 64 + 32 + lane], off);
    }
    // acc[0][l] = ((acc[0][l] + acc[1][l]) + acc[2][l]) + acc[3][l]
    const float b = __shfl_down_sync(0xffffffffu, a0, 16);
    const float d = __shfl_down_sync(0xffffffffu, a1, 16);
    float acc = __fadd_rn(__fadd_rn(__fadd_rn(a0, b), a1), d);  // valid for lane < 16
    // remaining full 16-chunks and the masked tail go into acc[0]
    int i = nfull * 64;
    if (lane < VL) {
        for (; i + VL <= n; i += VL) acc = fold_step<SQSUB>(acc, x[i + lane], off);
        if (i + lane < n) acc = fold_step<SQSUB>(acc, x[i + lane], off);
    }
    float s = 0.0f;
#pragma unroll
    for (int l = 0; l < VL; l++) s = __fadd_rn(s, __shfl_sync(0xffffffffu, acc, l));
    return s;
}

struct LayerNormParams {
    const float* x;
    float* y;
    long long rows;
    int n;
    const float* gamma;  // per element or null
    float gamma_scalar;
    const float* beta;  // per element or null
    float beta_scalar;
    float eps;
    // scalar scale / bias that live on the device (read by the kernel: the call stays asynchronous and capturable)
    const float* gamma_sp;
    const float* beta_sp;
};

__global__ void __launch_bounds__(256) layer_norm_kernel(const LayerNormParams p) {
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= p.rows) return;
    const float* x = p.x + row * p.n;
    float* y = p.y + row * p.n;
    const int n = p.n;
    const float gamma_scalar = p.gamma_sp ? __ldg(p.gamma_sp) : p.gamma_scalar;
    const float beta_scalar = p.beta_sp ? __ldg(p.beta_sp) : p.beta_scalar;
    const float mean = __fdiv_rn(simd_fold_unroll4<false>(x, n, 0.0f, lane), (float)n);
    const float var = __fdiv_rn(simd_fold_unroll4<true>(x, n, mean, lane), (float)n);
    const float rstd = __fdiv_rn(gamma_scalar, __fsqrt_rn(__fadd_rn(var, p.eps)));
    if (!p.gamma && !p.beta) {
        for (int i = lane; i < n; i += 32) y[i] = __fmaf_rn(__fsub_rn(x[i], mean), rstd, beta_scalar);
    } else if (p.gamma && !p.beta && beta_scalar == 0.0f) {
        for (int i = lane; i < n; i += 32) y[i] = __fmul_rn(__fsub_rn(x[i], mean), __fmul_rn(p.gamma[i], rstd));
    } else {
        for (int i = lane; i < n; i += 32) {
            const float sv = __fmul_rn(p.gamma ? p.gamma[i] : 1.0f, rstd);
            const float bv = __fadd_rn(p.beta ? p.beta[i] : 0.0f, beta_scalar);
            y[i] = __fmaf_rn(__fsub_rn(x[i], mean), sv, bv);
        }
    }
}

// -----------------------------------------------------------------------------------------
// Vectorised LayerNormalization: row in registers, one pass over global memory, 128-bit accesses.
// fold_unroll<4> over 16 lanes = 64 independent chains, chain p owning the elements i = p (mod 64) in ascending i
// (only full 64-element chunks exist here: n % 64 == 0).  The float4 at index f holds chains 4 (f mod 16) .. + 3:
// thread (c = f mod 16, segment s) keeps f = c + 16 (s F + k), k < F, and so owns its four chains outright; segment
// s continues from segment s - 1's sums.  Then acc[0][l] = ((acc[0][l] + acc[1][l]) + acc[2][l]) + acc[3][l] with
// chain p = 16 u + l, and the 16 lanes are summed in order (rten-vecmath/src/sum.rs:22-35, rten-simd/src/iter.rs:70-120).
// -----------------------------------------------------------------------------------------
template <int S, int FMAX>
__global__ void __launch_bounds__(128) layer_norm_vec_kernel(const LayerNormParams p) {
    constexpr int LPR = 16 * S;
    constexpr int RPW = 32 / LPR;
    const int lane = threadIdx.x & 31;
    const int c = lane & 15, seg = (lane >> 4) & (S - 1), rw = lane / LPR;
    const long long warp_id = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const long long row = warp_id * RPW + rw;
    const bool live = row < p.rows;
    const int n = p.n;
    const int F = n / (64 * S);
    const long long rr = live ? row : 0;
    const float4* x4 = reinterpret_cast<const float4*>(p.x + rr * n);
    float4 v[FMAX];
#pragma unroll
    for (int k = 0; k < FMAX; k++)
        if (k < F) v[k] = __ldg(x4 + c + 16 * (seg * F + k));
    const float gamma_scalar = p.gamma_sp ? __ldg(p.gamma_sp) : p.gamma_scalar;
    const float beta_scalar = p.beta_sp ? __ldg(p.beta_sp) : p.beta_scalar;
    const float mean = __fdiv_rn(ln_vec_fold<S, false, FMAX>(v, F, 0.0f, c, seg), (float)n);
    const float var = __fdiv_rn(ln_vec_fold<S, true, FMAX>(v, F, mean, c, seg), (float)n);
    const float rstd = __fdiv_rn(gamma_scalar, __fsqrt_rn(__fadd_rn(var, p.eps)));
    if (!live) return;
    float4* y4 = reinterpret_cast<float4*>(p.y + rr * n);
    const float4* g4 = reinterpret_cast<const float4*>(p.gamma);
    const float4* b4 = reinterpret_cast<const float4*>(p.beta);
    const int mode = (!p.gamma && !p.beta) ? 0 : ((p.gamma && !p.beta && beta_scalar == 0.0f) ? 1 : 2);
#pragma unroll
    for (int k = 0; k < FMAX; k++) {
        if (k < F) {
            const int f = c + 16 * (seg * F + k);
            const float4 a = v[k];
            float4 o;
            if (mode == 0) {
                o = make_float4(__fmaf_rn(__fsub_rn(a.x, mean), rstd, beta_scalar), __fmaf_rn(__fsub_rn(a.y, mean), rstd, beta_scalar),
                                __fmaf_rn(__fsub_rn(a.z, mean), rstd, beta_scalar), __fmaf_rn(__fsub_rn(a.w, mean), rstd, beta_scalar));
            } else if (mode == 1) {
                const float4 g = __ldg(g4 + f);
                o = make_float4(__fmul_rn(__fsub_rn(a.x, mean), __fmul_rn(g.x, rstd)), __fmul_rn(__fsub_rn(a.y, mean), __fmul_rn(g.y, rstd)),
                                __fmul_rn(__fsub_rn(a.z, mean), __fmul_rn(g.z, rstd)), __fmul_rn(__fsub_rn(a.w, mean), __fmul_rn(g.w, rstd)));
            } else {
                const float4 g = p.gamma ? __ldg(g4 + f) : make_float4(1.f, 1.f, 1.f, 1.f);
                const float4 b = p.beta ? __ldg(b4 + f) : make_float4(0.f, 0.f, 0.f, 0.f);
                o = make_float4(__fmaf_rn(__fsub_rn(a.x, mean), __fmul_rn(g.x, rstd), __fadd_rn(b.x, beta_scalar)),
                                __fmaf_rn(__fsub_rn(a.y, mean), __fmul_rn(g.y, rstd), __fadd_rn(b.y, beta_scalar)),
                                __fmaf_rn(__fsub_rn(a.z, mean), __fmul_rn(g.z, rstd), __fadd_rn(b.z, beta_scalar)),
                                __fmaf_rn(__fsub_rn(a.w, mean), __fmul_rn(g.w, rstd), __fadd_rn(b.w, beta_scalar)));
            }
            y4[f] = o;
        }
    }
}

rten_status launch_layer_norm(rten_ctx* ctx, const float* x, float* y, long long rows, int n, const float* gamma,
                              float gamma_scalar, const float* beta, float beta_scalar, float eps, const float* gamma_sp,
                              const float* beta_sp) {
    if (rows == 0 || n == 0) return RTEN_OK;
    LayerNormParams p{x, y, rows, n, gamma, gamma_scalar, beta, beta_scalar, eps, gamma_sp, beta_sp};
    const int wpb = 8;
    // 16 S lanes per row, F = n / (64 S) <= 16 float4s per thread; two segments per row when that is possible and the
    // rows alone would leave the SMs short of warps
    int S = 0;
    for (int c = 1; c <= 2; c *= 2) {
        if (n % (64 * c) != 0 || n / (64 * c) > 16) continue;
        S = c;
        const long long warps = (rows * 16 * c + 31) / 32;
        if (warps >= 32LL * ctx->num_sms) break;
    }
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    if (S && al16(x) && al16(y) && al16(gamma) && al16(beta) && !getenv("RTEN_B200_NO_VEC_ROWS")) {
        const int rpw = 2 / S;
        const int vwpb = 4;
        const long long warps = (rows + rpw - 1) / rpw;
        const unsigned blocks = (unsigned)((warps + vwpb - 1) / vwpb);
        const int F = n / (64 * S);
        const int fm = F <= 4 ? 4 : (F <= 8 ? 8 : (F <= 12 ? 12 : 16));
        cudaStream_t st = ctx->stream;
#define RTB_LN_CASE(SS, FF) \
    case SS * 100 + FF: layer_norm_vec_kernel<SS, FF><<<blocks, vwpb * 32, 0, st>>>(p); break;
        switch (S * 100 + fm) {
            RTB_LN_CASE(1, 4) RTB_LN_CASE(1, 8) RTB_LN_CASE(1, 12) RTB_LN_CASE(1, 16)
            RTB_LN_CASE(2, 4) RTB_LN_CASE(2, 8) RTB_LN_CASE(2, 12) RTB_LN_CASE(2, 16)
        }
#undef RTB_LN_CASE
    } else {
        const long long blocks = (rows + wpb - 1) / wpb;
        layer_norm_kernel<<<(unsigned)blocks, wpb * 32, 0, ctx->stream>>>(p);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "layer_norm launch");
    count_launch(ctx);
    return RTEN_OK;
}

// Row sums in the reference's Sum order (GlobalAveragePool = Sum / len, src/ops/pooling.rs:516-521).
// Element k of row r lives at x[r_off(r) + k * kstride].
__global__ void __launch_bounds__(256)
row_mean_kernel(const float* x, float* y, long long rows, int n, long long rows_inner, long long s_outer,
                long long s_inner, long long kstride) {
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const float* xr = x + (row / rows_inner) * s_outer + (row % rows_inner) * s_inner;
    float a0 = 0.0f, a1 = 0.0f;
    const int nfull = n / 64;
    for (int c = 0; c < nfull; c++) {
        a0 = __fadd_rn(a0, xr[(long long)(c * 64 + lane) * kstride]);
        a1 = __fadd_rn(a1, xr[(long long)(c * 64 + 32 + lane) * kstride]);
    }
    const float b = __shfl_down_sync(0xffffffffu, a0, 16);
    const float d = __shfl_down_sync(0xffffffffu, a1, 16);
    float acc = __fadd_rn(__fadd_rn(__fadd_rn(a0, b), a1), d);
    int i = nfull * 64;
    if (lane < VL) {
        for (; i + VL <= n; i += VL) acc = __fadd_rn(acc, xr[(long long)(i + lane) * kstride]);
        if (i + lane < n) acc = __fadd_rn(acc, xr[(long long)(i + lane) * kstride]);
    }
    float s = 0.0f;
#pragma unroll
    for (int l = 0; l < VL; l++) s = __fadd_rn(s, __shfl_sync(0xffffffffu, acc, l));
    if (lane == 0) y[row] = __fdiv_rn(s, (float)n);
}

// Same reduction order, one THREAD per row: for channels-last tensors consecutive rows (channels) are adjacent in
// memory, so a warp reads 32 consecutive floats per element index (coalesced) instead of one strided row per warp.
__global__ void __launch_bounds__(128)
row_mean_thread_kernel(const float* x, float* y, long long rows, int n, long long rows_inner, long long s_outer,
                       long long s_inner, long long kstride) {
    const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    const float* xr = x + (row / rows_inner) * s_outer + (row % rows_inner) * s_inner;
    float acc[4][VL];
#pragma unroll
    for (int u = 0; u < 4; u++)
#pragma unroll
        for (int l = 0; l < VL; l++) acc[u][l] = 0.0f;
    int i = 0;
    for (; i + 64 <= n; i += 64) {
#pragma unroll
        for (int u = 0; u < 4; u++)
#pragma unroll
            for (int l = 0; l < VL; l++) acc[u][l] = __fadd_rn(acc[u][l], xr[(long long)(i + u * VL + l) * kstride]);
    }
#pragma unroll
    for (int l = 0; l < VL; l++) acc[0][l] = __fadd_rn(__fadd_rn(__fadd_rn(acc[0][l], acc[1][l]), acc[2][l]), acc[3][l]);
    for (; i + VL <= n; i += VL) {
#pragma unroll
        for (int l = 0; l < VL; l++) acc[0][l] = __fadd_rn(acc[0][l], xr[(long long)(i + l) * kstride]);
    }
#pragma unroll
    for (int l = 0; l < VL; l++)
        if (i + l < n) acc[0][l] = __fadd_rn(acc[0][l], xr[(long long)(i + l) * kstride]);
    float s = 0.0f;
#pragma unroll
    for (int l = 0; l < VL; l++) s = __fadd_rn(s, acc[0][l]);
    y[row] = __fdiv_rn(s, (float)n);
}

rten_status launch_row_mean(rten_ctx* ctx, const float* x, float* y, long long rows, int n, long long rows_inner,
                            long long s_outer, long long s_inner, long long kstride) {
    if (rows == 0) return RTEN_OK;
    if (s_inner == 1 && kstride != 1) {
        row_mean_thread_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, ctx->stream>>>(x, y, rows, n, rows_inner, s_outer,
                                                                                        s_inner, kstride);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail_cuda(ctx, e, "row_mean launch");
        count_launch(ctx);
        return RTEN_OK;
    }
    const int wpb = 8;
    row_mean_kernel<<<(unsigned)((rows + wpb - 1) / wpb), wpb * 32, 0, ctx->stream>>>(x, y, rows, n, rows_inner,
                                                                                       s_outer, s_inner, kstride);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "row_mean launch");
    count_launch(ctx);
    return RTEN_OK;
}

// =========================================================================================
// Elementwise (contiguous): Erf, Gelu, ApproxGelu, Relu, and same-shape Add (+ optional Relu)
// 128-bit loads/stores, grid sized to fill the SMs.
// =========================================================================================
template <int OP>
__device__ __forceinline__ float unary_apply(float v) {
    if (OP == UNARY_ERF) return erf_ref(v);
    if (OP == UNARY_GELU) return gelu_ref(v);
    if (OP == UNARY_APPROX_GELU) return approx_gelu_ref(v);
    return v > 0.0f ? v : 0.0f;  // UNARY_RELU
}

template <int OP>
__global__ void __launch_bounds__(256)
unary_kernel(const float* __restrict__ x, float* __restrict__ y, long long n, int vec) {
    const long long n4 = vec ? (n >> 2) : 0;
    const long long stride = (long long)gridDim.x * blockDim.x;
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i < n4; i += stride) {
        float4 v = reinterpret_cast<const float4*>(x)[i];
        v.x = unary_apply<OP>(v.x);
        v.y = unary_apply<OP>(v.y);
        v.z = unary_apply<OP>(v.z);
        v.w = unary_apply<OP>(v.w);
        reinterpret_cast<float4*>(y)[i] = v;
    }
    // tail (everything when the buffers are not 16-B aligned)
    for (long long j = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride)
        y[j] = unary_apply<OP>(x[j]);
}

static int ew_grid(rten_ctx* ctx, long long work_items) {
    long long blocks = (work_items + 255) / 256;
    long long cap = (long long)ctx->num_sms * 8;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

rten_status launch_unary(rten_ctx* ctx, int op, const float* x, float* y, long long n) {
    if (n == 0) return RTEN_OK;
    const int vec = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0 ? 1 : 0;
    const int grid = ew_grid(ctx, vec ? (n + 3) / 4 : n);
    switch (op) {
        case UNARY_ERF: unary_kernel<UNARY_ERF><<<grid, 256, 0, ctx->stream>>>(x, y, n, vec); break;
        case UNARY_GELU: unary_kernel<UNARY_GELU><<<grid, 256, 0, ctx->stream>>>(x, y, n, vec); break;
        case UNARY_APPROX_GELU: unary_kernel<UNARY_APPROX_GELU><<<grid, 256, 0, ctx->stream>>>(x, y, n, vec); break;
        case UNARY_RELU: unary_kernel<UNARY_RELU><<<grid, 256, 0, ctx->stream>>>(x, y, n, vec); break;
        default: return fail(ctx, RTEN_ERR_INVALID_VALUE, "unknown unary op");
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "unary launch");
    count_launch(ctx);
    return RTEN_OK;
}

// General N-d strided kernels (up to 8 dims): copy / broadcast add.  Used for layout changes
// (NCHW <-> NHWC views, weight prepack), host staging of strided tensors and broadcast Add.
struct NdParams {
    int ndim;
    long long shape[RTEN_MAX_DIMS];
    long long sa[RTEN_MAX_DIMS];
    long long sb[RTEN_MAX_DIMS];
    long long sd[RTEN_MAX_DIMS];
    long long n;
};

template <typename T>
__global__ void __launch_bounds__(256) nd_copy_kernel(const T* __restrict__ src, T* __restrict__ dst, const NdParams p) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    if (p.n <= 0x7fffffffLL) {  // 32-bit index arithmetic: the emulated 64-bit division is ~10x the instructions
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < p.n; i += stride) {
            unsigned rem = (unsigned)i;
            long long so = 0, dof = 0;
#pragma unroll 1
            for (int d = p.ndim - 1; d >= 0; d--) {
                const unsigned sh = (unsigned)p.shape[d];
                const unsigned q = rem / sh;
                const unsigned idx = rem - q * sh;
                rem = q;
                so += (long long)idx * p.sa[d];
                dof += (long long)idx * p.sd[d];
            }
            dst[dof] = src[so];
        }
        return;
    }
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < p.n; i += stride) {
        long long rem = i, so = 0, dof = 0;
#pragma unroll 1
        for (int d = p.ndim - 1; d >= 0; d--) {
            const long long idx = rem % p.shape[d];
            rem /= p.shape[d];
            so += idx * p.sa[d];
            dof += idx * p.sd[d];
        }
        dst[dof] = src[so];
    }
}

__global__ void __launch_bounds__(256)
nd_add_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ d, const NdParams p, int relu) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < p.n; i += stride) {
        long long rem = i, ao = 0, bo = 0, dof = 0;
#pragma unroll 1
        for (int k = p.ndim - 1; k >= 0; k--) {
            const long long idx = rem % p.shape[k];
            rem /= p.shape[k];
            ao += idx * p.sa[k];
            bo += idx * p.sb[k];
            dof += idx * p.sd[k];
        }
        float v = (relu & 2) ? __fmul_rn(a[ao], b[bo]) : __fadd_rn(a[ao], b[bo]);  // flags: 1 = Relu after, 2 = Mul
        if (relu & 1) v = v > 0.0f ? v : 0.0f;
        d[dof] = v;
    }
}

__global__ void __launch_bounds__(256)
add_flat_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ d, long long n, int relu) {
    const long long n4 = n >> 2;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const float4 x = reinterpret_cast<const float4*>(a)[i];
        const float4 y = reinterpret_cast<const float4*>(b)[i];
        float4 o = (relu & 2) ? make_float4(__fmul_rn(x.x, y.x), __fmul_rn(x.y, y.y), __fmul_rn(x.z, y.z), __fmul_rn(x.w, y.w))
                              : make_float4(__fadd_rn(x.x, y.x), __fadd_rn(x.y, y.y), __fadd_rn(x.z, y.z), __fadd_rn(x.w, y.w));
        if (relu & 1) {
            o.x = o.x > 0.f ? o.x : 0.f;
            o.y = o.y > 0.f ? o.y : 0.f;
            o.z = o.z > 0.f ? o.z : 0.f;
            o.w = o.w > 0.f ? o.w : 0.f;
        }
        reinterpret_cast<float4*>(d)[i] = o;
    }
    for (long long j = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) {
        float v = (relu & 2) ? __fmul_rn(a[j], b[j]) : __fadd_rn(a[j], b[j]);
        if (relu & 1) v = v > 0.f ? v : 0.f;
        d[j] = v;
    }
}

// Collapse to the iteration order that makes the DESTINATION contiguous-fastest: dims are visited in
// the given order; callers pass dims sorted so that the last has the smallest dst stride.
rten_status launch_nd_copy(rten_ctx* ctx, int esize, const void* src, void* dst, int ndim, const long long* shape,
                           const long long* sstride, const long long* dstride) {
    NdParams p;
    memset(&p, 0, sizeof(p));
    p.ndim = ndim;
    p.n = 1;
    for (int i = 0; i < ndim; i++) {
        p.shape[i] = shape[i];
        p.sa[i] = sstride[i];
        p.sd[i] = dstride[i];
        p.n *= shape[i];
    }
    if (p.n == 0) return RTEN_OK;
    if (esize != 4 && esize != 1) return fail(ctx, RTEN_ERR_UNSUPPORTED_TYPE, "unsupported element size");
    // Wider elements when both sides are contiguous along the innermost visited dim: a padded copy of a channels-last
    // u8 tensor moves 16 bytes per thread instead of one.
    int es = esize;
    if (ndim >= 1 && p.sa[ndim - 1] == 1 && p.sd[ndim - 1] == 1) {
        while (es < 16) {
            const long long inner_bytes = p.shape[ndim - 1] * es;
            bool ok = inner_bytes % (2 * es) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) % (2 * es)) == 0;
            for (int i = 0; i < ndim - 1 && ok; i++)
                if ((p.sa[i] * es) % (2 * es) != 0 || (p.sd[i] * es) % (2 * es) != 0) ok = false;
            if (!ok) break;
            // strides are in units of the CURRENT element size: halve them together with the inner extent
            p.shape[ndim - 1] /= 2;
            for (int i = 0; i < ndim - 1; i++) {
                p.sa[i] /= 2;
                p.sd[i] /= 2;
            }
            p.n /= 2;
            es *= 2;
        }
    }
    const int grid = ew_grid(ctx, p.n);
    switch (es) {
        case 1: nd_copy_kernel<uint8_t><<<grid, 256, 0, ctx->stream>>>((const uint8_t*)src, (uint8_t*)dst, p); break;
        case 2: nd_copy_kernel<uint16_t><<<grid, 256, 0, ctx->stream>>>((const uint16_t*)src, (uint16_t*)dst, p); break;
        case 4: nd_copy_kernel<uint32_t><<<grid, 256, 0, ctx->stream>>>((const uint32_t*)src, (uint32_t*)dst, p); break;
        case 8: nd_copy_kernel<uint2><<<grid, 256, 0, ctx->stream>>>((const uint2*)src, (uint2*)dst, p); break;
        default: nd_copy_kernel<uint4><<<grid, 256, 0, ctx->stream>>>((const uint4*)src, (uint4*)dst, p); break;
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "nd_copy launch");
    count_launch(ctx);
    return RTEN_OK;
}

// a and d dense, b dense over the TRAILING dims and broadcast over the leading ones (bias rows, position embeddings):
// d[i] = a[i] (+|*) b[i mod period], 128 bits per thread, 32-bit index arithmetic
__global__ void __launch_bounds__(256)
add_periodic_kernel(const float4* __restrict__ a, const float4* __restrict__ b, float4* __restrict__ d, unsigned n4, unsigned period4, int relu) {
    const unsigned stride = gridDim.x * blockDim.x;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const float4 x = a[i];
        const float4 y = b[i % period4];
        float4 o = (relu & 2) ? make_float4(__fmul_rn(x.x, y.x), __fmul_rn(x.y, y.y), __fmul_rn(x.z, y.z), __fmul_rn(x.w, y.w))
                              : make_float4(__fadd_rn(x.x, y.x), __fadd_rn(x.y, y.y), __fadd_rn(x.z, y.z), __fadd_rn(x.w, y.w));
        if (relu & 1) {
            o.x = o.x > 0.f ? o.x : 0.f;
            o.y = o.y > 0.f ? o.y : 0.f;
            o.z = o.z > 0.f ? o.z : 0.f;
            o.w = o.w > 0.f ? o.w : 0.f;
        }
        d[i] = o;
    }
}

rten_status launch_nd_add(rten_ctx* ctx, const float* a, const float* b, float* d, int ndim, const long long* shape,
                          const long long* sa, const long long* sb, const long long* sd, int relu) {
    {
        // fast path: a / d dense, b = a dense block of the trailing dims repeated over the leading ones
        long long dense = 1, period = 0, n = 1;
        bool ok = ndim >= 1, in_bcast = false;
        for (int i = ndim - 1; i >= 0 && ok; i--) {
            if (shape[i] != 1) {
                ok = sa[i] == dense && sd[i] == dense;
                if (!in_bcast && sb[i] == dense) {
                } else if (sb[i] == 0) {
                    if (!in_bcast) period = dense;
                    in_bcast = true;
                } else {
                    ok = false;
                }
            }
            dense *= shape[i];
            n *= shape[i];
        }
        if (ok && in_bcast && period > 0 && (period & 3) == 0 && n < 0x7fffffffLL && n > 0 &&
            ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(d)) & 15) == 0) {
            add_periodic_kernel<<<ew_grid(ctx, n / 4), 256, 0, ctx->stream>>>(reinterpret_cast<const float4*>(a), reinterpret_cast<const float4*>(b),
                                                                               reinterpret_cast<float4*>(d), (unsigned)(n / 4), (unsigned)(period / 4), relu);
            cudaError_t e = cudaGetLastError();
            if (e != cudaSuccess) return fail_cuda(ctx, e, "nd_add launch");
            count_launch(ctx);
            return RTEN_OK;
        }
    }
    NdParams p;
    memset(&p, 0, sizeof(p));
    p.ndim = ndim;
    p.n = 1;
    for (int i = 0; i < ndim; i++) {
        p.shape[i] = shape[i];
        p.sa[i] = sa[i];
        p.sb[i] = sb[i];
        p.sd[i] = sd[i];
        p.n *= shape[i];
    }
    if (p.n == 0) return RTEN_OK;
    nd_add_kernel<<<ew_grid(ctx, p.n), 256, 0, ctx->stream>>>(a, b, d, p, relu);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "nd_add launch");
    count_launch(ctx);
    return RTEN_OK;
}

rten_status launch_add_flat(rten_ctx* ctx, const float* a, const float* b, float* d, long long n, int relu) {
    if (n == 0) return RTEN_OK;
    const bool aligned =
        ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(d)) & 15) == 0;
    if (!aligned) {
        long long shape[1] = {n}, s1[1] = {1};
        return launch_nd_add(ctx, a, b, d, 1, shape, s1, s1, s1, relu);
    }
    add_flat_kernel<<<ew_grid(ctx, (n + 3) / 4), 256, 0, ctx->stream>>>(a, b, d, n, relu);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "add launch");
    count_launch(ctx);
    return RTEN_OK;
}

// =========================================================================================
// DynamicQuantizeLinear (src/ops/quantize.rs:352-434; rten-vecmath/src/quantize.rs:38-77)
//   pass 1: min / max  (order independent) -> 2 floats (ordered-int atomics)
//   pass 2: scale, zero point (every thread recomputes the 6 scalar ops) + quantise
// =========================================================================================
__global__ void minmax_init_kernel(int* mm) {
    mm[0] = float_to_ordered(__int_as_float(0x7f800000));  // +inf
    mm[1] = float_to_ordered(__int_as_float(0xff800000));  // -inf
}

__global__ void __launch_bounds__(256) minmax_kernel(const float* __restrict__ x, long long n, int* mm) {
    float lo = __int_as_float(0x7f800000), hi = __int_as_float(0xff800000);
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long n4 = ((reinterpret_cast<uintptr_t>(x) & 15) == 0) ? (n >> 2) : 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const float4 v = reinterpret_cast<const float4*>(x)[i];
        lo = fminf(fminf(lo, v.x), fminf(v.y, fminf(v.z, v.w)));
        hi = fmaxf(fmaxf(hi, v.x), fmaxf(v.y, fmaxf(v.z, v.w)));
    }
    for (long long j = (n4 << 2) + (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride) {
        lo = fminf(lo, x[j]);
        hi = fmaxf(hi, x[j]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    __shared__ float slo[8], shi[8];
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) {
        slo[w] = lo;
        shi[w] = hi;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < 8; k++) {
            lo = fminf(lo, slo[k]);
            hi = fmaxf(hi, shi[k]);
        }
        atomicMin(&mm[0], float_to_ordered(lo));
        atomicMax(&mm[1], float_to_ordered(hi));
    }
}

__global__ void __launch_bounds__(256)
dql_quantize_kernel(const float* __restrict__ x, uint8_t* __restrict__ y, long long n, int* mm, float* scale_out,
                    uint8_t* zp_out, const RangeExchange xch) {
    // batch-sharded run: block 0 exchanges the local (min, max) with the other ranks over NVLink first (comm_device.cuh)
    range_exchange_begin(mm, xch);
    float scale, inv;
    int zp;
    dql_params(mm, scale, inv, zp);
    range_exchange_done(xch);  // (mm has been read by every thread of this block)
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        *scale_out = scale;
        *zp_out = (uint8_t)zp;
    }
    const long long stride = (long long)gridDim.x * blockDim.x;
    // A warp takes 2 KB of x per iteration as four fully coalesced 128-bit loads (lane l reads float4 j * 32 + l: whole
    // 512-byte rows per instruction, all four in flight) and writes the 512 quantised bytes as four coalesced 32-bit
    // stores.  (Sixteen consecutive floats per lane made every load instruction touch 32 half-used sectors.)
    const bool al = ((reinterpret_cast<uintptr_t>(x) & 15) == 0) && ((reinterpret_cast<uintptr_t>(y) & 3) == 0);
    const long long nblk = al ? (n >> 9) : 0;  // 512-element blocks, one per warp and iteration
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = stride >> 5;
    for (long long b = warp; b < nblk; b += nwarps) {
        const float4* xp = reinterpret_cast<const float4*>(x) + (b << 7) + lane;
        const float4 v0 = xp[0], v1 = xp[32], v2 = xp[64], v3 = xp[96];
        uint32_t* yp = reinterpret_cast<uint32_t*>(y) + (b << 7) + lane;
        const float4 vv[4] = {v0, v1, v2, v3};
#pragma unroll
        for (int g = 0; g < 4; g++)
            yp[32 * g] = (uint32_t)quant1(vv[g].x, inv, zp) | ((uint32_t)quant1(vv[g].y, inv, zp) << 8) |
                         ((uint32_t)quant1(vv[g].z, inv, zp) << 16) | ((uint32_t)quant1(vv[g].w, inv, zp) << 24);
    }
    for (long long j = (nblk << 9) + (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += stride)
        y[j] = quant1(x[j], inv, zp);
}

// Small tensors (decode-time activations): range and quantisation in ONE single-CTA kernel instead of three launches.
// min / max are order independent and the quantisation is the same per-element code, so results are identical.
__global__ void __launch_bounds__(1024)
dql_small_kernel(const float* __restrict__ x, uint8_t* __restrict__ y, int n, float* scale_out, uint8_t* zp_out) {
    __shared__ float slo[32], shi[32];
    __shared__ int mm[2];
    float lo = __int_as_float(0x7f800000), hi = __int_as_float(0xff800000);
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float v = x[i];
        lo = fminf(lo, v);
        hi = fmaxf(hi, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if ((threadIdx.x & 31) == 0) {
        slo[threadIdx.x >> 5] = lo;
        shi[threadIdx.x >> 5] = hi;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < (int)(blockDim.x >> 5); k++) {
            lo = fminf(lo, slo[k]);
            hi = fmaxf(hi, shi[k]);
        }
        mm[0] = float_to_ordered(lo);
        mm[1] = float_to_ordered(hi);
    }
    __syncthreads();
    float scale, inv;
    int zp;
    dql_params(mm, scale, inv, zp);
    if (threadIdx.x == 0) {
        *scale_out = scale;
        *zp_out = (uint8_t)zp;
    }
    for (int i = threadIdx.x; i < n; i += blockDim.x) y[i] = quant1(x[i], inv, zp);
}

// Quantise pass with a ROW-STRIDED destination: x is [rows, row_len] contiguous, row r of y starts at
// (r / rows_inner) * y_outer + (r % rows_inner) * y_inner -- the interior of a spatially pre-padded channels-last buffer.
__global__ void __launch_bounds__(256)
dql_quantize_rows_kernel(const float* __restrict__ x, uint8_t* __restrict__ y, long long rows, int row_len, int rows_inner,
                         long long y_inner, long long y_outer, int* mm, float* scale_out, uint8_t* zp_out, const RangeExchange xch) {
    range_exchange_begin(mm, xch);
    float scale, inv;
    int zp;
    dql_params(mm, scale, inv, zp);
    range_exchange_done(xch);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        *scale_out = scale;
        *zp_out = (uint8_t)zp;
    }
    const int groups = (row_len + 15) >> 4;
    const long long total = rows * groups;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const long long r = i / groups;
        const int g = (int)(i - r * groups);
        const float* xr = x + r * row_len + g * 16;
        uint8_t* yr = y + (r / rows_inner) * y_outer + (r % rows_inner) * y_inner + g * 16;
        const int nrem = row_len - g * 16;
        if (nrem >= 16 && ((reinterpret_cast<uintptr_t>(xr) | reinterpret_cast<uintptr_t>(yr)) & 15) == 0) {
            const float4* xp = reinterpret_cast<const float4*>(xr);
            const float4 v0 = xp[0], v1 = xp[1], v2 = xp[2], v3 = xp[3];
            const float f[16] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w, v2.x, v2.y, v2.z, v2.w, v3.x, v3.y, v3.z, v3.w};
            uint32_t w[4];
#pragma unroll
            for (int q = 0; q < 4; q++)
                w[q] = (uint32_t)quant1(f[4 * q], inv, zp) | ((uint32_t)quant1(f[4 * q + 1], inv, zp) << 8) |
                       ((uint32_t)quant1(f[4 * q + 2], inv, zp) << 16) | ((uint32_t)quant1(f[4 * q + 3], inv, zp) << 24);
            *reinterpret_cast<uint4*>(yr) = make_uint4(w[0], w[1], w[2], w[3]);
        } else {
            for (int j = 0; j < nrem && j < 16; j++) yr[j] = quant1(xr[j], inv, zp);
        }
    }
}

rten_status launch_dql_quantize_rows(rten_ctx* ctx, const float* x, uint8_t* y, long long rows, int row_len, int rows_inner,
                                     long long y_inner, long long y_outer, int* mm, float* scale_out, uint8_t* zp_out,
                                     const RangeExchange* xch) {
    const long long total = rows * ((row_len + 15) / 16);
    if (total == 0) return RTEN_OK;
    RangeExchange none;
    memset(&none, 0, sizeof(none));
    dql_quantize_rows_kernel<<<ew_grid(ctx, total), 256, 0, ctx->stream>>>(x, y, rows, row_len, rows_inner, y_inner, y_outer,
                                                                          mm, scale_out, zp_out, xch ? *xch : none);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "dql launch");
    count_launch(ctx);
    return RTEN_OK;
}

rten_status launch_dql_small(rten_ctx* ctx, const float* x, uint8_t* y, int n, float* scale_out, uint8_t* zp_out) {
    dql_small_kernel<<<1, 1024, 0, ctx->stream>>>(x, y, n, scale_out, zp_out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "dql launch");
    count_launch(ctx);
    return RTEN_OK;
}

__global__ void range_reset_kernel(int* mm, int pairs) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < pairs) {
        mm[2 * i] = float_to_ordered(__int_as_float(0x7f800000));      // +inf
        mm[2 * i + 1] = float_to_ordered(__int_as_float(0xff800000));  // -inf
    }
}

rten_status launch_range_reset(rten_ctx* ctx, int* mm, int pairs) {
    if (pairs == 0) return RTEN_OK;
    range_reset_kernel<<<(pairs + 127) / 128, 128, 0, ctx->stream>>>(mm, pairs);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "range reset launch");
    count_launch(ctx);
    return RTEN_OK;
}

rten_status launch_minmax(rten_ctx* ctx, const float* x, long long n, int* mm) {
    minmax_init_kernel<<<1, 1, 0, ctx->stream>>>(mm);
    count_launch(ctx);
    if (n > 0) {
        minmax_kernel<<<ew_grid(ctx, (n + 3) / 4), 256, 0, ctx->stream>>>(x, n, mm);
        count_launch(ctx);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "minmax launch");
    return RTEN_OK;
}

rten_status launch_dql_quantize(rten_ctx* ctx, const float* x, uint8_t* y, long long n, int* mm, float* scale_out,
                                uint8_t* zp_out, const RangeExchange* xch) {
    RangeExchange none;
    memset(&none, 0, sizeof(none));
    dql_quantize_kernel<<<ew_grid(ctx, (n + 15) / 16), 256, 0, ctx->stream>>>(x, y, n, mm, scale_out, zp_out, xch ? *xch : none);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "dql launch");
    count_launch(ctx);
    return RTEN_OK;
}

// =========================================================================================
// Integer helpers for the zero-point epilogue
// =========================================================================================
// sums over k of an 8-bit [rows, K] K-major matrix (row stride ld) -> i32
__global__ void __launch_bounds__(256)
rowsum8_kernel(const uint8_t* __restrict__ a, int is_signed, long long rows, int K, long long ld, int* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    const uint8_t* r = a + row * ld;
    int s = 0;
    for (int k = lane; k < K; k += 32) s += is_signed ? (int)(int8_t)r[k] : (int)r[k];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) out[row] = s;
}

rten_status launch_rowsum8(rten_ctx* ctx, const void* a, int is_signed, long long rows, int K, long long ld, int* out) {
    if (rows == 0) return RTEN_OK;
    const int wpb = 8;
    rowsum8_kernel<<<(unsigned)((rows + wpb - 1) / wpb), wpb * 32, 0, ctx->stream>>>((const uint8_t*)a, is_signed, rows,
                                                                                      K, ld, out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "rowsum launch");
    count_launch(ctx);
    return RTEN_OK;
}

// zero points (u8 or i8, element stride zs) -> i32
__global__ void zp_to_i32_kernel(const uint8_t* zp, int is_signed, int n, long long zs, int* out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = is_signed ? (int)(int8_t)zp[i * zs] : (int)zp[i * zs];
}

rten_status launch_zp_to_i32(rten_ctx* ctx, const void* zp, int is_signed, int n, long long zs, int* out) {
    if (n == 0) return RTEN_OK;
    zp_to_i32_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>((const uint8_t*)zp, is_signed, n, zs, out);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "zp_to_i32 launch");
    count_launch(ctx);
    return RTEN_OK;
}

__global__ void fill8_kernel(uint8_t* p, long long n, uint8_t v) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) p[i] = v;
}
rten_status launch_fill8(rten_ctx* ctx, void* p, long long n, uint8_t v) {
    if (n == 0) return RTEN_OK;
    fill8_kernel<<<ew_grid(ctx, n), 256, 0, ctx->stream>>>((uint8_t*)p, n, v);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "fill launch");
    count_launch(ctx);
    return RTEN_OK;
}

// cast_scale (src/ops/matmul.rs:734-773) for the unfused case
__global__ void __launch_bounds__(256)
cast_scale_kernel(const int* __restrict__ in, float* __restrict__ out, long long n, int cols, const float* scale,
                  int scale_len) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride)
        out[i] = __fmul_rn(__int2float_rn(in[i]), scale[scale_len == 1 ? 0 : (int)(i % cols)]);
}
rten_status launch_cast_scale(rten_ctx* ctx, const int* in, float* out, long long n, int cols, const float* scale,
                              int scale_len) {
    if (n == 0) return RTEN_OK;
    cast_scale_kernel<<<ew_grid(ctx, n), 256, 0, ctx->stream>>>(in, out, n, cols, scale, scale_len);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "cast_scale launch");
    count_launch(ctx);
    return RTEN_OK;
}

// =========================================================================================
// Explicit im2col (fallback for convolutions the TMA path cannot address: C*esize % 16 != 0, groups)
// out[(b,oy,ox), (ky,kx,c)] with row pitch kpad; taps outside the image get `pad_value`.
// =========================================================================================
template <typename T>
__global__ void __launch_bounds__(256)
im2col_kernel(const T* __restrict__ x, T* __restrict__ out, Im2ColParams p, T pad_value) {
    // one thread = 16 bytes of one im2col row (kpad is a multiple of 16 bytes): the pixel decode is shared by the
    // group and the store is one 128-bit transaction
    constexpr int VEC = 16 / (int)sizeof(T);
    const int groups = p.kpad / VEC;
    const long long total = (long long)p.B * p.OH * p.OW * groups;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const int kreal = p.kh * p.kw * p.C;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int g = (int)(i % groups);
        const long long pix = i / groups;
        const int ox = (int)(pix % p.OW);
        const long long r2 = pix / p.OW;
        const int oy = (int)(r2 % p.OH);
        const int b = (int)(r2 / p.OH);
        const T* xb = x + (long long)b * p.xs_b + (long long)p.c0 * p.xs_c;
        const int iy0 = oy * p.sy - p.pt, ix0 = ox * p.sx - p.pl;
        int k = g * VEC;
        int c = k % p.C, tap = k / p.C;
        int kx = tap % p.kw, ky = tap / p.kw;
        alignas(16) T v[VEC];
#pragma unroll
        for (int j = 0; j < VEC; j++, k++) {
            T val = 0;
            if (k < kreal) {
                const int iy = iy0 + ky * p.dy, ix = ix0 + kx * p.dx;
                val = (iy >= 0 && iy < p.H && ix >= 0 && ix < p.W)
                          ? xb[(long long)c * p.xs_c + (long long)iy * p.xs_h + (long long)ix * p.xs_w]
                          : pad_value;
            }
            v[j] = val;
            if (++c == p.C) {
                c = 0;
                if (++kx == p.kw) {
                    kx = 0;
                    ky++;
                }
            }
        }
        *reinterpret_cast<uint4*>(out + pix * p.kpad + (long long)g * VEC) = *reinterpret_cast<const uint4*>(v);
    }
}

rten_status launch_im2col(rten_ctx* ctx, int esize, const void* x, void* out, const Im2ColParams& p, int pad_value) {
    if (((long long)p.kpad * esize) % 16 != 0 || (reinterpret_cast<uintptr_t>(out) & 15) != 0)
        return fail(ctx, RTEN_ERR_INVALID_VALUE, "im2col rows must be multiples of 16 bytes");
    const long long total = (long long)p.B * p.OH * p.OW * (p.kpad * esize / 16);
    if (total == 0) return RTEN_OK;
    if (esize == 4) {
        float pv = 0.0f;
        im2col_kernel<float><<<ew_grid(ctx, total), 256, 0, ctx->stream>>>((const float*)x, (float*)out, p, pv);
    } else {
        im2col_kernel<uint8_t><<<ew_grid(ctx, total), 256, 0, ctx->stream>>>((const uint8_t*)x, (uint8_t*)out, p,
                                                                             (uint8_t)pad_value);
    }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "im2col launch");
    count_launch(ctx);
    return RTEN_OK;
}

// =========================================================================================
// Small-channel convolution support (C <= 4, e.g. the 3-channel ResNet stem): the image is copied once into a
// zero-padded NHWC4 buffer so that the kw pixels x 4 channels under a filter row are 4*kw CONTIGUOUS floats; the
// implicit-GEMM kernel then reads them as one 128-byte K block per filter row (ky).
// =========================================================================================
__global__ void __launch_bounds__(256)
smallc_pad_kernel(const float* __restrict__ x, float* __restrict__ xp, int B, int C, int H, int W, int Wp, int pl,
                  long long xs_b, long long xs_c, long long xs_h, long long xs_w) {
    const long long total = (long long)B * H * Wp;  // one thread per padded pixel (4 channels = one float4)
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int xw = (int)(i % Wp);
        const long long r = i / Wp;
        const int y = (int)(r % H);
        const int b = (int)(r / H);
        float v[4] = {0.f, 0.f, 0.f, 0.f};
        const int ix = xw - pl;
        if (ix >= 0 && ix < W) {
            const float* src = x + (long long)b * xs_b + (long long)y * xs_h + (long long)ix * xs_w;
            for (int c = 0; c < C; c++) v[c] = src[(long long)c * xs_c];
        }
        reinterpret_cast<float4*>(xp)[i] = make_float4(v[0], v[1], v[2], v[3]);
    }
}

// w [O, C, kh, kw] (strides) -> wp [O, kh, 32]: element (kx*4 + c) of filter row ky, zero elsewhere
__global__ void smallc_pack_w_kernel(const float* __restrict__ w, float* __restrict__ wp, int O, int C, int kh, int kw,
                                     long long ws_o, long long ws_c, long long ws_h, long long ws_w) {
    const int total = O * kh * 32;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        const int j = i % 32;
        const int ky = (i / 32) % kh;
        const int o = i / (32 * kh);
        const int kx = j >> 2, c = j & 3;
        wp[i] = (kx < kw && c < C) ? w[o * ws_o + c * ws_c + ky * ws_h + kx * ws_w] : 0.0f;
    }
}

rten_status launch_smallc_pad(rten_ctx* ctx, const float* x, float* xp, int B, int C, int H, int W, int Wp, int pl,
                              long long xs_b, long long xs_c, long long xs_h, long long xs_w) {
    const long long total = (long long)B * H * Wp;
    if (total == 0) return RTEN_OK;
    smallc_pad_kernel<<<ew_grid(ctx, total), 256, 0, ctx->stream>>>(x, xp, B, C, H, W, Wp, pl, xs_b, xs_c, xs_h, xs_w);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "smallc_pad launch");
    count_launch(ctx);
    return RTEN_OK;
}

rten_status launch_smallc_pack_w(rten_ctx* ctx, const float* w, float* wp, int O, int C, int kh, int kw, long long ws_o,
                                 long long ws_c, long long ws_h, long long ws_w) {
    const int total = O * kh * 32;
    if (total == 0) return RTEN_OK;
    smallc_pack_w_kernel<<<(total + 255) / 256, 256, 0, ctx->stream>>>(w, wp, O, C, kh, kw, ws_o, ws_c, ws_h, ws_w);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "smallc_pack_w launch");
    count_launch(ctx);
    return RTEN_OK;
}

// =========================================================================================
// Pooling / gather
// =========================================================================================
// channels-last fast path: one thread per (pixel, 4 channels), 128-bit loads/stores
__global__ void __launch_bounds__(256) maxpool_cl4_kernel(const float* __restrict__ x, float* __restrict__ y, PoolParams p) {
    const int C4 = p.C >> 2;
    const long long total = (long long)p.B * p.OH * p.OW * C4;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        long long rem = i;
        const int c = (int)(rem % C4) << 2;
        rem /= C4;
        const int ox = (int)(rem % p.OW);
        rem /= p.OW;
        const int oy = (int)(rem % p.OH);
        const int b = (int)(rem / p.OH);
        const float ninf = __int_as_float(0xff800000);
        float4 m = make_float4(ninf, ninf, ninf, ninf);
        for (int ky = 0; ky < p.kh; ky++) {
            const int iy = oy * p.sy - p.pt + ky;
            if (iy < 0 || iy >= p.H) continue;
            for (int kx = 0; kx < p.kw; kx++) {
                const int ix = ox * p.sx - p.pl + kx;
                if (ix < 0 || ix >= p.W) continue;
                const float4 v = *reinterpret_cast<const float4*>(x + (long long)b * p.xs_b + (long long)iy * p.xs_h + (long long)ix * p.xs_w + c);
                m.x = v.x > m.x ? v.x : m.x;
                m.y = v.y > m.y ? v.y : m.y;
                m.z = v.z > m.z ? v.z : m.z;
                m.w = v.w > m.w ? v.w : m.w;
            }
        }
        *reinterpret_cast<float4*>(y + (long long)b * p.ys_b + (long long)oy * p.ys_h + (long long)ox * p.ys_w + c) = m;
    }
}

__global__ void __launch_bounds__(256) maxpool_kernel(const float* __restrict__ x, float* __restrict__ y, PoolParams p) {
    const long long total = (long long)p.B * p.C * p.OH * p.OW;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        int b, c, oy, ox;
        long long rem = i;
        if (p.channels_fastest) {
            c = (int)(rem % p.C);
            rem /= p.C;
            ox = (int)(rem % p.OW);
            rem /= p.OW;
            oy = (int)(rem % p.OH);
            b = (int)(rem / p.OH);
        } else {
            ox = (int)(rem % p.OW);
            rem /= p.OW;
            oy = (int)(rem % p.OH);
            rem /= p.OH;
            c = (int)(rem % p.C);
            b = (int)(rem / p.C);
        }
        float m = __int_as_float(0xff800000);
        for (int ky = 0; ky < p.kh; ky++) {
            const int iy = oy * p.sy - p.pt + ky;
            if (iy < 0 || iy >= p.H) continue;
            for (int kx = 0; kx < p.kw; kx++) {
                const int ix = ox * p.sx - p.pl + kx;
                if (ix < 0 || ix >= p.W) continue;
                const float v = x[(long long)b * p.xs_b + (long long)c * p.xs_c + (long long)iy * p.xs_h + (long long)ix * p.xs_w];
                m = v > m ? v : m;
            }
        }
        y[(long long)b * p.ys_b + (long long)c * p.ys_c + (long long)oy * p.ys_h + (long long)ox * p.ys_w] = m;
    }
}

rten_status launch_maxpool(rten_ctx* ctx, const float* x, float* y, const PoolParams& p) {
    const long long total = (long long)p.B * p.C * p.OH * p.OW;
    if (total == 0) return RTEN_OK;
    const bool cl4 = p.xs_c == 1 && p.ys_c == 1 && (p.C % 4) == 0 && (p.xs_b % 4) == 0 && (p.xs_h % 4) == 0 &&
                     (p.xs_w % 4) == 0 && (p.ys_b % 4) == 0 && (p.ys_h % 4) == 0 && (p.ys_w % 4) == 0 &&
                     ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0;
    if (cl4)
        maxpool_cl4_kernel<<<ew_grid(ctx, total / 4), 256, 0, ctx->stream>>>(x, y, p);
    else
        maxpool_kernel<<<ew_grid(ctx, total), 256, 0, ctx->stream>>>(x, y, p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "maxpool launch");
    count_launch(ctx);
    return RTEN_OK;
}

__global__ void __launch_bounds__(256)
gather_rows_kernel(const float* __restrict__ table, const int* __restrict__ idx, float* __restrict__ out, long long nidx,
                   int width, long long t_rs, long long t_cs, long long rows) {
    const long long total = nidx * width;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const long long r = i / width;
        const int c = (int)(i % width);
        long long id = idx[r];
        if (id < 0) id += rows;  // negative indices count from the end (src/ops/gather.rs)
        out[i] = table[id * t_rs + c * t_cs];
    }
}

// contiguous table rows, width % 4 == 0: one float4 per thread, 32-bit index arithmetic
__global__ void __launch_bounds__(256)
gather_rows_vec_kernel(const float* __restrict__ table, const int* __restrict__ idx, float4* __restrict__ out, unsigned n4, unsigned w4,
                       long long t_rs, long long rows) {
    const unsigned stride = gridDim.x * blockDim.x;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const unsigned r = i / w4, c4 = i - r * w4;
        long long id = idx[r];
        if (id < 0) id += rows;
        out[i] = *reinterpret_cast<const float4*>(table + id * t_rs + 4 * c4);
    }
}

rten_status launch_gather_rows(rten_ctx* ctx, const float* table, const int* idx, float* out, long long nidx, int width,
                               long long t_rs, long long t_cs, long long rows) {
    if (nidx * width == 0) return RTEN_OK;
    if (t_cs == 1 && (width & 3) == 0 && (t_rs & 3) == 0 && nidx * width < 0x7fffffffLL &&
        ((reinterpret_cast<uintptr_t>(table) | reinterpret_cast<uintptr_t>(out)) & 15) == 0) {
        gather_rows_vec_kernel<<<ew_grid(ctx, nidx * width / 4), 256, 0, ctx->stream>>>(table, idx, reinterpret_cast<float4*>(out),
                                                                                       (unsigned)(nidx * width / 4), (unsigned)(width / 4), t_rs, rows);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail_cuda(ctx, e, "gather launch");
        count_launch(ctx);
        return RTEN_OK;
    }
    gather_rows_kernel<<<ew_grid(ctx, nidx * width), 256, 0, ctx->stream>>>(table, idx, out, nidx, width, t_rs, t_cs,
                                                                            rows);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "gather launch");
    count_launch(ctx);
    return RTEN_OK;
}


// 8-bit small-channel path (the quantised RGB stem): [B, Hp, Wp, 16] copy with BOTH paddings materialised (the reference
// pads u8 images with 128, which TMA's zero fill cannot produce) and channels padded to 16 bytes per pixel, so that one
// 128-byte K block = 8 pixels = one filter row and every TMA stride is a multiple of 16 bytes.
__global__ void __launch_bounds__(256)
smallc8_pad_kernel(const uint8_t* __restrict__ x, uint8_t* __restrict__ xp, int B, int C, int H, int W, int Hp, int Wp,
                   int pt, int pl, long long xs_b, long long xs_c, long long xs_h, long long xs_w, int pad_value) {
    const long long total = (long long)B * Hp * Wp;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int xw = (int)(i % Wp);
        const long long r = i / Wp;
        const int yh = (int)(r % Hp);
        const int b = (int)(r / Hp);
        const int iy = yh - pt, ix = xw - pl;
        alignas(16) uint8_t v[16];
#pragma unroll
        for (int c = 0; c < 16; c++) v[c] = 0;
        if (iy >= 0 && iy < H && ix >= 0 && ix < W) {
            const uint8_t* src = x + (long long)b * xs_b + (long long)iy * xs_h + (long long)ix * xs_w;
            for (int c = 0; c < C; c++) v[c] = src[(long long)c * xs_c];
        } else {
            for (int c = 0; c < C; c++) v[c] = (uint8_t)pad_value;
        }
        reinterpret_cast<uint4*>(xp)[i] = *reinterpret_cast<const uint4*>(v);
    }
}

// weights OIHW (any strides) -> [O, kh, 8 pixels, 16 channels], zero where kx >= kw or c >= C
__global__ void smallc8_pack_w_kernel(const uint8_t* __restrict__ w, uint8_t* __restrict__ wp, int O, int C, int kh, int kw,
                                      long long ws_o, long long ws_c, long long ws_h, long long ws_w) {
    const int total = O * kh * 128;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const int c = i & 15, kx = (i >> 4) & 7;
    const int r = i >> 7;
    const int ky = r % kh, o = r / kh;
    uint8_t v = 0;
    if (c < C && kx < kw) v = w[(long long)o * ws_o + (long long)c * ws_c + (long long)ky * ws_h + (long long)kx * ws_w];
    wp[i] = v;
}

rten_status launch_smallc8_pad(rten_ctx* ctx, const void* x, void* xp, int B, int C, int H, int W, int Hp, int Wp, int pt,
                               int pl, long long xs_b, long long xs_c, long long xs_h, long long xs_w, int pad_value) {
    const long long total = (long long)B * Hp * Wp;
    if (total == 0) return RTEN_OK;
    smallc8_pad_kernel<<<ew_grid(ctx, total), 256, 0, ctx->stream>>>((const uint8_t*)x, (uint8_t*)xp, B, C, H, W, Hp, Wp,
                                                                     pt, pl, xs_b, xs_c, xs_h, xs_w, pad_value);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "smallc8 pad launch");
    count_launch(ctx);
    return RTEN_OK;
}

rten_status launch_smallc8_pack_w(rten_ctx* ctx, const void* w, void* wp, int O, int C, int kh, int kw, long long ws_o,
                                  long long ws_c, long long ws_h, long long ws_w) {
    const int total = O * kh * 128;
    if (total == 0) return RTEN_OK;
    smallc8_pack_w_kernel<<<(total + 255) / 256, 256, 0, ctx->stream>>>((const uint8_t*)w, (uint8_t*)wp, O, C, kh, kw,
                                                                         ws_o, ws_c, ws_h, ws_w);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "smallc8 pack launch");
    count_launch(ctx);
    return RTEN_OK;
}

// ScatterElements-style row update (the KV-cache append of rten-generate when the write position lives on the device):
// table[idx[r], c] = src[r, c].  Rows named by `idx` must be distinct.
__global__ void __launch_bounds__(256)
scatter_rows_kernel(float* __restrict__ table, const int* __restrict__ idx, const float* __restrict__ src, long long nidx,
                    int width, long long t_rs, long long t_cs, long long s_rs, long long s_cs, long long rows) {
    const long long total = nidx * width;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const long long r = i / width;
        const int c = (int)(i % width);
        long long id = idx[r];
        if (id < 0) id += rows;
        if (id >= 0 && id < rows) table[id * t_rs + c * t_cs] = src[r * s_rs + c * s_cs];
    }
}

rten_status launch_scatter_rows(rten_ctx* ctx, float* table, const int* idx, const float* src, long long nidx, int width,
                                long long t_rs, long long t_cs, long long s_rs, long long s_cs, long long rows) {
    if (nidx * width == 0) return RTEN_OK;
    scatter_rows_kernel<<<ew_grid(ctx, nidx * width), 256, 0, ctx->stream>>>(table, idx, src, nidx, width, t_rs, t_cs,
                                                                             s_rs, s_cs, rows);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "scatter launch");
    count_launch(ctx);
    return RTEN_OK;
}

// =========================================================================================
// 3xTF32 operand split (RTEN_F32_TF32X3): x = hi + lo with hi = x truncated to TF32 (low 13 mantissa bits cleared,
// exactly what kind::tf32 reads) and lo = x - hi (exact in f32).  The tensor-core product over a reduction dimension
// that holds [lo | hi | hi] for one operand and [hi | lo | hi] for the other is
//     sum a_lo*b_hi + a_hi*b_lo + a_hi*b_hi      (a_lo*b_lo ~ 2^-22 |ab| dropped)
// i.e. an f32-accurate product from three TF32 passes, small terms first.  Source: rank-4 tensor with inner stride 1;
// destination: contiguous [d3][d2][d1][3 * d0p], each third zero-padded from d0 to d0p elements.
// =========================================================================================
struct SplitParams {
    long long d0, d0p, d1, d2, d3;
    long long s1, s2, s3;  // source strides (elements) of dims 1..3
    long long n;           // d3 * d2 * d1 * d0p
    int role;              // 0: [lo | hi | hi] (A operand), 1: [hi | lo | hi] (B operand), 2: [lo] only (two-plane A)
};

__global__ void __launch_bounds__(256) tf32x3_split_kernel(const float* __restrict__ x, float* __restrict__ y, const SplitParams p) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < p.n; i += stride) {
        const long long c = i % p.d0p;
        long long r = i / p.d0p;
        const long long i1 = r % p.d1;
        r /= p.d1;
        const long long i2 = r % p.d2, i3 = r / p.d2;
        float v = 0.0f;
        if (c < p.d0) v = x[i3 * p.s3 + i2 * p.s2 + i1 * p.s1 + c];
        const float hi = __uint_as_float(__float_as_uint(v) & 0xffffe000u);
        const float lo = __fsub_rn(v, hi);
        if (p.role == 2) {
            y[((i3 * p.d2 + i2) * p.d1 + i1) * p.d0p + c] = lo;
            continue;
        }
        float* row = y + ((i3 * p.d2 + i2) * p.d1 + i1) * (3 * p.d0p);
        row[c] = p.role == 0 ? lo : hi;
        row[p.d0p + c] = p.role == 0 ? hi : lo;
        row[2 * p.d0p + c] = hi;
    }
}

// 128-bit variant: one float4 of the (padded) inner dimension per thread, 32-bit index arithmetic
__global__ void __launch_bounds__(256) tf32x3_split_vec_kernel(const float* __restrict__ x, float* __restrict__ y, const SplitParams p) {
    const unsigned q0 = (unsigned)(p.d0p >> 2), d1 = (unsigned)p.d1, d2 = (unsigned)p.d2;
    const unsigned n4 = (unsigned)(p.n >> 2);
    const unsigned stride = gridDim.x * blockDim.x;
    for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += stride) {
        const unsigned c4 = i % q0;
        unsigned r = i / q0;
        const unsigned i1 = r % d1;
        r /= d1;
        const unsigned i2 = r % d2, i3 = r / d2;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if ((long long)c4 * 4 < p.d0) v = *reinterpret_cast<const float4*>(x + (long long)i3 * p.s3 + (long long)i2 * p.s2 + (long long)i1 * p.s1 + c4 * 4);
        float4 hi, lo;
        hi.x = __uint_as_float(__float_as_uint(v.x) & 0xffffe000u);
        hi.y = __uint_as_float(__float_as_uint(v.y) & 0xffffe000u);
        hi.z = __uint_as_float(__float_as_uint(v.z) & 0xffffe000u);
        hi.w = __uint_as_float(__float_as_uint(v.w) & 0xffffe000u);
        lo = make_float4(__fsub_rn(v.x, hi.x), __fsub_rn(v.y, hi.y), __fsub_rn(v.z, hi.z), __fsub_rn(v.w, hi.w));
        if (p.role == 2) {
            reinterpret_cast<float4*>(y)[i] = lo;
            continue;
        }
        float4* row = reinterpret_cast<float4*>(y + (long long)(i / q0) * (3 * p.d0p)) + c4;
        row[0] = p.role == 0 ? lo : hi;
        row[q0] = p.role == 0 ? hi : lo;
        row[2 * q0] = hi;
    }
}

// low parts of a DENSE tensor (role 2, no padding): a flat stream, 4 x 128 bits per lane and iteration, all loads of a warp
// coalesced and in flight together -- no index arithmetic (the strided kernel spends ~40 integer instructions per float4
// on its divisions, which caps it near 2.5 TB/s)
__global__ void __launch_bounds__(256) tf32x3_lo_flat_kernel(const float4* __restrict__ x, float4* __restrict__ y, long long n4) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    const long long nblk = n4 >> 7;  // 128 float4 per warp and iteration
    auto lo4 = [](float4 v) {
        float4 h;
        h.x = __uint_as_float(__float_as_uint(v.x) & 0xffffe000u);
        h.y = __uint_as_float(__float_as_uint(v.y) & 0xffffe000u);
        h.z = __uint_as_float(__float_as_uint(v.z) & 0xffffe000u);
        h.w = __uint_as_float(__float_as_uint(v.w) & 0xffffe000u);
        return make_float4(__fsub_rn(v.x, h.x), __fsub_rn(v.y, h.y), __fsub_rn(v.z, h.z), __fsub_rn(v.w, h.w));
    };
    for (long long b = warp; b < nblk; b += nwarps) {
        const float4* xp = x + (b << 7) + lane;
        const float4 v0 = xp[0], v1 = xp[32], v2 = xp[64], v3 = xp[96];
        float4* yp = y + (b << 7) + lane;
        yp[0] = lo4(v0);
        yp[32] = lo4(v1);
        yp[64] = lo4(v2);
        yp[96] = lo4(v3);
    }
    for (long long i = (nblk << 7) + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) y[i] = lo4(x[i]);
}

rten_status launch_tf32x3_split(rten_ctx* ctx, const float* x, float* y, const long long dims[4], const long long strides[4],
                                long long d0p, int role) {
    SplitParams p;
    p.d0 = dims[0];
    p.d0p = d0p;
    p.d1 = dims[1];
    p.d2 = dims[2];
    p.d3 = dims[3];
    p.s1 = strides[1];
    p.s2 = strides[2];
    p.s3 = strides[3];
    p.n = p.d3 * p.d2 * p.d1 * p.d0p;
    p.role = role;
    if (p.n == 0) return RTEN_OK;
    const bool dense = role == 2 && p.d0 == p.d0p && (p.d0 & 3) == 0 && (p.d1 == 1 || p.s1 == p.d0) && (p.d2 == 1 || p.s2 == p.d0 * p.d1) &&
                       (p.d3 == 1 || p.s3 == p.d0 * p.d1 * p.d2) && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
                       (reinterpret_cast<uintptr_t>(y) & 15) == 0;
    if (dense) {
        tf32x3_lo_flat_kernel<<<ew_grid(ctx, p.n / 16), 256, 0, ctx->stream>>>(reinterpret_cast<const float4*>(x), reinterpret_cast<float4*>(y), p.n / 4);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail_cuda(ctx, e, "tf32x3 split launch");
        count_launch(ctx);
        return RTEN_OK;
    }
    const bool vec = (p.d0 & 3) == 0 && (p.d0p & 3) == 0 && (p.s1 & 3) == 0 && (p.s2 & 3) == 0 && (p.s3 & 3) == 0 &&
                     (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 && p.n < 0x7fffffffLL;
    if (vec)
        tf32x3_split_vec_kernel<<<ew_grid(ctx, p.n / 4), 256, 0, ctx->stream>>>(x, y, p);
    else
        tf32x3_split_kernel<<<ew_grid(ctx, p.n), 256, 0, ctx->stream>>>(x, y, p);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "tf32x3 split launch");
    count_launch(ctx);
    return RTEN_OK;
}

}  // namespace rtb
