// Skinny-M kernels for autoregressive decode: HBM-streaming vector-matrix products with the surrounding operators fused
// in, and single-query attention over a KV cache.  See skinny.h.
//
// These replace, for M <= 16 (int8) / M <= 32 (f32) rows, the reference's gemv path (rten-gemm/src/lib.rs:668-747,
// rten-gemm/src/kernels/simd_generic.rs:14-197,795-1129): the weight matrix is read exactly once from HBM with
// 128-bit loads, the activations sit in shared memory, and there is no tensor-core tile to pad M up to.
#include <cuda_runtime.h>

#include <algorithm>
#include <cfloat>
#include <cstdint>
#include <cstdlib>

#include "math.cuh"
#include "rowmath.cuh"
#include "skinny.h"

namespace rtb {

namespace {

__device__ __forceinline__ int dp4a_us(unsigned a, unsigned b, int c) {
    int d;
    asm("dp4a.u32.s32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ int dp4a_uu(unsigned a, unsigned b, int c) {
    unsigned d;
    asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"((unsigned)c));
    return (int)d;
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

// Sum of v[i] over the 32 lanes for NV values with ~NV shuffles instead of 5 NV: at every step a lane hands half of
// its values to its partner and keeps (and accumulates) the other half.  On return lane `l` holds `nout` complete sums,
// v[0 .. nout), of the indices base .. base + nout - 1.  Integer or float; the float order is fixed (deterministic).
template <int NV, typename T>
__device__ __forceinline__ void reduce_scatter_warp(T (&v)[NV], int lane, int& base, int& nout) {
    base = 0;
    int n = NV;
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        if (n > 1) {
            const int half = n >> 1;
            const bool upper = (lane & o) != 0;
#pragma unroll
            for (int i = 0; i < NV / 2; i++) {
                if (i < half) {
                    const T send = upper ? v[i] : v[i + half];
                    const T keep = upper ? v[i + half] : v[i];
                    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
                }
            }
            if (upper) base += half;
            n = half;
        } else {
            v[0] = v[0] + __shfl_xor_sync(0xffffffffu, v[0], o);
        }
    }
    nout = n;
}

}  // namespace

// =========================================================================================
// Fused [LayerNorm] -> DynamicQuantizeLinear -> int8 GEMV -> scale / bias / residual / activation
//
// Everything here is latency, not throughput (a decode step moves a few megabytes): the kernel is organised so that
// every long-latency access is issued as early as its address is known -- the weight tile of a warp (CPW columns x K
// bytes, <= 16 x 16 bytes per lane) is loaded into REGISTERS before the kernel even waits for its predecessor (the
// weights do not depend on it), the next tile's weights and epilogue vectors are loaded while the current tile is
// multiplied, LayerNorm's gamma / beta are requested together with the row.
// =========================================================================================
struct QLinearParams {
    QLinearLaunch L;
    int tiles;  // column tiles of 8 * CPW columns
};

__device__ __forceinline__ uint32_t quant4(float4 a, float inv, int zp) {
    return (uint32_t)quant1(a.x, inv, zp) | ((uint32_t)quant1(a.y, inv, zp) << 8) | ((uint32_t)quant1(a.z, inv, zp) << 16) |
           ((uint32_t)quant1(a.w, inv, zp) << 24);
}

// One row of x, layer-normalised, as float4s in the vector-LayerNorm mapping (32 lanes per row): thread
// (c = lane & 15, seg = lane >> 4) holds the float4s f = c + 16 (seg F + k), k < F = K / 128 <= 8.  Same arithmetic
// as layer_norm_vec_kernel<2, .> (rowops.cu), so the values equal the LayerNormalization operator's bit for bit.
template <int FLN>
__device__ __forceinline__ void qlin_ln_row(const QLinearLaunch& L, int r, int lane, float4 (&v)[FLN]) {
    const int c = lane & 15, seg = lane >> 4;
    const int F = L.K >> 7;
    const float4* x4 = reinterpret_cast<const float4*>(L.x + (long long)r * L.xs);
    const float4* g4 = reinterpret_cast<const float4*>(L.ln_gamma);
    const float4* b4 = reinterpret_cast<const float4*>(L.ln_beta);
    float4 g[FLN], bt[FLN];
#pragma unroll
    for (int k = 0; k < FLN; k++)
        if (k < F) v[k] = x4[c + 16 * (seg * F + k)];
#pragma unroll
    for (int k = 0; k < FLN; k++) {  // requested now, needed after the two reductions
        if (k < F) {
            g[k] = __ldg(g4 + c + 16 * (seg * F + k));
            if (L.ln_beta) bt[k] = __ldg(b4 + c + 16 * (seg * F + k));
        }
    }
    const float mean = __fdiv_rn(ln_vec_fold<2, false, FLN>(v, F, 0.0f, c, seg), (float)L.K);
    const float var = __fdiv_rn(ln_vec_fold<2, true, FLN>(v, F, mean, c, seg), (float)L.K);
    const float rstd = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(var, L.ln_eps)));
#pragma unroll
    for (int k = 0; k < FLN; k++) {
        if (k < F) {
            const float4 a = v[k];
            if (!L.ln_beta) {  // (same arm as layer_norm_vec_kernel's mode 1)
                v[k] = make_float4(__fmul_rn(__fsub_rn(a.x, mean), __fmul_rn(g[k].x, rstd)), __fmul_rn(__fsub_rn(a.y, mean), __fmul_rn(g[k].y, rstd)),
                                   __fmul_rn(__fsub_rn(a.z, mean), __fmul_rn(g[k].z, rstd)), __fmul_rn(__fsub_rn(a.w, mean), __fmul_rn(g[k].w, rstd)));
            } else {  // (mode 2: beta + the scalar bias 0.0)
                v[k] = make_float4(__fmaf_rn(__fsub_rn(a.x, mean), __fmul_rn(g[k].x, rstd), __fadd_rn(bt[k].x, 0.0f)),
                                   __fmaf_rn(__fsub_rn(a.y, mean), __fmul_rn(g[k].y, rstd), __fadd_rn(bt[k].y, 0.0f)),
                                   __fmaf_rn(__fsub_rn(a.z, mean), __fmul_rn(g[k].z, rstd), __fadd_rn(bt[k].z, 0.0f)),
                                   __fmaf_rn(__fsub_rn(a.w, mean), __fmul_rn(g[k].w, rstd), __fadd_rn(bt[k].w, 0.0f)));
            }
        }
    }
}

// The (row m, column offset j) whose complete sum lane `lane` holds after reduce_scatter_warp<NV> (a function of the
// lane number only), so that the epilogue vectors of that output can be requested together with the weights.
template <int NV>
__device__ __forceinline__ int scatter_base(int lane) {
    int base = 0, n = NV;
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) {
        if (n > 1) {
            n >>= 1;
            if (lane & o) base += n;
        }
    }
    return base;
}

// Registers of one column tile of a warp: the weights (KI x CPW 16-byte chunks per lane) and the per-output epilogue
// operands of the (at most two) outputs this lane will finish.
template <int MT, int CPW, int KI>
struct QTile {
    static constexpr int NV = MT * CPW;
    static constexpr int NOUT = NV > 32 ? NV / 32 : 1;
    uint4 w[KI][CPW];
    int colsum[NOUT];
    float wscale[NOUT], bias[NOUT], res[NOUT];
    unsigned zb[NOUT];

    __device__ __forceinline__ void load(const QLinearLaunch& L, int n0, int lane, int base) {
        const uint8_t* wp = reinterpret_cast<const uint8_t*>(L.w);
        const int KC = L.K >> 4;
#pragma unroll
        for (int it = 0; it < KI; it++) {
            const int c = lane + 32 * it;
#pragma unroll
            for (int j = 0; j < CPW; j++) {
                const int n = n0 + j < L.N ? n0 + j : L.N - 1;  // (clamped: the duplicate column is never stored)
                w[it][j] = (c < KC && n0 < L.N) ? __ldg(reinterpret_cast<const uint4*>(wp + (long long)n * L.ldw) + c) : make_uint4(0u, 0u, 0u, 0u);
            }
        }
#pragma unroll
        for (int i = 0; i < NOUT; i++) {
            const int idx = base + i;
            const int m = idx / CPW, n = n0 + idx % CPW;
            const bool ok = m < L.M && n < L.N;
            colsum[i] = ok ? __ldg(L.colsum + n) : 0;
            wscale[i] = ok ? __ldg(L.w_scale + (L.w_scale_len == 1 ? 0 : n)) : 0.0f;
            bias[i] = (ok && L.bias) ? __ldg(L.bias + n) : 0.0f;
            zb[i] = (ok && L.zb) ? (unsigned)__ldg(L.zb + (L.zb_len == 1 ? 0 : n)) : 0u;
        }
    }
    // the residual is written by the predecessor kernel: only after griddepcontrol.wait
    __device__ __forceinline__ void load_residual(const QLinearLaunch& L, int n0, int base) {
#pragma unroll
        for (int i = 0; i < NOUT; i++) {
            const int idx = base + i;
            const int m = idx / CPW, n = n0 + idx % CPW;
            res[i] = (L.residual && m < L.M && n < L.N) ? L.residual[(long long)m * L.rs + n] : 0.0f;
        }
    }
};

template <int MT, int CPW, int KI, bool WSIGNED>
__device__ __forceinline__ void qlin_tile(const QLinearLaunch& L, QTile<MT, CPW, KI>& t, const uint4* aq4, const int* s_rowsum,
                                          int n0, int lane, int base, float x_scale, int zp) {
    constexpr int NV = MT * CPW;
    const int KC = L.K >> 4;
    int acc[NV];
#pragma unroll
    for (int i = 0; i < NV; i++) acc[i] = 0;
#pragma unroll
    for (int it = 0; it < KI; it++) {
        const int c = lane + 32 * it;
        if (c < KC) {
#pragma unroll
            for (int m = 0; m < MT; m++) {
                const uint4 av = aq4[m * KC + c];
#pragma unroll
                for (int j = 0; j < CPW; j++) {
                    int a = acc[m * CPW + j];
                    const uint4 wv = t.w[it][j];
                    if (WSIGNED) {
                        a = dp4a_us(av.x, wv.x, a);
                        a = dp4a_us(av.y, wv.y, a);
                        a = dp4a_us(av.z, wv.z, a);
                        a = dp4a_us(av.w, wv.w, a);
                    } else {
                        a = dp4a_uu(av.x, wv.x, a);
                        a = dp4a_uu(av.y, wv.y, a);
                        a = dp4a_uu(av.z, wv.z, a);
                        a = dp4a_uu(av.w, wv.w, a);
                    }
                    acc[m * CPW + j] = a;
                }
            }
        }
    }
    int b2, nout;
    reduce_scatter_warp<NV>(acc, lane, b2, nout);
    // ---- epilogue: lane holds the exact i32 dot products of (m, j) = divmod(base + i, CPW)
#pragma unroll
    for (int i = 0; i < QTile<MT, CPW, KI>::NOUT; i++) {
        const int idx = base + i;
        const int m = idx / CPW, n = n0 + idx % CPW;
        if (m < L.M && n < L.N) {
            // C = acc - za*colsum[n] - zb[n]*(rowsum[m] - K*za), wrapping 32-bit (rten-gemm/src/kernels/simd_generic.rs:676-746)
            unsigned cval = (unsigned)acc[i] - (unsigned)zp * (unsigned)t.colsum[i];
            if (L.zb) cval -= t.zb[i] * ((unsigned)s_rowsum[m] - (unsigned)L.K * (unsigned)zp);
            // Mul(x_scale, w_scale), cast * scale, Add(bias), Add(residual), activation: separate exactly rounded ops
            const float sc = __fmul_rn(x_scale, t.wscale[i]);
            float xv = __fmul_rn(__int2float_rn((int)cval), sc);
            if (L.bias) xv = __fadd_rn(xv, t.bias[i]);
            if (L.residual) xv = __fadd_rn(xv, t.res[i]);
            L.out[(long long)m * L.os + n] = apply_act(xv, L.act);
        }
    }
}

template <int MT, int CPW, int KI, bool WSIGNED, int FLN, bool DB>
__global__ void __launch_bounds__(256, 2) qlinear_kernel(const QLinearParams p) {
    extern __shared__ __align__(16) uint8_t sm_raw[];
    const QLinearLaunch& L = p.L;
    const int K = L.K, M = L.M;
    uint8_t* aq = sm_raw;  // [MT][K]
    int* s_rowsum = reinterpret_cast<int*>(aq + (size_t)MT * K);
    float* s_lo = reinterpret_cast<float*>(s_rowsum + MT);
    float* s_hi = s_lo + 8;
    int* s_mm = reinterpret_cast<int*>(s_hi + 8);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr int NT = 8 * CPW;
    const int base = scatter_base<MT * CPW>(lane);
    const int G = gridDim.x;

    // the weights do not depend on the previous kernel: this warp's first tile is on its way before we wait for it
    QTile<MT, CPW, KI> t0;
    int tile = blockIdx.x;
    t0.load(L, tile * NT + warp * CPW, lane, base);
    pdl_wait();
    pdl_launch_dependents();
    t0.load_residual(L, tile * NT + warp * CPW, base);

    // ---- range of the (normalised) input, then quantisation into shared memory (rows >= M are zero)
    uint32_t* aq32 = reinterpret_cast<uint32_t*>(aq);
    const int k4 = K >> 2;
    float lo = __int_as_float(0x7f800000), hi = __int_as_float(0xff800000);
    float4 v[FLN];
    if (L.has_ln) {
        const int F = K >> 7;
        for (int r = warp; r < M; r += 8) {
            qlin_ln_row<FLN>(L, r, lane, v);
#pragma unroll
            for (int k = 0; k < FLN; k++) {
                if (k < F) {
                    lo = fminf(fminf(lo, v[k].x), fminf(v[k].y, fminf(v[k].z, v[k].w)));
                    hi = fmaxf(fmaxf(hi, v[k].x), fmaxf(v[k].y, fmaxf(v[k].z, v[k].w)));
                }
            }
        }
    } else {
        for (int i = tid; i < M * k4; i += 256) {
            const int r = i / k4, f = i - r * k4;
            const float4 a = reinterpret_cast<const float4*>(L.x + (long long)r * L.xs)[f];
            lo = fminf(fminf(lo, a.x), fminf(a.y, fminf(a.z, a.w)));
            hi = fmaxf(fmaxf(hi, a.x), fmaxf(a.y, fmaxf(a.z, a.w)));
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if (lane == 0) {
        s_lo[warp] = lo;
        s_hi[warp] = hi;
    }
    __syncthreads();
    if (tid == 0) {
        for (int k = 1; k < 8; k++) {
            lo = fminf(lo, s_lo[k]);
            hi = fmaxf(hi, s_hi[k]);
        }
        s_mm[0] = float_to_ordered(lo);
        s_mm[1] = float_to_ordered(hi);
    }
    __syncthreads();
    float x_scale, inv;
    int zp;
    dql_params(s_mm, x_scale, inv, zp);
    if (L.has_ln) {
        const int c = lane & 15, seg = lane >> 4, F = K >> 7;
        for (int r = warp; r < M; r += 8) {
            // (M <= 8: the row of pass 1 is still in registers; two rows per warp: recompute, same values)
            if (MT > 8) qlin_ln_row<FLN>(L, r, lane, v);
#pragma unroll
            for (int k = 0; k < FLN; k++)
                if (k < F) aq32[r * k4 + c + 16 * (seg * F + k)] = quant4(v[k], inv, zp);
        }
    } else {
        for (int i = tid; i < M * k4; i += 256) {
            const int r = i / k4, f = i - r * k4;
            aq32[i] = quant4(reinterpret_cast<const float4*>(L.x + (long long)r * L.xs)[f], inv, zp);
        }
    }
    for (int i = M * k4 + tid; i < MT * k4; i += 256) aq32[i] = 0u;
    __syncthreads();
    if (L.zb) {  // row sums of the quantised activations for the weight-zero-point term
        for (int r = warp; r < MT; r += 8) {
            int s = 0;
            for (int i = lane; i < k4; i += 32) s = dp4a_uu(aq32[r * k4 + i], 0x01010101u, s);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
            if (lane == 0) s_rowsum[r] = s;
        }
        __syncthreads();
    }

    // ---- GEMV.  DB (wide outputs, several tiles per CTA): tiles double-buffered in registers -- tile t + G is requested
    // before tile t is multiplied.  Otherwise one tile per CTA (the launcher sizes the grid so) and half the registers,
    // which lets the CTAs of the NEXT kernel become resident (and fetch their weights) while this one still runs.
    const uint4* aq4 = reinterpret_cast<const uint4*>(aq);
    if (!DB) {
        while (tile < p.tiles) {
            qlin_tile<MT, CPW, KI, WSIGNED>(L, t0, aq4, s_rowsum, tile * NT + warp * CPW, lane, base, x_scale, zp);
            tile += G;
            if (tile < p.tiles) {
                t0.load(L, tile * NT + warp * CPW, lane, base);
                t0.load_residual(L, tile * NT + warp * CPW, base);
            }
        }
        return;
    }
    QTile<MT, CPW, KI> t1;
    while (tile < p.tiles) {
        int nxt = tile + G;
        if (nxt < p.tiles) {
            t1.load(L, nxt * NT + warp * CPW, lane, base);
            t1.load_residual(L, nxt * NT + warp * CPW, base);
        }
        qlin_tile<MT, CPW, KI, WSIGNED>(L, t0, aq4, s_rowsum, tile * NT + warp * CPW, lane, base, x_scale, zp);
        tile = nxt;
        if (tile >= p.tiles) break;
        nxt = tile + G;
        if (nxt < p.tiles) {
            t0.load(L, nxt * NT + warp * CPW, lane, base);
            t0.load_residual(L, nxt * NT + warp * CPW, base);
        }
        qlin_tile<MT, CPW, KI, WSIGNED>(L, t1, aq4, s_rowsum, tile * NT + warp * CPW, lane, base, x_scale, zp);
        tile = nxt;
    }
}

static void qlinear_shape(const QLinearLaunch& L, int& mt, int& cpw, int& ki) {
    mt = L.M <= 8 ? 8 : 16;
    const int kc = L.K >> 4;
    ki = kc <= 64 ? 2 : 6;
    // columns per warp: more bytes in flight per SM for wide outputs, fewer for narrow ones so that the tiles cover the SMs
    cpw = ki == 6 ? 1 : (L.N >= 8192 ? 4 : (L.N >= 2048 ? 2 : 1));
}

bool qlinear_supported(const QLinearLaunch& L) {
    if (getenv("RTEN_B200_NO_SKINNY")) return false;
    if (L.M < 1 || L.M > 16 || L.N < 1 || L.K < 16 || (L.K & 15)) return false;
    if ((L.K >> 4) > 192) return false;  // weights of a tile live in registers: K <= 3072
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    if (!al16(L.x) || (L.xs & 3) || !al16(L.w) || (L.ldw & 15)) return false;
    if (L.has_ln && ((L.K & 127) || (L.K >> 7) > 8 || !L.ln_gamma || !al16(L.ln_gamma) || !al16(L.ln_beta))) return false;
    if (!L.colsum || !L.w_scale) return false;
    return true;
}

rten_status launch_qlinear(rten_ctx* ctx, const QLinearLaunch& L) {
    QLinearParams p;
    p.L = L;
    int mt, cpw, ki;
    qlinear_shape(L, mt, cpw, ki);
    const int nt = 8 * cpw;
    p.tiles = (L.N + nt - 1) / nt;
    const int grid = cpw == 4 ? std::min(p.tiles, 2 * ctx->num_sms) : p.tiles;  // (one tile per CTA unless double-buffered)
    const size_t smem = (size_t)mt * L.K + mt * sizeof(int) + 16 * sizeof(float) + 16;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    fill_launch_attrs(cfg, attr, false);
    auto go = [&](auto kern) -> cudaError_t {
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        return cudaLaunchKernelEx(&cfg, kern, p);
    };
    cudaError_t e = cudaSuccess;
    const int fln = (L.has_ln && (L.K >> 7) > 6) ? 8 : 6;
    const int key = (mt == 16 ? 10000 : 0) + cpw * 1000 + ki * 100 + fln * 10 + (L.w_signed ? 1 : 0);
    switch (key) {
#define RTB_QL_CASE(MT_, CPW_, KI_, FLN_)                                                                                          \
    case (MT_ == 16 ? 10000 : 0) + CPW_ * 1000 + KI_ * 100 + FLN_ * 10 + 0: e = go(qlinear_kernel<MT_, CPW_, KI_, false, FLN_, (CPW_ == 4)>); break; \
    case (MT_ == 16 ? 10000 : 0) + CPW_ * 1000 + KI_ * 100 + FLN_ * 10 + 1: e = go(qlinear_kernel<MT_, CPW_, KI_, true, FLN_, (CPW_ == 4)>); break;
        RTB_QL_CASE(8, 1, 2, 6) RTB_QL_CASE(8, 2, 2, 6) RTB_QL_CASE(8, 4, 2, 6) RTB_QL_CASE(8, 1, 6, 6)
        RTB_QL_CASE(16, 1, 2, 6) RTB_QL_CASE(16, 2, 2, 6) RTB_QL_CASE(16, 4, 2, 6) RTB_QL_CASE(16, 1, 6, 6)
        RTB_QL_CASE(8, 1, 2, 8) RTB_QL_CASE(8, 2, 2, 8) RTB_QL_CASE(8, 4, 2, 8)
        RTB_QL_CASE(16, 1, 2, 8) RTB_QL_CASE(16, 2, 2, 8) RTB_QL_CASE(16, 4, 2, 8)
#undef RTB_QL_CASE
        default: return fail(ctx, RTEN_ERR_UNSUPPORTED_VALUE, "quantized linear: no kernel variant for this shape");
    }
    if (e != cudaSuccess) return fail_cuda(ctx, e, "qlinear launch");
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "qlinear launch");
    count_launch(ctx);
    return RTEN_OK;
}

// =========================================================================================
// f32 skinny GEMM (exact FMA arithmetic): A staged through shared memory in K chunks, B streamed once
// =========================================================================================
struct SkinnyF32Params {
    SkinnyF32Launch L;
    int tiles, kc;  // column tiles of 8 * CPW columns; K chunk (floats) held in shared memory
};

template <int MT, int CPW>
__global__ void __launch_bounds__(256) skinny_f32_kernel(const SkinnyF32Params p) {
    extern __shared__ __align__(16) uint8_t sm_raw[];
    const SkinnyF32Launch& L = p.L;
    float4* as4 = reinterpret_cast<float4*>(sm_raw);  // [MT][kc / 4]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    constexpr int NT = 8 * CPW;
    const int K = L.K, M = L.M, N = L.N;
    pdl_wait();
    pdl_launch_dependents();
    for (int tile = blockIdx.x; tile < p.tiles; tile += gridDim.x) {
        const int n0 = tile * NT + warp * CPW;
        float acc[MT * CPW];
#pragma unroll
        for (int i = 0; i < MT * CPW; i++) acc[i] = 0.0f;
        for (int k0 = 0; k0 < K; k0 += p.kc) {
            const int kn = min(p.kc, K - k0);  // multiple of 4
            const int q4 = kn >> 2, ld4 = p.kc >> 2;
            // this warp's slice of B for the chunk goes to registers first (kc <= 1024 floats: 8 float4 per lane and
            // column), so its latency overlaps the staging of A below
            float4 wreg[8][CPW];
#pragma unroll
            for (int it = 0; it < 8; it++) {
                const int c = lane + 32 * it;
#pragma unroll
                for (int j = 0; j < CPW; j++) {
                    const int n = n0 + j < N ? n0 + j : N - 1;
                    wreg[it][j] = (c < q4 && n0 < N) ? __ldg(reinterpret_cast<const float4*>(L.b + (long long)n * L.bs + k0) + c)
                                                     : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            }
            __syncthreads();  // the previous chunk has been consumed
            for (int i = tid; i < MT * q4; i += 256) {
                const int r = i / q4, f = i - r * q4;
                as4[r * ld4 + f] = r < M ? reinterpret_cast<const float4*>(L.a + (long long)r * L.as + k0)[f] : make_float4(0.f, 0.f, 0.f, 0.f);
            }
            __syncthreads();
            if (n0 < N) {
#pragma unroll
                for (int it = 0; it < 8; it++) {
                    const int c = lane + 32 * it;
                    if (c < q4) {
#pragma unroll
                        for (int m = 0; m < MT; m++) {
                            const float4 av = as4[m * ld4 + c];
#pragma unroll
                            for (int j = 0; j < CPW; j++) {
                                float a = acc[m * CPW + j];
                                a = __fmaf_rn(av.x, wreg[it][j].x, a);
                                a = __fmaf_rn(av.y, wreg[it][j].y, a);
                                a = __fmaf_rn(av.z, wreg[it][j].z, a);
                                a = __fmaf_rn(av.w, wreg[it][j].w, a);
                                acc[m * CPW + j] = a;
                            }
                        }
                    }
                }
            }
        }
        int base, nout;
        reduce_scatter_warp<MT * CPW>(acc, lane, base, nout);
#pragma unroll
        for (int i = 0; i < (MT * CPW + 31) / 32; i++) {
            if (i < nout) {
                const int idx = base + i;
                const int m = idx / CPW, n = n0 + idx % CPW;
                if (m < M && n < N) {
                    // same epilogue arithmetic as the tensor-core kernel: act(alpha * acc + r_scale * R + bias)
                    float xv = acc[i] * L.alpha;
                    if (L.residual) xv = fmaf(L.r_scale, L.residual[(long long)m * L.rs + n], xv);
                    if (L.bias) xv = xv + __ldg(L.bias + n);
                    L.out[(long long)m * L.os + n] = apply_act(xv, L.act);
                }
            }
        }
    }
}

bool skinny_f32_supported(const SkinnyF32Launch& L) {
    if (getenv("RTEN_B200_NO_SKINNY")) return false;
    if (L.M < 1 || L.M > 32 || L.N < 1 || L.K < 4 || (L.K & 3)) return false;
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    return al16(L.a) && al16(L.b) && !(L.as & 3) && !(L.bs & 3);
}

rten_status launch_skinny_f32(rten_ctx* ctx, const SkinnyF32Launch& L) {
    SkinnyF32Params p;
    p.L = L;
    const int mt = L.M <= 8 ? 8 : (L.M <= 16 ? 16 : 32);
    const int cpw = mt == 32 ? 1 : (L.N >= 4096 ? 2 : 1);
    const int nt = 8 * cpw;
    p.tiles = (L.N + nt - 1) / nt;
    p.kc = std::min((L.K + 3) / 4 * 4, 1024);
    const int grid = std::min(p.tiles, 2 * ctx->num_sms);
    const size_t smem = (size_t)mt * p.kc * sizeof(float);
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(256);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    fill_launch_attrs(cfg, attr, false);
    auto go = [&](auto kern) -> cudaError_t {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
        if (e != cudaSuccess) return e;
        return cudaLaunchKernelEx(&cfg, kern, p);
    };
    cudaError_t e;
    if (mt == 8)
        e = cpw == 2 ? go(skinny_f32_kernel<8, 2>) : go(skinny_f32_kernel<8, 1>);
    else if (mt == 16)
        e = cpw == 2 ? go(skinny_f32_kernel<16, 2>) : go(skinny_f32_kernel<16, 1>);
    else
        e = go(skinny_f32_kernel<32, 1>);
    if (e != cudaSuccess) return fail_cuda(ctx, e, "skinny f32 launch");
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "skinny f32 launch");
    count_launch(ctx);
    return RTEN_OK;
}

// =========================================================================================
// Single-query attention over a KV cache (flash-decoding split over the cached sequence)
//
// One CTA = one (batch, query head, split of <= 128 cached positions).  Latency organisation as above: the CTA's K rows
// (2 x 16 bytes per lane and position, <= 4 positions per lane) and, for a transposed value cache, its V rows are
// requested in one burst and consumed afterwards.
// =========================================================================================
struct AttnDecodeParams {
    AttnDecodeLaunch L;
    int nsplit;
    float* ws;  // [B * q_heads][nsplit][2 + dh]  partial (max, sum, unnormalised output)
    int* cnt;   // [B * q_heads] arrival counters (zero between launches)
};

constexpr int ATTN_CHUNK = 128;  // cached positions per CTA (eight warps; the six-warp variant covers 96)

// NW warps per CTA (8 or 6).  Registers cap the kernel at 80 per thread either way, so 256-thread CTAs run three to an SM
// (444 on the chip) and 192-thread CTAs four (592): the launcher takes the variant whose grid needs fewer waves -- GPT-2's
// 96 (batch x head) pairs over a 576-position cache are 480 CTAs of 8 warps (two waves, the second nearly empty) or 576 of 6
// (one wave).
template <int DH, int NW>
__global__ void __launch_bounds__(NW * 32, DH == 64 ? (NW == 8 ? 3 : 4) : 1) attn_decode_kernel(const AttnDecodeParams p) {
    // Every warp owns 16 consecutive cached positions of the CTA's chunk and runs the whole attention on them by itself
    // (scores, local max, exponentials, local sum, value product): no block barrier until the warps' partial
    // (max, sum, output) triples are merged -- the same merge that later combines the splits of a (batch, head).
    __shared__ __align__(16) float s_pw[NW][16];
    __shared__ float s_m[NW], s_s[NW];
    __shared__ float s_o[NW][DH];
    __shared__ int s_last;
    const AttnDecodeLaunch& L = p.L;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int bh = blockIdx.x / p.nsplit, split = blockIdx.x - bh * p.nsplit;
    const int b = bh / L.q_heads, h = bh - b * L.q_heads;
    const int group = L.q_heads / L.kv_heads;
    const int hk = h / group;
    pdl_wait();
    pdl_launch_dependents();
    int len = L.len ? L.len[b] : L.kv_cap;
    len = max(0, min(len, L.kv_cap));
    const int per = ((len + p.nsplit - 1) / p.nsplit + 3) & ~3;  // multiple of 4: 16-byte aligned rows of a transposed V
    const int l0 = min(len, split * per), l1 = min(len, l0 + per);
    const int nl = l1 - l0;      // <= ATTN_CHUNK (the launcher picks nsplit accordingly)
    const int w0 = warp * 16;    // first position of this warp inside the chunk
    float* kc = L.k + (long long)b * L.k_b + (long long)hk * L.k_h;
    float* vc = L.v + (long long)b * L.v_b + (long long)hk * L.v_h;
    const float* knew = L.k_new ? L.k_new + (long long)b * L.kn_b + (long long)hk * L.kn_h : nullptr;
    const float* vnew = L.v_new ? L.v_new + (long long)b * L.vn_b + (long long)hk * L.vn_h : nullptr;
    // ---- everything this warp will need is requested here: K rows (8 lanes per position, DH / 8 floats per lane) ...
    constexpr int PER_LANE = DH / 8;
    constexpr int NV4 = PER_LANE / 4;
    const int sub = lane >> 3, l8 = lane & 7;
    float4 kreg[4][NV4], qreg[NV4];
    const float4* q4 = reinterpret_cast<const float4*>(L.q + (long long)b * L.q_b + (long long)h * L.q_h + l8 * PER_LANE);
#pragma unroll
    for (int j = 0; j < NV4; j++) qreg[j] = q4[j];
#pragma unroll
    for (int it = 0; it < 4; it++) {
        const int i = w0 + it * 4 + sub;
        if (i < nl) {
            const int l = l0 + i;
            const float* kr = (knew && l == len - 1) ? knew : kc + (long long)l * L.k_l;  // (the new row may not be in the cache yet)
            const float4* k4 = reinterpret_cast<const float4*>(kr + l8 * PER_LANE);
#pragma unroll
            for (int j = 0; j < NV4; j++) kreg[it][j] = k4[j];
        }
    }
    // ... and its V tile.  Transposed cache [.., dh, cap]: lane = (channel row lane >> 2, float4 lane & 3 of the 16
    // positions); natural cache [.., cap, dh]: lane owns DH / 32 consecutive channels of every position.
    constexpr int DPW = DH / 8, CH = DH / 32;
    const bool vt = L.v_l == 1;
    const int dq = lane >> 2, f4 = lane & 3;
    float4 vreg[DPW];
    float vnat[16][CH];
    if (vt) {
#pragma unroll
        for (int j = 0; j < DPW; j++)
            vreg[j] = (w0 + 4 * f4 < nl) ? *reinterpret_cast<const float4*>(vc + (long long)(dq + 8 * j) * L.v_d + l0 + w0 + 4 * f4)
                                        : make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
#pragma unroll
        for (int i = 0; i < 16; i++) {
            if (w0 + i < nl) {
                const float* vr = (vnew && l0 + w0 + i == len - 1) ? vnew : vc + (long long)(l0 + w0 + i) * L.v_l;
#pragma unroll
                for (int j = 0; j < CH; j++) vnat[i][j] = vr[(long long)(lane * CH + j) * L.v_d];
            }
        }
    }
    // fused cache append: the split that owns position len - 1 writes the new key / value there (one CTA per kv head:
    // the query heads of a group share the cache row; every reader of that position takes k_new / v_new instead)
    if (knew && len > 0 && l1 == len && nl > 0 && (h % group) == 0 && tid < DH) {
        kc[(long long)(len - 1) * L.k_l + tid] = knew[tid];
        vc[(long long)(len - 1) * L.v_l + (long long)tid * L.v_d] = vnew[tid];
    }
    // ---- scores of the warp's 16 positions
    const float* mrow = L.mask ? L.mask + (long long)b * L.m_b + (long long)h * L.m_h : nullptr;
    float sc[4];
    float mw = -FLT_MAX;
#pragma unroll
    for (int it = 0; it < 4; it++) {
        const int i = w0 + it * 4 + sub;
        float s = 0.0f;
        if (i < nl) {
#pragma unroll
            for (int j = 0; j < NV4; j++) {
                s = fmaf(qreg[j].x, kreg[it][j].x, s);
                s = fmaf(qreg[j].y, kreg[it][j].y, s);
                s = fmaf(qreg[j].z, kreg[it][j].z, s);
                s = fmaf(qreg[j].w, kreg[it][j].w, s);
            }
        }
        s += __shfl_xor_sync(0xffffffffu, s, 4);
        s += __shfl_xor_sync(0xffffffffu, s, 2);
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        if (i < nl) {
            s *= L.scale;
            if (mrow) s += mrow[(long long)(l0 + i) * L.m_l];
            mw = fmaxf(mw, s);
        }
        sc[it] = s;
    }
    mw = fmaxf(mw, __shfl_xor_sync(0xffffffffu, mw, 8));
    mw = fmaxf(mw, __shfl_xor_sync(0xffffffffu, mw, 16));
    // ---- exponentials (the reference's polynomial, rten-vecmath/src/exp.rs:140-191), local sum, p staged per warp
    float sw = 0.0f;
#pragma unroll
    for (int it = 0; it < 4; it++) {
        const int i = w0 + it * 4 + sub;
        const float e = i < nl ? reduced_range_exp(sc[it] - mw) : 0.0f;
        sw += e;
        if (l8 == 0) s_pw[warp][it * 4 + sub] = e;
    }
    sw += __shfl_xor_sync(0xffffffffu, sw, 8);
    sw += __shfl_xor_sync(0xffffffffu, sw, 16);
    __syncwarp();
    // ---- the warp's unnormalised output o_w[d] = sum_{its positions} p V
    if (vt) {
        const float4 p4 = reinterpret_cast<const float4*>(s_pw[warp])[f4];
        const int pbase = w0 + 4 * f4;                                                   // chunk position of component .x
        const int inew = (vnew && l1 == len) ? (len - 1 - l0) - pbase : -1;             // component that is the new position
#pragma unroll
        for (int j = 0; j < DPW; j++) {
            const int d = dq + 8 * j;
            float4 vv = vreg[j];
            if (inew >= 0 && inew < 4) {
                const float nv = vnew[d];
                if (inew == 0) vv.x = nv;
                if (inew == 1) vv.y = nv;
                if (inew == 2) vv.z = nv;
                if (inew == 3) vv.w = nv;
            }
            // (positions beyond nl hold p = 0 but their V may be uninitialised memory: never multiply it)
            float a = 0.0f;
            if (pbase < nl) a = fmaf(p4.x, vv.x, a);
            if (pbase + 1 < nl) a = fmaf(p4.y, vv.y, a);
            if (pbase + 2 < nl) a = fmaf(p4.z, vv.z, a);
            if (pbase + 3 < nl) a = fmaf(p4.w, vv.w, a);
            a += __shfl_xor_sync(0xffffffffu, a, 1);
            a += __shfl_xor_sync(0xffffffffu, a, 2);
            if (f4 == 0) s_o[warp][d] = a;
        }
    } else {
        float a[CH];
#pragma unroll
        for (int j = 0; j < CH; j++) a[j] = 0.0f;
#pragma unroll
        for (int i = 0; i < 16; i++) {
            if (w0 + i < nl) {
                const float pw = s_pw[warp][i];
#pragma unroll
                for (int j = 0; j < CH; j++) a[j] = fmaf(pw, vnat[i][j], a[j]);
            }
        }
#pragma unroll
        for (int j = 0; j < CH; j++) s_o[warp][lane * CH + j] = a[j];
    }
    if (lane == 0) {
        s_m[warp] = w0 < nl ? mw : -FLT_MAX;
        s_s[warp] = sw;
    }
    __syncthreads();
    // ---- merge the warps
    float m = -FLT_MAX, num = 0.0f, den = 0.0f;
    if (tid < DH) {
#pragma unroll
        for (int w = 0; w < NW; w++) m = fmaxf(m, s_m[w]);
#pragma unroll
        for (int w = 0; w < NW; w++) {
            const float e = reduced_range_exp(s_m[w] - m);
            den = fmaf(s_s[w], e, den);
            num = fmaf(s_o[w][tid], e, num);
        }
    }
    float* outp = L.out + (long long)b * L.o_b + (long long)h * L.o_h;
    if (p.nsplit == 1) {
        if (tid < DH) {
            float r = num / den;
            if (r != r) r = 0.0f;  // fully masked row -> zeros (sdpa_head flushes NaNs)
            outp[tid] = r;
        }
        return;
    }
    // ---- merge the splits: the last CTA of (b, h) to arrive combines the partial (max, sum, output) triples
    float* wsp = p.ws + ((long long)bh * p.nsplit + split) * (2 + DH);
    if (tid == 0) {
        wsp[0] = m;
        wsp[1] = den;
    }
    if (tid < DH) wsp[2 + tid] = num;
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const int old = atomicAdd(p.cnt + bh, 1);
        s_last = old == p.nsplit - 1;
        if (s_last) p.cnt[bh] = 0;
        __threadfence();
    }
    __syncthreads();
    if (!s_last) return;
    if (tid < DH) {
        const float* w0p = p.ws + (long long)bh * p.nsplit * (2 + DH);
        float mm = -FLT_MAX;
        for (int s2 = 0; s2 < p.nsplit; s2++) mm = fmaxf(mm, __ldcg(w0p + s2 * (2 + DH)));
        float nn = 0.0f, dd = 0.0f;
        for (int s2 = 0; s2 < p.nsplit; s2++) {
            const float* ww = w0p + s2 * (2 + DH);
            const float e = reduced_range_exp(__ldcg(ww) - mm);
            dd = fmaf(__ldcg(ww + 1), e, dd);
            nn = fmaf(__ldcg(ww + 2 + tid), e, nn);
        }
        float r = nn / dd;
        if (r != r) r = 0.0f;
        outp[tid] = r;
    }
}

bool attn_decode_supported(const AttnDecodeLaunch& L) {
    if (getenv("RTEN_B200_NO_SKINNY")) return false;
    if (L.dh != 64 && L.dh != 128) return false;
    if (L.B < 1 || L.q_heads < 1 || L.kv_heads < 1 || L.q_heads % L.kv_heads) return false;
    if (L.kv_cap < 1 || L.kv_cap > 64 * ATTN_CHUNK) return false;
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    if (!al16(L.k) || (L.k_b & 3) || (L.k_h & 3) || (L.k_l & 3)) return false;
    if (!al16(L.q) || (L.q_b & 3) || (L.q_h & 3)) return false;
    if (L.k_new && (!al16(L.k_new) || (L.kn_b & 3) || (L.kn_h & 3) || !L.v_new)) return false;
    if (L.v_l != 1 && L.v_d != 1) return false;
    if (L.v_l == 1 && (!al16(L.v) || (L.v_b & 3) || (L.v_h & 3) || (L.v_d & 3))) return false;  // float4 along the positions
    return true;
}

rten_status launch_attn_decode(rten_ctx* ctx, const AttnDecodeLaunch& L) {
    AttnDecodeParams p;
    p.L = L;
    const int bh = L.B * L.q_heads;
    // a split covers at most `chunk` positions (rounded to 4); more splits when (batch x heads) alone leaves SMs idle
    auto splits_for = [&](int chunk) {
        int ns = (L.kv_cap + chunk - 1) / chunk;
        ns = std::max(ns, std::min(16, (2 * ctx->num_sms + bh - 1) / bh));
        ns = std::max(1, std::min(ns, std::max(1, (L.kv_cap + 15) / 16)));
        while ((((L.kv_cap + ns - 1) / ns + 3) & ~3) > chunk) ns++;
        return ns;
    };
    int nw = 8, ns = splits_for(ATTN_CHUNK);
    if (L.dh == 64 && !getenv("RTEN_B200_ATTN_8WARPS")) {  // six-warp CTAs when their grid needs fewer waves (see the kernel's comment)
        const int ns6 = splits_for(96);
        const long long waves8 = ((long long)bh * ns + 3LL * ctx->num_sms - 1) / (3LL * ctx->num_sms);
        const long long waves6 = ((long long)bh * ns6 + 4LL * ctx->num_sms - 1) / (4LL * ctx->num_sms);
        if (waves6 < waves8) {
            nw = 6;
            ns = ns6;
        }
    }
    p.nsplit = ns;
    p.ws = nullptr;
    p.cnt = nullptr;
    if (ns > 1) {
        if (!ctx->attn_cnt || ctx->attn_cnt_len < bh) {
            if (ctx->attn_cnt) cudaFree(ctx->attn_cnt);
            const int cap = std::max(bh, 1024);
            cudaError_t ce = cudaMalloc(&ctx->attn_cnt, (size_t)cap * sizeof(int));
            if (ce != cudaSuccess) return fail_cuda(ctx, ce, "attention counters");
            ce = cudaMemset(ctx->attn_cnt, 0, (size_t)cap * sizeof(int));
            if (ce != cudaSuccess) return fail_cuda(ctx, ce, "attention counters");
            ctx->attn_cnt_len = cap;
        }
        void* ws = nullptr;
        RTB_TRY(temp_alloc(ctx, (size_t)bh * ns * (2 + L.dh) * sizeof(float), &ws));
        p.ws = reinterpret_cast<float*>(ws);
        p.cnt = reinterpret_cast<int*>(ctx->attn_cnt);
    }
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(bh * ns);
    cfg.blockDim = dim3(nw * 32);
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    fill_launch_attrs(cfg, attr, false);
    cudaError_t e = L.dh == 64 ? (nw == 6 ? cudaLaunchKernelEx(&cfg, attn_decode_kernel<64, 6>, p) : cudaLaunchKernelEx(&cfg, attn_decode_kernel<64, 8>, p))
                               : cudaLaunchKernelEx(&cfg, attn_decode_kernel<128, 8>, p);
    if (e != cudaSuccess) return fail_cuda(ctx, e, "attention launch");
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "attention launch");
    count_launch(ctx);
    return RTEN_OK;
}

}  // namespace rtb
