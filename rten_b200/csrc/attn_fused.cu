// Fused attention for encoder-sized sequences (BERT: 128 keys, head size 64) on tcgen05: one CTA per (batch, head,
// 128-query tile) computes  O = softmax(scale * Q K^T + mask) V  without the score matrix ever leaving the SM:
//   TMA: Q, K tiles (K-major, 128B swizzle), V^T tiles           ->  shared memory
//   tcgen05.mma kind::tf32:  S = Q K^T                            ->  TMEM columns [0, 128)
//   4 warps, one query row per thread: tcgen05.ld S, scale, + mask, the reference's softmax (rten-vecmath/src/softmax.rs:
//       60-101,176-228: ReducedRangeExp, 16 lane partial sums in index order) -> P written as the A operand (128B-swizzled
//       K-major tiles) in shared memory
//   tcgen05.mma kind::tf32:  O = P V                              ->  TMEM columns [128, 192)
//   tcgen05.ld O -> global
// Replaces, for these shapes, FusedMatMul(QK^T) + AddSoftmax + MatMul(PV) (src/ops/attention.rs:30-165, :518-560): three
// launches and two round trips of the [batch, heads, 128, 128] score tensor through HBM per layer.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cfloat>
#include <cstdint>
#include <cstdlib>
#include <cstring>

#include "attn_fused.h"
#include "math.cuh"
#include "ptx.cuh"
#include "umma_gemm.h"

namespace rtb {

namespace {

constexpr int AF_THREADS = 192;  // warps 0-3: one query row per thread; warp 4: TMA + MMA issue; warp 5: TMEM allocation
constexpr int SQ = 128, SK = 128, DH = 64;
constexpr uint32_t TILE = 128 * 128;      // a [128 rows x 32 floats] K-major tile
constexpr uint32_t VT_TILE = DH * 128;    // a [64 rows x 32 floats] tile of V^T

struct AttnFusedParams {
    int B, heads, q_tiles;
    const float* v;  // natural value tensor [b][h][s][d] (d contiguous): transposed into the V^T tiles by the kernel; null = TMA from V^T
    long long v_b, v_h, v_s;
    float scale;
    const float* mask;  // additive [B, keys] (row stride m_b) or null
    long long m_b;
    float* out;
    long long o_b, o_h, o_s;
};

__global__ void __launch_bounds__(AF_THREADS, 2)
attn_fused_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_k,
                  const __grid_constant__ CUtensorMap tma_v, const __grid_constant__ AttnFusedParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* bar_qk = reinterpret_cast<uint64_t*>(base);
    uint64_t* bar_v = bar_qk + 1;
    uint64_t* bar_s = bar_qk + 2;
    uint64_t* bar_p = bar_qk + 3;
    uint64_t* bar_o = bar_qk + 4;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bar_qk + 6);
    uint8_t* sq = base + 1024;              // 2 tiles
    uint8_t* sk = sq + 2 * TILE;            // 2 tiles
    uint8_t* sv = sk + 2 * TILE;            // 4 tiles of V^T
    uint8_t* sp = sq;                       // 4 tiles of P: over Q and K, which are dead once S = Q K^T has completed (bar_s)
                                            // -> 98 KB per CTA, two CTAs per SM: one CTA's softmax overlaps the other's TMA / MMA
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int u = blockIdx.x;
    const int qt = u % p.q_tiles, h = (u / p.q_tiles) % p.heads, b = u / (p.q_tiles * p.heads);

    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tma_q);
        tma_prefetch_desc(&tma_k);
        tma_prefetch_desc(&tma_v);
        mbar_init(bar_qk, 1);
        mbar_init(bar_v, p.v ? 4 : 1);
        mbar_init(bar_s, 1);
        mbar_init(bar_p, 4);
        mbar_init(bar_o, 1);
        fence_mbar_init();
    }
    if (warp == 5) {
        tmem_alloc(tmem_ptr, 256);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_ptr;
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

    if (warp == 4) {
        if (elect_one()) {
            mbar_expect_tx(bar_qk, 4 * TILE);
            for (int kb = 0; kb < 2; kb++) {
                tma_load_4d(sq + kb * TILE, &tma_q, bar_qk, kb * 32, qt * SQ, h, b);
                tma_load_4d(sk + kb * TILE, &tma_k, bar_qk, kb * 32, 0, h, b);
            }
            if (!p.v) {
                mbar_expect_tx(bar_v, 4 * VT_TILE);
                for (int kb = 0; kb < 4; kb++) tma_load_4d(sv + kb * VT_TILE, &tma_v, bar_v, kb * 32, 0, h, b);
            }
        }
        __syncwarp();
        // ---- S = Q K^T
        mbar_wait(bar_qk, 0);
        tc_fence_after();
        if (elect_one()) {
            const uint32_t idesc = make_idesc(1, 2, 2, 128, SK);
            for (int kb = 0; kb < 2; kb++) {
                const uint64_t ad = make_kmajor_sw128_desc(smem_u32(sq + kb * TILE)), bd = make_kmajor_sw128_desc(smem_u32(sk + kb * TILE));
#pragma unroll
                for (int k = 0; k < 4; k++) umma_tf32(tmem, ad + 2 * k, bd + 2 * k, idesc, (kb | k) ? 1u : 0u);
            }
            umma_commit(bar_s);
        }
        __syncwarp();
        // ---- O = P V
        mbar_wait(bar_p, 0);
        mbar_wait(bar_v, 0);
        tc_fence_after();
        if (elect_one()) {
            const uint32_t idesc = make_idesc(1, 2, 2, 128, DH);
            for (int kb = 0; kb < 4; kb++) {
                const uint64_t ad = make_kmajor_sw128_desc(smem_u32(sp + kb * TILE)), bd = make_kmajor_sw128_desc(smem_u32(sv + kb * VT_TILE));
#pragma unroll
                for (int k = 0; k < 4; k++) umma_tf32(tmem + 128, ad + 2 * k, bd + 2 * k, idesc, (kb | k) ? 1u : 0u);
            }
            umma_commit(bar_o);
        }
        __syncwarp();
    } else if (warp < 4) {
        // ---- one query row per thread
        const int r = warp * 32 + lane;
        const uint32_t t_row = tmem + ((uint32_t)(warp * 32) << 16);
        const float* mrow = p.mask ? p.mask + (long long)b * p.m_b : nullptr;
        if (p.v) {
            // natural V [s][d]: this thread's key row s = r goes into column r of the K-major, 128B-swizzled V^T tiles
            // (tile r / 32, row d, 16-byte chunk ((r % 32) / 4) ^ (d & 7)) while the tensor core is busy with Q K^T
            const float4* vrow = reinterpret_cast<const float4*>(p.v + (long long)b * p.v_b + (long long)h * p.v_h + (long long)r * p.v_s);
            float4 vv[DH / 4];
#pragma unroll
            for (int j = 0; j < DH / 4; j++) vv[j] = vrow[j];
            uint8_t* tile = sv + (r >> 5) * VT_TILE;
            const int col = r & 31;
#pragma unroll
            for (int j = 0; j < DH / 4; j++) {
                const float e[4] = {vv[j].x, vv[j].y, vv[j].z, vv[j].w};
#pragma unroll
                for (int t = 0; t < 4; t++) {
                    const int d = 4 * j + t;
                    *reinterpret_cast<float*>(tile + d * 128 + (((col >> 2) ^ (d & 7)) << 4) + ((col & 3) << 2)) = e[t];
                }
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_v);
        }
        float z[SK];
        mbar_wait(bar_s, 0);
        tc_fence_after();
        float mx = -FLT_MAX;
        const f32x2 sc2 = splat2(p.scale);
#pragma unroll
        for (int c = 0; c < 4; c++) {
            uint32_t v[32];
            tmem_ld_32x32(t_row + c * 32, v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
                // FusedMatMul's alpha, then AddSoftmax's z = qk + mask: two lanes per packed instruction (same roundings)
                f32x2 a = mul2(pack2(__uint_as_float(v[j]), __uint_as_float(v[j + 1])), sc2);
                f32x2 b2 = mul2(pack2(__uint_as_float(v[j + 2]), __uint_as_float(v[j + 3])), sc2);
                if (mrow) {
                    const float4 m4 = __ldg(reinterpret_cast<const float4*>(mrow + c * 32 + j));
                    a = add2(a, pack2(m4.x, m4.y));
                    b2 = add2(b2, pack2(m4.z, m4.w));
                }
                unpack2(a, z[c * 32 + j], z[c * 32 + j + 1]);
                unpack2(b2, z[c * 32 + j + 2], z[c * 32 + j + 3]);
                mx = fmaxf(fmaxf(mx, z[c * 32 + j]), fmaxf(z[c * 32 + j + 1], fmaxf(z[c * 32 + j + 2], z[c * 32 + j + 3])));
            }
        }
        // exponentials and the 16 lane partial sums, lane l owning the elements i = l (mod 16) in ascending i (pairs of lanes
        // in one packed register: the same additions in the same order)
        f32x2 part[8];
#pragma unroll
        for (int l = 0; l < 8; l++) part[l] = splat2(0.0f);
        const f32x2 nmx = splat2(-mx);
#pragma unroll
        for (int i = 0; i < SK; i += 2) {
            float e0, e1;
            unpack2(add2(pack2(z[i], z[i + 1]), nmx), e0, e1);  // z - max
            reduced_range_exp_x2(e0, e1);
            z[i] = e0;
            z[i + 1] = e1;
            part[(i & 15) >> 1] = add2(part[(i & 15) >> 1], pack2(e0, e1));
        }
        float s = 0.0f;
#pragma unroll
        for (int l = 0; l < 8; l++) {
            float a, b2;
            unpack2(part[l], a, b2);
            s = __fadd_rn(s, a);
            s = __fadd_rn(s, b2);
        }
        const f32x2 inv = splat2(__fdiv_rn(1.0f, s));
        // P as the A operand: tile c holds keys [32 c, 32 c + 32); row r = 128 bytes, 16-byte chunks XOR-swizzled by r & 7
        const int sw = r & 7;
#pragma unroll
        for (int c = 0; c < 4; c++) {
            uint8_t* rowp = sp + c * TILE + r * 128;
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int i = c * 32 + 4 * j;
                float4 o;
                unpack2(mul2(pack2(z[i], z[i + 1]), inv), o.x, o.y);
                unpack2(mul2(pack2(z[i + 2], z[i + 3]), inv), o.z, o.w);
                *reinterpret_cast<float4*>(rowp + ((j ^ sw) << 4)) = o;
            }
        }
        fence_proxy_async();  // the tensor core reads these bytes through the async proxy
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_p);
        // ---- O rows -> shared memory (the P tiles are dead once P V has completed) -> global, two whole 256-byte rows per
        // warp instruction (a thread writing its own row costs 32 half-used sectors per instruction: tools/store_probe.cu)
        mbar_wait(bar_o, 0);
        tc_fence_after();
        uint8_t* so = sp + warp * (32 * 256);  // this warp's 32 rows x 256 B
        {
            uint8_t* rowp = so + lane * 256;
#pragma unroll
            for (int c = 0; c < 2; c++) {
                uint32_t v[32];
                tmem_ld_32x32(t_row + 128 + c * 32, v);
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 8; j++)
                    *reinterpret_cast<uint4*>(rowp + c * 128 + ((j ^ (lane & 7)) << 4)) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            }
        }
        __syncwarp();
        float* obase = p.out + (long long)b * p.o_b + (long long)h * p.o_h + (long long)(qt * SQ + warp * 32) * p.o_s;
#pragma unroll
        for (int it = 0; it < 16; it++) {
            const int row = it * 2 + (lane >> 4), jj = lane & 15;
            const uint4 d = *reinterpret_cast<const uint4*>(so + row * 256 + (jj >> 3) * 128 + (((jj & 7) ^ (row & 7)) << 4));
            *reinterpret_cast<uint4*>(obase + (long long)row * p.o_s + jj * 4) = d;
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) {
        tc_fence_after();
        tmem_dealloc(tmem, 256);
    }
}

}  // namespace

bool attn_fused_supported(const AttnFusedLaunch& L) {
    if (getenv("RTEN_B200_NO_FUSED_ATTN")) return false;
    if (L.dh != DH || L.kv_seq != SK || L.q_seq < SQ || L.q_seq % SQ) return false;
    if (L.B < 1 || L.heads < 1) return false;
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    if (!al16(L.out) || (L.o_b & 3) || (L.o_h & 3) || (L.o_s & 3)) return false;
    if (L.mask && (!al16(L.mask) || (L.m_b & 3))) return false;  // the mask row is read 128 bits at a time
    // Q, K: head dimension contiguous; V: key dimension contiguous (a transposed value tensor)
    if (!tma_compatible(L.q, 4, 4) || !tma_compatible(L.k, 4, 4)) return false;
    if (L.v ? (!al16(L.v) || (L.v_b & 3) || (L.v_h & 3) || (L.v_s & 3)) : !tma_compatible(L.vt, 4, 4)) return false;
    return true;
}

rten_status launch_attn_fused(rten_ctx* ctx, const AttnFusedLaunch& L) {
    AttnFusedParams p;
    memset(&p, 0, sizeof(p));
    p.B = L.B;
    p.heads = L.heads;
    p.q_tiles = L.q_seq / SQ;
    p.scale = L.scale;
    p.mask = L.mask;
    p.m_b = L.m_b;
    p.v = L.v;
    p.v_b = L.v_b;
    p.v_h = L.v_h;
    p.v_s = L.v_s;
    p.out = L.out;
    p.o_b = L.o_b;
    p.o_h = L.o_h;
    p.o_s = L.o_s;
    uint32_t ones[4] = {1, 1, 1, 1};
    uint32_t qbox[4] = {32u, (uint32_t)SQ, 1u, 1u}, kbox[4] = {32u, (uint32_t)SK, 1u, 1u}, vbox[4] = {32u, (uint32_t)DH, 1u, 1u};
    CUtensorMap mq, mk, mv;
    if (!encode_map(ctx, &mq, L.q, 4, true, qbox, ones) || !encode_map(ctx, &mk, L.k, 4, true, kbox, ones)) return RTEN_ERR_UNSUPPORTED_VALUE;
    mv = mq;  // (unused when the kernel transposes a natural V itself)
    if (!L.v && !encode_map(ctx, &mv, L.vt, 4, true, vbox, ones)) return RTEN_ERR_UNSUPPORTED_VALUE;
    const size_t smem = 1024 + 1024 + 4 * (size_t)TILE + 4 * (size_t)VT_TILE;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(L.B * L.heads * p.q_tiles);
    cfg.blockDim = dim3(AF_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    fill_launch_attrs(cfg, attr, false);
    cudaError_t e = cudaFuncSetAttribute(attn_fused_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) e = cudaLaunchKernelEx(&cfg, attn_fused_kernel, mq, mk, mv, p);
    if (e != cudaSuccess) return fail_cuda(ctx, e, "fused attention launch");
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "fused attention launch");
    count_launch(ctx);
    return RTEN_OK;
}

}  // namespace rtb
