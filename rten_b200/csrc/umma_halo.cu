// Halo-reuse convolution on tcgen05: stride-1 convolutions with a kh x kw window (the 3x3 layers of ResNet-50).
//
// The generic implicit-GEMM kernel (umma_gemm.cu) streams one activation box per filter tap from L2: a 3x3 layer moves
// its input nine times into shared memory, and at 4 bytes per TF32 operand the L2 -> SM stream, not the tensor pipe, sets
// its pace (profiles/r01_trace_pipeline_v2.txt).  Here a CTA loads ONE zero-padded activation patch per 32-channel block
//     patch[b][y][x][32 ch]   y in [oy0 - pt, oy0 + R + kh - 1 - pt),  x in [-pl, -pl + P),  P = OW + kw - 1
// with a single TMA box (out-of-bounds -> 0 = the padding) and treats it as a LINEAR array of P-pitched pixel slots of
// 128 bytes: output slot s = y P + x reads, for tap (ky, kx), input slot s + ky P + kx.  Every tap is therefore the same
// patch seen through a shared-memory matrix descriptor whose start address is shifted by (ky P + kx) x 128 bytes -- the
// 128B swizzle is a function of the absolute shared-memory address, so TMA's layout and the shifted descriptor agree
// (measured: tools/desc_probe.cu, profiles/r02_desc_probe.txt).  Slots with x >= OW (and the rows past the strip) are
// computed and thrown away: 2 / P of the MMA rows for a 3x3 window.  The weights stream through a ring of
// stages of `tps` taps x (bn x 32 channel) tiles (one barrier hand-off per stage).
//
// Replaces rten-gemm/src/im2col.rs:110-212 (the A-operand gather of the packed GEMM) for these layers.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "math.cuh"
#include "ptx.cuh"
#include "umma_gemm.h"

namespace rtb {

namespace {

constexpr int HALO_THREADS = 384;  // warp 0 TMA, warp 1 MMA, warp 2 TMEM, warps 4-11 epilogue
constexpr int HB_MAX = 8;          // weight ring stages

struct HaloParams {
    // geometry
    int B, OH, OW, N, C;
    int kh, kw, pt, pl;
    int P;         // slot pitch of a patch row = OW + kw - 1
    int R;         // output rows per unit
    int tb;        // images per unit
    int nr;        // patch rows per image = R + kh - 1
    int T;         // 128-slot MMA tiles per unit
    int bn;        // output channels per unit
    int c_blocks;  // 32-channel blocks
    int taps;
    int strips, units_n, units_total;
    int acc_stages;     // 1 or 2 TMEM accumulator stages of T * bn columns
    int b_stages;       // weight ring depth
    int tps;            // filter taps per weight-ring stage (one barrier hand-off per stage: taps, kw or 1)
    uint32_t patch_bytes, patch_tx, b_bytes;
    uint32_t idesc;
    long long* trace;  // debug (rten_b200_debug_trace + RTEN_B200_TRACE_FAST): clock64 stamps of CTA 0, layout of the GEMM kernel's
    uint32_t tap_off[32];  // (ky P + kx) * 8: descriptor offset (16-byte units) of filter tap ky * kw + kx inside the patch
    uint32_t m_img, m_P;  // floor(2^32 / d) + 1 for d = nr * P and d = P: n / d == __umulhi(n, m) for the slot numbers of a unit
    EpilogueDesc epi;
};

// (a0, a1) += (b0, b1): one packed FADD2, each half rounded to nearest like a scalar add
__device__ __forceinline__ void add_pair(uint32_t& a0, uint32_t& a1, float b0, float b1) {
    unsigned long long a, b, d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "r"(a0), "r"(a1));
    asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    asm("mov.b64 {%0, %1}, %2;" : "=r"(a0), "=r"(a1) : "l"(d));
}

__device__ __forceinline__ void halo_unit(const HaloParams& p, int u, int& n0, int& oy0, int& b0) {
    const int nt = u % p.units_n;
    const int rest = u / p.units_n;
    const int st = rest % p.strips;
    n0 = nt * p.bn;
    oy0 = st * p.R;
    b0 = (rest / p.strips) * p.tb;
}

__global__ void __launch_bounds__(HALO_THREADS, 1)
umma_halo_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b, const __grid_constant__ HaloParams p) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    uint64_t* patch_full = reinterpret_cast<uint64_t*>(base);  // [2]
    uint64_t* patch_empty = patch_full + 2;
    uint64_t* b_full = patch_empty + 2;                         // [HB_MAX]
    uint64_t* b_empty = b_full + HB_MAX;
    uint64_t* tmem_full = b_empty + HB_MAX;                     // [2]
    uint64_t* tmem_empty = tmem_full + 2;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);
    float* bias_s = reinterpret_cast<float*>(base + 1024);  // [2 groups][128]: column bias of the current unit
    uint8_t* stage0 = base + 2048;                             // [2 groups] 128 slots x 128 B output staging (128B-swizzled)
    uint8_t* patch0 = stage0 + 2 * 16384;
    uint8_t* bring = patch0 + 2 * (size_t)p.patch_bytes;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    const bool tr0 = p.trace && blockIdx.x == 0;
    if (tr0 && threadIdx.x == 0) p.trace[6144 + 1100] = clock64();
    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tma_a);
        tma_prefetch_desc(&tma_b);
    }
    if (warp == 1) {
        if (lane < 2) {
            mbar_init(&patch_full[lane], 1);
            mbar_init(&patch_empty[lane], 1);
            mbar_init(&tmem_full[lane], 1);
            mbar_init(&tmem_empty[lane], 8);  // one arrival per epilogue warp
        }
        if (lane < HB_MAX) {
            mbar_init(&b_full[lane], 1);
            mbar_init(&b_empty[lane], 1);
        }
        fence_mbar_init();
    }
    if (warp == 2) {
        tmem_alloc(tmem_ptr, 512);
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    if (tr0 && threadIdx.x == 0) p.trace[6144 + 1101] = clock64();
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (tr0 && threadIdx.x == 0) p.trace[6144 + 1102] = clock64();

    if (warp == 0) {
        // ===================== TMA producer =====================
        uint32_t pphase = 0, bphase = 0;  // bit s = uses of stage s so far, mod 2
        int ps = 0, bs = 0, tr_p = 0;
        for (int u = blockIdx.x; u < p.units_total; u += gridDim.x) {
            int n0, oy0, b0;
            halo_unit(p, u, n0, oy0, b0);
            for (int cb = 0; cb < p.c_blocks; cb++) {
                mbar_wait(&patch_empty[ps], ((pphase >> ps) & 1) ^ 1);
                if (elect_one()) {
                    mbar_expect_tx(&patch_full[ps], p.patch_tx);
                    tma_load_4d(patch0 + (size_t)ps * p.patch_bytes, &tma_a, &patch_full[ps], cb * 32, -p.pl, oy0 - p.pt, b0);
                }
                __syncwarp();
                pphase ^= 1u << ps;
                ps ^= 1;
                for (int tap = 0; tap < p.taps; tap += p.tps) {
                    mbar_wait(&b_empty[bs], ((bphase >> bs) & 1) ^ 1);
                    if (elect_one()) {
                        if (tr0 && tr_p < 2048) p.trace[tr_p++] = clock64();
                        mbar_expect_tx(&b_full[bs], p.b_bytes);
                        tma_load_4d(bring + (size_t)bs * p.b_bytes, &tma_b, &b_full[bs], cb * 32, n0, tap, 0);  // box: tps taps
                    }
                    __syncwarp();
                    bphase ^= 1u << bs;
                    if (++bs == p.b_stages) bs = 0;
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        uint32_t pphase = 0, bphase = 0, aphase = 0;
        int ps = 0, bs = 0, it = 0, tr_m = 0;
        // debug trace: where the issuing warp's clocks go (registers; written once at the end)
        long long c_acc = 0, c_patch = 0, c_b = 0, c_issue = 0, c_commit = 0, n_mma = 0, tq = 0;
        if (tr0) tq = clock64();
#define HALO_LAP(var)                    \
    if (tr0) {                           \
        const long long now = clock64(); \
        var += now - tq;                 \
        tq = now;                        \
    }
        for (int u = blockIdx.x; u < p.units_total; u += gridDim.x, it++) {
            const int acc = p.acc_stages == 2 ? (it & 1) : 0;
            mbar_wait(&tmem_empty[acc], ((aphase >> acc) & 1) ^ 1);
            aphase ^= 1u << acc;
            tc_fence_after();
            HALO_LAP(c_acc)
            const uint32_t d_tmem = tmem_base + acc * 256;
            for (int cb = 0; cb < p.c_blocks; cb++) {
                mbar_wait(&patch_full[ps], (pphase >> ps) & 1);
                HALO_LAP(c_patch)
                const uint64_t adesc0 = make_kmajor_sw128_desc(smem_u32(patch0 + (size_t)ps * p.patch_bytes));
                for (int tap0 = 0; tap0 < p.taps; tap0 += p.tps) {
                    mbar_wait(&b_full[bs], (bphase >> bs) & 1);
                    tc_fence_after();
                    HALO_LAP(c_b)
                    if (elect_one()) {
                        if (tr0 && tr_m < 2048) p.trace[2048 + tr_m++] = tq;
                        const uint64_t bdesc0 = make_kmajor_sw128_desc(smem_u32(bring + (size_t)bs * p.b_bytes));
                        for (int ti = 0; ti < p.tps; ti++) {
                            // the tap is the SAME patch seen (ky P + kx) pixel slots of 128 bytes further on (descriptor
                            // addresses count 16-byte units; offsets tabulated on the host -- an integer division per tap
                            // costs the single issuing thread ~200 clk)
                            const uint64_t adesc = adesc0 + (uint64_t)p.tap_off[tap0 + ti];
                            const uint64_t bdesc = bdesc0 + (uint64_t)(ti * p.bn * 8);
                            const uint32_t first = (cb | tap0 | ti) ? 1u : 0u;
                            for (int t = 0; t < p.T; t++) {
#pragma unroll
                                for (int k = 0; k < 4; k++)
                                    umma_tf32(d_tmem + t * p.bn, adesc + (uint64_t)(t * 1024 + 2 * k), bdesc + 2 * k, p.idesc, (first | (uint32_t)k) ? 1u : 0u);
                            }
                        }
                    }
                    __syncwarp();
                    HALO_LAP(c_issue)
                    n_mma += p.tps * p.T * 4;
                    if (elect_one()) {
                        umma_commit(&b_empty[bs]);
                        if (tap0 + p.tps >= p.taps) {
                            umma_commit(&patch_empty[ps]);
                            if (cb == p.c_blocks - 1) umma_commit(&tmem_full[acc]);
                        }
                    }
                    __syncwarp();
                    bphase ^= 1u << bs;
                    if (++bs == p.b_stages) bs = 0;
                    HALO_LAP(c_commit)
                }
                pphase ^= 1u << ps;
                ps ^= 1;
            }
        }
#undef HALO_LAP
        if (tr0 && lane == 0) {
            p.trace[6144 + 1030] = c_issue;
            p.trace[6144 + 1031] = n_mma;
            p.trace[6144 + 1032] = c_acc;
            p.trace[6144 + 1033] = c_patch;
            p.trace[6144 + 1034] = c_b;
            p.trace[6144 + 1035] = c_commit;
        }
    } else if (warp >= 4) {
        // ===================== epilogue: TMEM -> registers -> (+ bias, Relu) -> shared memory -> coalesced global stores ====
        // A thread owns one slot (TMEM lane) of the 32-column chunk; writing its 128 bytes to global memory directly costs
        // 32 scattered 16-byte sectors per instruction (8-10 B/clk/SM measured, tools/store_probe.cu).  The chunk is staged
        // in shared memory (128B-swizzled rows) instead, and every warp instruction then writes four WHOLE 128-byte slot
        // rows (~24 B/clk/SM, the SM's store port).  Slots that are padding (x >= OW, rows past the strip / image, tail
        // images) are skipped on the way out.
        const EpilogueDesc& e = p.epi;
        const int q = warp & 3, grp = (warp - 4) >> 2;
        const int r = q * 32 + lane;
        const bool has_bias = e.bias_kind == 1;
        const bool do_relu = e.act == 1;
        const uint32_t img_slots = (uint32_t)(p.nr * p.P);
        uint8_t* stg = stage0 + grp * 16384;
        uint8_t* rowp = stg + r * 128;
        const int sw = r & 7;
        float* bias_g = bias_s + grp * 128;
        const int piece = lane & 7;  // 16-byte piece of a slot row on the way out
        uint32_t aphase = 0;
        int it = 0;
        float* outp = reinterpret_cast<float*>(e.d);
        for (int u = blockIdx.x; u < p.units_total; u += gridDim.x, it++) {
            int n0, oy0, b0;
            halo_unit(p, u, n0, oy0, b0);
            const int acc = p.acc_stages == 2 ? (it & 1) : 0;
            float bv = 0.0f;
            if (has_bias) {  // thread i of the group: column (i / 32) * 64 + grp * 32 + i % 32 of the unit
                const int c = (r >> 5) * 64 + grp * 32 + (r & 31);
                if (c < p.bn && n0 + c < p.N) bv = __ldg(e.bias + n0 + c);
            }
            mbar_wait(&tmem_full[acc], (aphase >> acc) & 1);
            if (tr0 && warp == 4 && lane == 0 && it < 1024) p.trace[4096 + it] = clock64();
            aphase ^= 1u << acc;
            tc_fence_after();
            bias_g[r] = bv;  // (readers of the previous unit's values are past that unit's last barrier)
            for (int t = 0; t < p.T; t++) {
                // the eight slots this thread writes out per chunk: slot = t * 128 + q * 32 + i * 4 + lane / 8
                long long off[8];
                unsigned valid = 0;
#pragma unroll
                for (int i = 0; i < 8; i++) {
                    const uint32_t slot = (uint32_t)(t * 128 + q * 32 + i * 4 + (lane >> 3));
                    const uint32_t img = __umulhi(slot, p.m_img);
                    const uint32_t rem = slot - img * img_slots;
                    const uint32_t yy = __umulhi(rem, p.m_P);
                    const uint32_t ox = rem - yy * (uint32_t)p.P;
                    const int oy = oy0 + (int)yy, b = b0 + (int)img;
                    if ((int)img < p.tb && b < p.B && (int)yy < p.R && oy < p.OH && (int)ox < p.OW) valid |= 1u << i;
                    off[i] = (long long)b * e.s_z0 + (long long)oy * e.s_row + (long long)ox * e.s_z1 + n0 + piece * 4;
                }
                const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + acc * 256 + t * p.bn;
                int k = 0;
                for (int c0 = grp * 32; c0 < p.bn; c0 += 64, k++) {
                    uint32_t v[32];
                    tmem_ld_32x32(t_row + c0, v);
                    tmem_ld_wait();
                    // every warp of the group has read the previous chunk out of the staging buffer (and, for the first
                    // chunk of a unit, the bias values are in place)
                    asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
                    const float4* bq = reinterpret_cast<const float4*>(bias_g + 32 * k);
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 bb = bq[j >> 2];
                        add_pair(v[j], v[j + 1], bb.x, bb.y);
                        add_pair(v[j + 2], v[j + 3], bb.z, bb.w);
                        if (do_relu) {
#pragma unroll
                            for (int w = 0; w < 4; w++) v[j + w] = __float_as_uint(fmaxf(__uint_as_float(v[j + w]), 0.0f));
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 8; j++)
                        *reinterpret_cast<uint4*>(rowp + ((j ^ sw) << 4)) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                    asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
                    if (n0 + c0 < p.N) {
#pragma unroll
                        for (int i = 0; i < 8; i++) {
                            const int sl = q * 32 + i * 4 + (lane >> 3);  // slot of the chunk (= staging row)
                            const uint4 d = *reinterpret_cast<const uint4*>(stg + sl * 128 + ((piece ^ (sl & 7)) << 4));
                            if (valid & (1u << i)) *reinterpret_cast<uint4*>(outp + off[i] + c0) = d;
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tmem_empty[acc]);
            if (tr0 && warp == 4 && lane == 0 && it < 1024) p.trace[6144 + it] = clock64();
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        tc_fence_after();
        tmem_dealloc(tmem_base, 512);
    }
    if (tr0 && threadIdx.x == 0) p.trace[6144 + 1104] = clock64();
}

}  // namespace

// force_bn / force_T > 0: that unit shape or RTEN_ERR_UNSUPPORTED_VALUE (the autotuner times a few of them against the
// generic kernel's plans and records the winner); 0: the cost model's choice, and only with RTEN_B200_HALO=1 -- without
// measurements the generic kernel stays the default (profiles/r02_halo_sweep.txt: the two are within a few percent of each
// other on ResNet-50's layers, which one wins depends on the layer).
rten_status launch_umma_halo_conv(rten_ctx* ctx, const GemmLaunch& L, int force_bn, int force_T) {
    if (getenv("RTEN_B200_NO_HALO")) return RTEN_ERR_UNSUPPORTED_VALUE;
    if (!force_bn) {
        const char* on = getenv("RTEN_B200_HALO");
        if (!on || atoi(on) == 0) return RTEN_ERR_UNSUPPORTED_VALUE;
    }
    if (!L.conv || L.kind != 0) return RTEN_ERR_UNSUPPORTED_VALUE;
    const ConvGeom& g = L.g;
    const EpilogueDesc& e = L.epi;
    if (g.sy != 1 || g.sx != 1 || g.dy != 1 || g.dx != 1 || g.kh * g.kw < 2 || g.kh * g.kw > 32) return RTEN_ERR_UNSUPPORTED_VALUE;
    if (g.C % 32 || g.C < 32) return RTEN_ERR_UNSUPPORTED_VALUE;
    if (L.N % 32 || L.N < 32) return RTEN_ERR_UNSUPPORTED_VALUE;
    if (e.r || e.range || e.bias_kind == 2 || e.act > 1 || e.s_col != 1 || e.d_is_i32 || e.alpha != 1.0f) return RTEN_ERR_UNSUPPORTED_VALUE;
    auto al16 = [](const void* q) { return (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
    if (!al16(e.d) || (e.s_z0 & 3) || (e.s_row & 3) || (e.s_z1 & 3) || (e.bias_kind == 1 && !al16(e.bias))) return RTEN_ERR_UNSUPPORTED_VALUE;
    if (!tma_compatible(L.a, 4, 4) || !tma_compatible(L.b, 4, 4)) return RTEN_ERR_UNSUPPORTED_VALUE;
    HaloParams p;
    memset(&p, 0, sizeof(p));
    p.B = g.B;
    p.OH = g.OH;
    p.OW = g.OW;
    p.N = L.N;
    p.C = g.C;
    p.kh = g.kh;
    p.kw = g.kw;
    p.pt = g.pt;
    p.pl = g.pl;
    p.P = g.OW + g.kw - 1;
    p.c_blocks = g.C / 32;
    p.taps = g.kh * g.kw;
    p.epi = e;
    p.trace = reinterpret_cast<long long*>(ctx->trace);
    if (p.P > 256) return RTEN_ERR_UNSUPPORTED_VALUE;
    // ---- unit shape.  Candidates: output-channel tile bn, MMA tiles T per unit, whole images (tb >= 1 images of
    // OH + kh - 1 patch rows) or row strips (R rows of one image).  Ranked by waves x (MMA clocks of a unit), with the
    // slots that are thrown away counted in.
    const int num_sms = ctx->num_sms;
    double best = 1e30;
    int bbn = 0, bT = 0, bR = 0, btb = 0, btps = 1;
    const char* fbn = getenv("RTEN_B200_HALO_BN");
    const char* fT = getenv("RTEN_B200_HALO_T");
    const int want_bn = force_bn ? force_bn : (fbn ? atoi(fbn) : 0), want_T = force_T ? force_T : (fT ? atoi(fT) : 0);
    for (int bn = 32; bn <= std::min(L.N, 256); bn += 32) {
        if (L.N % bn) continue;
        if (want_bn && bn != want_bn) continue;
        for (int T = 1; T <= 4; T++) {
            if (T * bn > 512) break;
            if (want_T && T != want_T) continue;
            // whole-image mode when tb >= 1 padded images fit T tiles, else strips of R rows
            const int img_slots = (g.OH + g.kh - 1) * p.P;
            int tb = 1, R = 0;
            if (g.OH * p.P <= T * 128) {
                R = g.OH;
                tb = 1 + (T * 128 - g.OH * p.P) / img_slots;
                tb = std::min(tb, g.B);
            } else {
                R = (T * 128) / p.P;
                if (R < 1) continue;
            }
            const int nr = R + g.kh - 1;
            if (nr > 256 || tb > 256) continue;
            const long long alloc_slots = (long long)T * 128 + (g.kh - 1) * p.P + g.kw - 1;
            const long long loaded_slots = (long long)tb * nr * p.P;
            const long long patch_bytes = (std::max(alloc_slots, loaded_slots) * 128 + 1023) / 1024 * 1024;
            // taps per weight stage: the whole window, one window row, or one tap -- the most that leaves >= 2 stages
            const long long budget = 227 * 1024 - 3072 - 2 * 16384 - 2 * patch_bytes;  // alignment, barriers, bias, output staging
            // a stage must be requested ~1500 clk (TMA latency + its own transfer) before its MMAs start: four stages in
            // flight keep the tensor pipe fed, two leave it waiting for every other stage
            // (and every hand-off costs the issuing warp ~300 clk: the most taps per stage that still leaves three stages)
            int tps = 0;
            for (int cand : {g.kh * g.kw, g.kw, 1}) {
                if ((long long)cand * bn * 128 * 3 <= budget) {
                    tps = cand;
                    break;
                }
            }
            if (!tps || tps > 256) continue;
            const long long b_bytes = (long long)tps * bn * 128;
            const long long strips = (g.OH + R - 1) / R;
            const long long units = strips * ((g.B + tb - 1) / tb) * (L.N / bn);
            const double waves = std::ceil((double)units / num_sms);
            // per unit: MMA clocks (T tiles x taps x c_blocks x 4 instructions of bn / 2 clocks, issue >= 40 clk each) vs the
            // operand bytes entering the SM at ~55 B/clk; epilogue not overlapped when there is a single accumulator stage
            // (~42 clk to issue an MMA, ~320 clk per barrier hand-off of a weight stage: profiles/r01_trace_pipeline_v2.txt)
            const double mma = (double)p.c_blocks * ((double)T * p.taps * 4.0 * std::max(42.0, bn / 2.0) + 320.0 * (p.taps / tps));
            const double bytes = (double)p.c_blocks * (loaded_slots * 128.0 + (double)p.taps * bn * 128.0);
            const double ingest = bytes / 55.0;
            const double epi = (double)T * (bn / 32.0) * 350.0 / 2.0;
            const int acc_stages = (2 * T * bn <= 512) ? 2 : 1;
            const double unit = std::max(mma, ingest) + (acc_stages == 2 ? 0.25 * epi : epi) + 800.0;
            const double cost = waves * unit + 4000.0;
            if (cost < best) {
                best = cost;
                bbn = bn;
                bT = T;
                bR = R;
                btb = tb;
                btps = tps;
            }
        }
    }
    if (!bbn) return RTEN_ERR_UNSUPPORTED_VALUE;
    p.bn = bbn;
    p.T = bT;
    p.R = bR;
    p.tb = btb;
    p.nr = p.R + g.kh - 1;
    p.acc_stages = (2 * p.T * p.bn <= 512) ? 2 : 1;
    p.strips = (g.OH + p.R - 1) / p.R;
    p.units_n = L.N / p.bn;
    p.units_total = p.strips * ((g.B + p.tb - 1) / p.tb) * p.units_n;
    const long long alloc_slots = (long long)p.T * 128 + (g.kh - 1) * p.P + g.kw - 1;
    const long long loaded_slots = (long long)p.tb * p.nr * p.P;
    p.patch_bytes = (uint32_t)((std::max(alloc_slots, loaded_slots) * 128 + 1023) / 1024 * 1024);
    p.patch_tx = (uint32_t)(loaded_slots * 128);
    p.tps = btps;
    p.b_bytes = (uint32_t)(p.tps * p.bn) * 128u;
    p.b_stages = (int)std::min<long long>(HB_MAX, (227 * 1024 - 3072 - 2 * 16384 - 2LL * p.patch_bytes) / p.b_bytes);
    p.idesc = make_idesc(1 /*F32*/, 2 /*TF32*/, 2, 128, p.bn);
    for (int ky = 0; ky < g.kh; ky++)
        for (int kx = 0; kx < g.kw; kx++) p.tap_off[ky * g.kw + kx] = (uint32_t)((ky * p.P + kx) * 8);
    p.m_img = (uint32_t)(0x100000000ull / (unsigned long long)(p.nr * p.P)) + 1u;
    p.m_P = (uint32_t)(0x100000000ull / (unsigned long long)p.P) + 1u;

    uint32_t abox[4] = {32u, (uint32_t)p.P, (uint32_t)p.nr, (uint32_t)p.tb}, ones[4] = {1, 1, 1, 1};
    uint32_t bbox[4] = {32u, (uint32_t)p.bn, (uint32_t)p.tps, 1u};
    CUtensorMap map_a, map_b;
    if (!encode_map(ctx, &map_a, L.a, 4, true, abox, ones)) return RTEN_ERR_UNSUPPORTED_VALUE;
    if (!encode_map(ctx, &map_b, L.b, 4, true, bbox, ones)) return RTEN_ERR_UNSUPPORTED_VALUE;
    if (getenv("RTEN_B200_VERBOSE"))
        fprintf(stderr, "[umma_halo] B=%d %dx%d C=%d N=%d k=%dx%d: bn=%d T=%d R=%d tb=%d P=%d units=%d acc_stages=%d b_stages=%d tps=%d patch=%u B\n", g.B,
                g.OH, g.OW, g.C, L.N, g.kh, g.kw, p.bn, p.T, p.R, p.tb, p.P, p.units_total, p.acc_stages, p.b_stages, p.tps, p.patch_bytes);
    const size_t smem = 1024 /*align*/ + 2048 /*barriers, bias*/ + 2 * 16384 /*output staging*/ + 2 * (size_t)p.patch_bytes + (size_t)p.b_stages * p.b_bytes;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(std::min(p.units_total, num_sms));
    cfg.blockDim = dim3(HALO_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    fill_launch_attrs(cfg, attr, false);
    cudaError_t ce = cudaFuncSetAttribute(umma_halo_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (ce == cudaSuccess) ce = cudaLaunchKernelEx(&cfg, umma_halo_kernel, map_a, map_b, p);
    if (ce != cudaSuccess) return fail_cuda(ctx, ce, "umma_halo launch");
    ce = cudaGetLastError();
    if (ce != cudaSuccess) return fail_cuda(ctx, ce, "umma_halo launch");
    count_launch(ctx);
    return RTEN_OK;
}

}  // namespace rtb
