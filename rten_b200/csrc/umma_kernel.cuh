// Device side of the tcgen05 GEMM / implicit-GEMM convolution: tile decode, the warp-specialised persistent kernel
// (TMA producer / MMA issuer / TMEM allocator / two epilogue groups).  Included ONLY by umma_gemm.cu, which holds the
// host side (launch plans, cost model, autotuner, tensor maps).  See umma_gemm.cu's header comment for the design.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "math.cuh"
#include "ptx.cuh"
#include "umma_gemm.h"

namespace rtb {

constexpr int BM = 128;            // UMMA M (cta_group::1)
constexpr int KBYTES = 128;        // bytes of K per stage row = one 128B swizzle atom
constexpr int A_STAGE_BYTES = BM * KBYTES;
constexpr int TMEM_COLS = 512;
constexpr int ACC_STRIDE = 256;    // TMEM columns per accumulator stage
constexpr int NUM_THREADS = 384;   // 4 control warps + 8 epilogue warps (two groups of 4)
constexpr int STG_BYTES = 128 * 128;  // one 128-row x 128-byte output staging buffer per epilogue group
constexpr int MAX_STAGES = 8;

// Division by a launch-time constant as multiply-high + shift (exact for 0 <= n < 2^31): the tile decode sits on the
// critical path at the start of every kernel and of every tile, and a hardware-emulated 32-bit division costs ~100
// instructions.
struct FastDiv {
    uint32_t d = 1, mul = 0, shr = 0;
    __host__ void set(int div) {
        d = (uint32_t)(div < 1 ? 1 : div);
        if (d == 1) {
            mul = 0;
            shr = 0;
            return;
        }
        uint32_t lg = 0;
        while ((1ull << lg) < d) lg++;  // ceil(log2(d))
        const uint32_t p = 31 + lg;
        mul = (uint32_t)(((1ull << p) + d - 1) / d);
        shr = p - 32;
    }
    __device__ __forceinline__ int div(int n) const { return d == 1 ? n : (int)(__umulhi((uint32_t)n, mul) >> shr); }
    __device__ __forceinline__ void divmod(int n, int& q, int& r) const {
        q = div(n);
        r = n - q * (int)d;
    }
};

struct KParams {
    int M, N, K, z0, z1;
    int tiles_m, tiles_n, tiles_total;
    int k_blocks, kelems;
    int bn, stages;
    uint32_t stage_bytes, tx_bytes;
    uint32_t idesc;
    int conv;
    int tw, th, tb, tiles_x, tiles_y;
    int OH, OW, Bn;
    int sy, sx, dy, dx, pt, pl, kw, c_blocks;
    int a_bcast0, a_bcast1, b_bcast0, b_bcast1;
    long long* trace;  // debug: per-event clock64 timestamps of CTA 0 (4 rows x 2048), or null
    int pair;       // 1: each CTA iteration computes TWO 128-row tiles sharing one B tile (interleaved MMAs on two
                    //    accumulators hide the dependent-accumulate latency when bn <= 128)
    int katoms;     // consecutive 128-byte K blocks loaded / multiplied per pipeline stage (1 or 2): amortises the fixed
                    // per-stage barrier round trip of the issuing threads when tiles are small
    uint32_t atom_bytes;
    int ksplit;     // 1: (single-tile mode, bn <= 128) even / odd K blocks accumulate into two TMEM accumulators that the
                    //    epilogue adds: consecutive MMAs never depend on each other (no dependent-accumulate stall)
    int nbuf;       // staging buffers per epilogue group (ring): nbuf-1 (nbuf-2 with res_tma) bulk stores stay in flight
    int res_tma;    // 1: the residual tile is prefetched by TMA into the staging buffer (needs tma_store)
    uint32_t res_tx_bytes;
    int tma_store;  // 1: epilogue stages 128x32 chunks in smem and writes them with TMA (output rows contiguous)
    int acc1;       // 1: ONE accumulator stage of 512 TMEM columns (pair mode with bn = 256: a 256 x 256 tile per CTA halves
                    //    the L2 -> SM operand traffic per flop; the epilogue no longer overlaps the next main loop)
    int splitk;     // > 1: `splitk` CTAs share one output tile, each over `kb_per` K blocks; raw partial accumulators go
                    // to `sk_ws`, the LAST CTA to arrive (per tile and epilogue group, `sk_cnt`) sums them in split order
                    // (deterministic) and runs the epilogue
    int kb_per;
    int cta2;       // 1: CTA pairs (cluster 2x1x1) execute 256-row tcgen05.mma.cta_group::2 tiles; each CTA loads its own
                    //    128 rows of A and HALF of the B tile, so operand bytes entering an SM per flop drop by up to 2x
    int units_total;  // tiles_total * splitk
    int x3_cb;      // > 0: 3xTF32 over TWO planes of A -- the K (channel) range is three segments of x3_cb K blocks,
                    //      [lo | hi | hi]: segment 0 reads the low-part plane (tma_a2), segments 1 and 2 read the ORIGINAL f32
                    //      tensor (kind::tf32 ignores the 13 low mantissa bits, so the raw values ARE the high parts)
    FastDiv d_tiles_n, d_units_m, d_z0, d_tiles_x, d_tiles_y, d_tiles_total, d_c_blocks, d_kw, d_tw, d_th;
    uint32_t* sk_ws;
    int* sk_cnt;
    EpilogueDesc epi;
};

struct TileCoord {
    int n0;
    int m0;          // plain: first row; conv: unused
    int z0, z1;      // plain batch coords
    int ox0, oy0, b0;  // conv
};

// t indexes work units: (n tile, m tile or PAIR of m tiles, batch); `sub` selects the tile inside a pair.
__device__ __forceinline__ TileCoord decode_tile(const KParams& p, int t, int sub, int rank = 0) {
    TileCoord c;
    int n_blk, rest, m_blk, z;
    p.d_tiles_n.divmod(t, rest, n_blk);
    // one unit = (pair + 1) MMA tiles of (cta2 + 1) x 128 rows: `mult` consecutive 128-row blocks
    const int mult = (p.pair + 1) * (p.cta2 + 1);
    p.d_units_m.divmod(rest, z, m_blk);
    m_blk = m_blk * mult + sub * (p.cta2 + 1) + rank;  // may be >= tiles_m in the tail: every row is then out of range
    c.n0 = n_blk * p.bn;
    c.m0 = m_blk * BM;
    p.d_z0.divmod(z, c.z1, c.z0);
    c.ox0 = c.oy0 = c.b0 = 0;
    if (p.conv) {
        int xt, r2, yt, bt;
        p.d_tiles_x.divmod(m_blk, r2, xt);
        p.d_tiles_y.divmod(r2, bt, yt);  // bt >= number of batch tiles for the odd tail of a pair -> b0 >= B
        c.ox0 = xt * p.tw;
        c.oy0 = yt * p.th;
        c.b0 = bt * p.tb;
    }
    return c;
}

// (a0, a1) += (b0, b1): one packed FADD2, each half rounded to nearest like a scalar add
__device__ __forceinline__ void add_f32x2(uint32_t& a0, uint32_t& a1, float b0, float b1) {
    unsigned long long a, b, d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "r"(a0), "r"(a1));
    asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    asm("mov.b64 {%0, %1}, %2;" : "=r"(a0), "=r"(a1) : "l"(d));
}

// (a0, a1) *= (b0, b1): one packed FMUL2, each half rounded to nearest like a scalar multiply
__device__ __forceinline__ void mul_f32x2(uint32_t& a0, uint32_t& a1, float b0, float b1) {
    unsigned long long a, b, d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "r"(a0), "r"(a1));
    asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    asm("mov.b64 {%0, %1}, %2;" : "=r"(a0), "=r"(a1) : "l"(d));
}

// cp.async.bulk.wait_group.read takes an immediate: leave at most `n` of this thread's bulk stores un-read
__device__ __forceinline__ void bulk_wait_read(int n) {
    switch (n) {
        case 0: asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); break;
        case 1: asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); break;
        case 2: asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory"); break;
        default: asm volatile("cp.async.bulk.wait_group.read 3;" ::: "memory"); break;
    }
}

__device__ __forceinline__ int f32_to_ordered(float f) {  // same encoding as rowops.cu's min / max kernels
    const int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
// fold a warp's running (min, max) into the launch-wide range (EpilogueDesc::range)
__device__ __forceinline__ void range_commit(int* range, float lo, float hi) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fminf(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmaxf(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if ((threadIdx.x & 31) == 0 && lo <= hi) {
        atomicMin(&range[0], f32_to_ordered(lo));
        atomicMax(&range[1], f32_to_ordered(hi));
    }
}

// Gelu (erf / tanh form) of four values as an out-of-line call: the specialised epilogue stays short straight-line
// code (an unrolled polynomial per element would multiply its size and thrash the instruction cache), yet Gelu no
// longer forces a launch into the generic epilogue.
__device__ __noinline__ float4 act4(float4 x, int act) {
    if (act == 2) {  // Gelu: two lanes per packed instruction (bit-identical to gelu_ref, math.cuh)
        gelu_ref_x2(x.x, x.y);
        gelu_ref_x2(x.z, x.w);
        return x;
    }
    x.x = apply_act(x.x, act);
    x.y = apply_act(x.y, act);
    x.z = apply_act(x.z, act);
    x.w = apply_act(x.w, act);
    return x;
}

// Split-K hand-off of one epilogue group (128 threads): store this CTA's raw accumulator chunks, then count arrivals.
// Returns true for the group of the CTA that arrived last: it owns the epilogue of (tile, group).
// Workspace layout: [tile][sub][split][chunk][column j][row r] so that a warp's 32 rows are contiguous.
__device__ __forceinline__ bool splitk_publish(const KParams& p, int t, int ks, int grp, int q, int lane, uint32_t t_acc,
                                               int* flag) {  // t = tile slot (tile, or 2 * tile + cluster rank)
    const int r = q * 32 + lane;
    const int nchunks = p.bn >> 5;
    for (int sub = 0; sub <= p.pair; sub++) {
        for (int c0 = grp * 32; c0 < p.bn; c0 += 64) {
            uint32_t v[32];
            tmem_ld_32x32(t_acc + sub * p.bn + c0, v);
            tmem_ld_wait();
            uint32_t* w = p.sk_ws + ((((size_t)(t * 2 + sub) * p.splitk + ks) * nchunks + (c0 >> 5)) << 12) + r;
#pragma unroll
            for (int j = 0; j < 32; j++) __stcg(w + j * 128, v[j]);
        }
    }
    __threadfence();
    asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
    if (q == 0 && lane == 0) {
        int* cnt = p.sk_cnt + t * 2 + grp;
        const int old = atomicAdd(cnt, 1);
        const int last = old == p.splitk - 1;
        if (last) *cnt = 0;  // every split has arrived: re-arm for the next launch
        __threadfence();
        *flag = last;
    }
    asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
    return *reinterpret_cast<volatile int*>(flag) != 0;
}

// Sum of the `splitk` partial chunks in split order (the same order whichever CTA arrived last).
template <int KIND>
__device__ __forceinline__ void splitk_sum(const KParams& p, int t, int sub, int c0, int r, uint32_t (&v)[32]) {
    const int nchunks = p.bn >> 5;
    const uint32_t* w = p.sk_ws + ((((size_t)(t * 2 + sub) * p.splitk) * nchunks + (c0 >> 5)) << 12) + r;
    const size_t stride = (size_t)nchunks << 12;
#pragma unroll
    for (int j = 0; j < 32; j++) v[j] = __ldcg(w + j * 128);
#pragma unroll 1
    for (int s = 1; s < p.splitk; s++) {
        w += stride;
#pragma unroll
        for (int j = 0; j < 32; j++) {
            const uint32_t x = __ldcg(w + j * 128);
            if (KIND == 0)
                v[j] = __float_as_uint(__fadd_rn(__uint_as_float(v[j]), __uint_as_float(x)));
            else
                v[j] += x;
        }
    }
}

// Per-thread pipeline state of one launch: parity bits of the operand ring (bit s = uses of stage s so far, mod 2), of
// the two accumulator barriers, of the residual barriers, and the running tile count that picks the accumulator stage.
// Each role keeps its own copy.
struct PipeState {
    uint32_t ring = 0, acc = 0, rphase = 0;
    int it = 0;
};

struct SmemLayout {
    uint8_t* smem;  // operand stages (1024-B aligned), staging buffers behind them
    uint64_t *full_bar, *empty_bar, *tmem_full, *tmem_empty, *res_bar;
    int* sk_flag;
    float* bias;
};

}  // namespace rtb

#include "umma_epilogue_plain.cuh"
#include "umma_epilogue_generic.cuh"

namespace rtb {

// One launch worth of work (all roles).  FAST = the launch satisfies, for EVERY chunk, the conditions of the register
// fast path (TMA-store output, N % 32 == 0, f32 with act in {none, relu} and bias / residual absent or
// vector-addressable [residual via TMA], or raw i32): the epilogue is then a short straight-line loop.  The generic
// variant (FAST = 0) keeps every edge case.
template <int KIND, int FAST, int CTA2>
__device__ __forceinline__ void run_layer(const KParams& p, const CUtensorMap* tma_a, const CUtensorMap* tma_a2,
                                          const CUtensorMap* tma_b, const CUtensorMap* tma_d, const CUtensorMap* tma_r, const SmemLayout& L,
                                          uint32_t tmem_base, int cta_rank, int worker, int n_workers) {
    PipeState st;
    uint8_t* smem = L.smem;
    uint8_t* stg_base = smem + (size_t)p.stages * p.stage_bytes;
    const int nbuf = p.nbuf;
    uint64_t* full_bar = L.full_bar;
    uint64_t* empty_bar = L.empty_bar;
    uint64_t* tmem_full = L.tmem_full;
    uint64_t* tmem_empty = L.tmem_empty;
    uint64_t* res_bar = L.res_bar;
    int* sk_flag = L.sk_flag;
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    // Control warps run their loops WARP-UNIFORMLY (all 32 lanes wait on the barriers, one elected lane issues the
    // TMA / MMA instructions): addresses and descriptors then live in uniform registers instead of being moved
    // there (R2UR) for every instruction, which is what bounds a single issuing thread.
    if (warp == 0) {
        // ===================== TMA producer =====================
        int stage = 0;
        int tr_p = 0;
        const uint32_t smem0 = smem_u32(smem);
        const uint32_t full0 = smem_u32(full_bar);
        const uint32_t a_bytes = (p.pair ? 2 : 1) * A_STAGE_BYTES;
        const int b_row0 = CTA2 ? cta_rank * (p.bn >> 1) : 0;  // this CTA's half of the B tile
        for (int u = worker; u < p.units_total; u += n_workers) {
            int t, ks;
            p.d_tiles_total.divmod(u, ks, t);
            const int kb0 = ks * p.kb_per, kb1 = min(p.k_blocks, kb0 + p.kb_per);
            const TileCoord tc = decode_tile(p, t, 0, cta_rank);
            const TileCoord tc1 = p.pair ? decode_tile(p, t, 1, cta_rank) : tc;
            // conv: K block -> (filter tap, channel block), kept incrementally
            int tap, cb, ky, kx;
            p.d_c_blocks.divmod(kb0, tap, cb);
            p.d_kw.divmod(tap, ky, kx);
            // two-plane 3xTF32: segment of the K / channel range and block inside it (kept incrementally)
            int seg = 0, sblk = p.conv ? cb : kb0;
            if (p.x3_cb)
                while (sblk >= p.x3_cb) {
                    sblk -= p.x3_cb;
                    seg++;
                }
            // programmatic dependent launch: the producer is the first to touch the predecessor's output; everything
            // above (tile decode) ran while the predecessor grid was still draining
            if (u == worker) asm volatile("griddepcontrol.wait;" ::: "memory");
            for (int kb = kb0; kb < kb1; kb += p.katoms) {
                const int natoms = min(p.katoms, kb1 - kb);
                mbar_wait(&empty_bar[stage], ((st.ring >> stage) & 1) ^ 1);
                const bool leader = elect_one();
                // CTA pair: both CTAs' loads complete on the LEADER's barrier, which expects the bytes of both
                const uint32_t fb = CTA2 ? ((full0 + stage * 8) & PEER_BIT_MASK) : (full0 + stage * 8);
                if (leader) {
                    if (p.trace && blockIdx.x == 0 && tr_p < 2048) p.trace[tr_p++] = clock64();
                    if (!CTA2)
                        mbar_expect_tx_u32(fb, p.tx_bytes * natoms);
                    else if (cta_rank == 0)
                        mbar_expect_tx_u32(fb, 2 * p.tx_bytes * natoms);
                }
                for (int a = 0; a < natoms; a++) {
                    if (leader) {
                        const uint32_t sa = smem0 + stage * p.stage_bytes + a * p.atom_bytes;
                        const uint32_t sb = sa + a_bytes;
                        auto load = [&](uint32_t dst, const CUtensorMap* m, int c0, int c1, int c2, int c3) {
                            if (CTA2)
                                tma_load_4d_2sm(dst, m, fb, c0, c1, c2, c3);
                            else
                                tma_load_4d_u32(dst, m, fb, c0, c1, c2, c3);
                        };
                        const CUtensorMap* ma = (p.x3_cb && seg == 0) ? tma_a2 : tma_a;
                        if (p.conv) {
                            const int c0 = cb * p.kelems;
                            const int ca = p.x3_cb ? sblk * p.kelems : c0;
                            load(sa, ma, ca, tc.ox0 * p.sx - p.pl + kx * p.dx, tc.oy0 * p.sy - p.pt + ky * p.dy, tc.b0);
                            if (p.pair)
                                load(sa + A_STAGE_BYTES, ma, ca, tc1.ox0 * p.sx - p.pl + kx * p.dx,
                                     tc1.oy0 * p.sy - p.pt + ky * p.dy, tc1.b0);
                            load(sb, tma_b, c0, tc.n0 + b_row0, tap, 0);
                        } else {
                            const int k0 = (kb + a) * p.kelems;
                            const int ka = p.x3_cb ? sblk * p.kelems : k0;
                            const int az0 = p.a_bcast0 ? 0 : tc.z0, az1 = p.a_bcast1 ? 0 : tc.z1;
                            load(sa, ma, ka, tc.m0, az0, az1);
                            if (p.pair) load(sa + A_STAGE_BYTES, ma, ka, tc1.m0, az0, az1);
                            load(sb, tma_b, k0, tc.n0 + b_row0, p.b_bcast0 ? 0 : tc.z0, p.b_bcast1 ? 0 : tc.z1);
                        }
                    }
                    if (p.x3_cb && ++sblk == p.x3_cb) {
                        sblk = 0;
                        seg = seg == 2 ? 0 : seg + 1;  // (conv: the next filter tap starts over at segment 0)
                    }
                    if (++cb == p.c_blocks) {
                        cb = 0;
                        tap++;
                        if (++kx == p.kw) {
                            kx = 0;
                            ky++;
                        }
                    }
                }
                __syncwarp();
                st.ring ^= 1u << stage;
                if (++stage == p.stages) stage = 0;
            }
        }
    } else if (warp == 1 && cta_rank == 0) {
        // ===================== MMA issuer (pair mode: the leader CTA only) =====================
        int stage = 0;
        int tr_m = 0;
        const uint32_t smem0 = smem_u32(smem);
        const uint32_t empty0 = smem_u32(empty_bar);
        const uint32_t b_off = (p.pair ? 2 : 1) * A_STAGE_BYTES;
        const uint32_t d1_off = (p.pair || p.ksplit) ? p.bn : 0;
        for (int u = worker; u < p.units_total; u += n_workers, st.it++) {
            const int kb0 = p.d_tiles_total.div(u) * p.kb_per, kb1 = min(p.k_blocks, kb0 + p.kb_per);
            const int acc = p.acc1 ? 0 : (st.it & 1);
            mbar_wait(&tmem_empty[acc], ((st.acc >> acc) & 1) ^ 1);
            st.acc ^= 1u << acc;
            tc_fence_after();
            const uint32_t d_tmem = tmem_base + acc * ACC_STRIDE;
            for (int kb = kb0; kb < kb1; kb += p.katoms) {
                const int natoms = min(p.katoms, kb1 - kb);
                mbar_wait(&full_bar[stage], (st.ring >> stage) & 1);
                tc_fence_after();
                if (elect_one()) {
                    if (p.trace && blockIdx.x == 0 && tr_m < 2048) p.trace[2048 + tr_m++] = clock64();
                    for (int a = 0; a < natoms; a++) {
                        const uint32_t sa = smem0 + stage * p.stage_bytes + a * p.atom_bytes;
                        const uint64_t adesc = make_kmajor_sw128_desc(sa);
                        const uint64_t bdesc = make_kmajor_sw128_desc(sa + b_off);
                        const uint32_t first = (kb + a) == kb0 ? 0u : 1u;
                        auto mma = [&](uint32_t d, uint64_t ad, uint64_t bd, uint32_t accum) {
                            if (CTA2)
                                umma2<KIND>(d, ad, bd, p.idesc, accum);
                            else
                                umma<KIND>(d, ad, bd, p.idesc, accum);
                        };
                        if (p.pair) {
                            const uint64_t adesc1 = make_kmajor_sw128_desc(sa + A_STAGE_BYTES);
#pragma unroll
                            for (int k = 0; k < 4; k++) {  // +2 in the (addr >> 4) field = 32 B along K in the swizzle atom
                                mma(d_tmem, adesc + 2 * k, bdesc + 2 * k, k == 0 ? first : 1u);
                                mma(d_tmem + d1_off, adesc1 + 2 * k, bdesc + 2 * k, k == 0 ? first : 1u);
                            }
                        } else if (p.ksplit) {
#pragma unroll
                            for (int k = 0; k < 4; k++)  // k even -> accumulator 0, k odd -> accumulator 1
                                mma(d_tmem + (k & 1) * d1_off, adesc + 2 * k, bdesc + 2 * k, k < 2 ? first : 1u);
                        } else {
#pragma unroll
                            for (int k = 0; k < 4; k++)
                                mma(d_tmem, adesc + 2 * k, bdesc + 2 * k, k == 0 ? first : 1u);
                        }
                    }
                    // smem slot reusable once these MMAs retire; accumulator complete -> epilogue (of both CTAs)
                    if (CTA2) {
                        umma_commit_mc(empty0 + stage * 8, 3);
                        if (kb + natoms >= kb1) umma_commit_mc(smem_u32(&tmem_full[acc]), 3);
                    } else {
                        umma_commit_u32(empty0 + stage * 8);
                        if (kb + natoms >= kb1) umma_commit(&tmem_full[acc]);
                    }
                }
                __syncwarp();
                st.ring ^= 1u << stage;
                if (++stage == p.stages) stage = 0;
            }
        }
    } else if (warp >= 4) {
        // ===================== epilogue warps: one of four variants (umma_epilogue_plain.cuh / umma_epilogue_generic.cuh)
        const EpiCtx c{p, L, stg_base, nbuf, tmem_full, tmem_empty, res_bar, sk_flag, tma_d, tma_r, tmem_base, cta_rank, worker, n_workers, st, warp, lane};
        if (KIND == 0 && (FAST == 3 || FAST == 5))
            epilogue_plain_f32<FAST, CTA2>(c);
        else if (KIND == 1 && (FAST == 4 || FAST == 6))
            epilogue_plain_i8<FAST, CTA2>(c);
        else if (FAST)
            epilogue_fast<KIND, FAST, CTA2>(c);
        else
            epilogue_generic<KIND, CTA2>(c);
    }

}

// Shared-memory carve-up: a fixed 1 KB block of mbarriers first, operand stages behind it.
template <int KIND>
__device__ __forceinline__ SmemLayout carve_smem(uint8_t* smem_raw) {
    // 1024-B alignment required by the 128B swizzle atoms / UMMA descriptors (base_offset = 0).
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    SmemLayout L;
    L.full_bar = reinterpret_cast<uint64_t*>(base);
    L.empty_bar = L.full_bar + MAX_STAGES;
    L.tmem_full = L.empty_bar + MAX_STAGES;
    L.tmem_empty = L.tmem_full + 2;
    L.res_bar = L.tmem_empty + 2;  // [group][buffer], up to 4 buffers per group
    L.sk_flag = reinterpret_cast<int*>(L.res_bar + 8) + 2;  // [group]; the two ints before it hold the TMEM base
    // column vectors of the current unit for the plain epilogues: f32 [group][128] bias (1 KB); integer kind
    // [3][group][128]: za * colsum, scale product, bias (3 KB)
    L.bias = reinterpret_cast<float*>(base + 1024);
    L.smem = base + (KIND == 0 ? 2048 : 4096);
    return L;
}

template <int CTA2>
__device__ __forceinline__ uint32_t kernel_setup(const SmemLayout& L) {
    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(L.res_bar + 8);
    if (warp == 0 && !CTA2) {
        // the producer initialises its own ring barriers and does NOT wait for the rest of the set-up (TMEM allocation,
        // the CTA-wide barrier): it only arrives on a named barrier, so its first TMA is issued that much earlier
        if (lane < 2 * MAX_STAGES) mbar_init(&L.full_bar[lane], 1);  // full_bar and empty_bar are contiguous
        fence_mbar_init();
        __syncwarp();
        asm volatile("bar.arrive 15, %0;" ::"r"(NUM_THREADS) : "memory");
        return 0;  // (the producer never touches TMEM)
    }
    if (warp == 1) {
        // one barrier per lane (a single thread initialising them serially sat on the start-up critical path):
        // lanes 0-15 ring full / empty (pair mode only, else the producer's), 16-17 accumulator full, 18-19 accumulator
        // empty, 20-27 residual
        if (lane < 2 * MAX_STAGES) {
            if (CTA2) mbar_init(&L.full_bar[lane], 1);
        } else if (lane < 2 * MAX_STAGES + 2) {
            mbar_init(&L.tmem_full[lane - 2 * MAX_STAGES], 1);
        } else if (lane < 2 * MAX_STAGES + 4) {
            mbar_init(&L.tmem_empty[lane - 2 * MAX_STAGES - 2], CTA2 ? 16 : 8);  // one arrival per epilogue warp (of both CTAs of a pair)
        } else if (lane < 2 * MAX_STAGES + 12) {
            mbar_init(&L.res_bar[lane - 2 * MAX_STAGES - 4], 1);
        }
        fence_mbar_init();
    }
    if (warp == 2) {
        if (CTA2) {
            tmem_alloc2(tmem_ptr, TMEM_COLS);
            tmem_relinquish2();
        } else {
            tmem_alloc(tmem_ptr, TMEM_COLS);
            tmem_relinquish();
        }
    }
    tc_fence_before();
    if (CTA2)
        cluster_sync_all();  // the peer's barriers must be initialised before any remote arrive / multicast commit
    else
        asm volatile("bar.sync 15, %0;" ::"r"(NUM_THREADS) : "memory");  // 11 warps wait, the producer warp only arrives
    tc_fence_after();
    return *tmem_ptr;
}

template <int CTA2>
__device__ __forceinline__ void kernel_teardown(uint32_t tmem_base) {
    tc_fence_before();
    if (CTA2)
        cluster_sync_all();  // neither CTA may exit (or free TMEM) while the pair's MMAs / remote arrives are in flight
    else
        __syncthreads();
    if ((threadIdx.x >> 5) == 2) {
        tc_fence_after();
        if (CTA2)
            tmem_dealloc2(tmem_base, TMEM_COLS);
        else
            tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

template <int KIND, int FAST, int CTA2>
__global__ void __launch_bounds__(NUM_THREADS, 1)
umma_gemm_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_b,
                 const __grid_constant__ CUtensorMap tma_d, const __grid_constant__ CUtensorMap tma_r,
                 const __grid_constant__ CUtensorMap tma_a2, const __grid_constant__ KParams p) {
    extern __shared__ uint8_t smem_raw[];
    const SmemLayout L = carve_smem<KIND>(smem_raw);
    if (p.trace && blockIdx.x == 0 && threadIdx.x == 0) p.trace[6144 + 1100] = clock64();  // kernel entry
    // CTA pair: cluster rank 0 is the leader (issues the MMAs); work is distributed over clusters
    const int cta_rank = CTA2 ? (int)cluster_ctarank() : 0;
    const int worker = CTA2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int n_workers = CTA2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    if (threadIdx.x == 0) {
        tma_prefetch_desc(&tma_a);
        tma_prefetch_desc(&tma_b);
        if (p.tma_store) tma_prefetch_desc(&tma_d);
        if (p.res_tma) tma_prefetch_desc(&tma_r);
        if (p.x3_cb) tma_prefetch_desc(&tma_a2);
    }
    const uint32_t tmem_base = kernel_setup<CTA2>(L);
    // Programmatic dependent launch: everything above (barrier init, TMEM allocation, descriptor prefetch) overlaps
    // the tail of the previous kernel in the stream; global memory is only touched after this point.
    if (p.trace && blockIdx.x == 0 && threadIdx.x == 0) p.trace[6144 + 1101] = clock64();  // set-up done
    if (threadIdx.x >= 32) asm volatile("griddepcontrol.wait;" ::: "memory");  // (the producer warp waits after its tile decode)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (p.trace && blockIdx.x == 0 && threadIdx.x == 0) p.trace[6144 + 1102] = clock64();  // predecessor complete
    run_layer<KIND, FAST, CTA2>(p, &tma_a, &tma_a2, &tma_b, &tma_d, &tma_r, L, tmem_base, cta_rank, worker, n_workers);
    if (p.trace && blockIdx.x == 0 && threadIdx.x == 0) p.trace[6144 + 1103] = clock64();  // control thread done
    kernel_teardown<CTA2>(tmem_base);
    if (p.trace && blockIdx.x == 0 && threadIdx.x == 0) p.trace[6144 + 1104] = clock64();  // exit
}

}  // namespace rtb
