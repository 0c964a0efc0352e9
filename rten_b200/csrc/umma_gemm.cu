// tcgen05 GEMM / implicit-GEMM convolution for sm_100a.
//
// Replaces rten-gemm's packed BLIS-style GEMM (rten-gemm/src/lib.rs:794-1093, micro-kernels
// rten-gemm/src/kernels/simd_generic.rs:285,576) and the im2col packing
// (rten-gemm/src/im2col.rs:110-389) on the MatMul / MatMulInteger / Conv / ConvInteger path.
//
// Persistent, warp-specialised kernel, one CTA of 384 threads per SM (or one CTA per SM of a CTA pair):
//   warp 0   : TMA producer   -- cp.async.bulk.tensor tiles of A (128 rows x 128 B, two of them in pair mode) and B
//                                (bn rows x 128 B; half of them per CTA in CTA-pair mode) into a ring of 128B-swizzled
//                                shared-memory stages; starts before the rest of the CTA has finished its set-up
//   warp 1   : MMA issuer     -- one elected thread issues tcgen05.mma (kind::tf32 or kind::i8, cta_group::1 or ::2),
//                                4 instructions per 128-byte K block, accumulating in TMEM
//   warp 2   : TMEM allocator -- 512 columns = 2 accumulator stages of up to 256 columns (or one of 512)
//   warps 4-11: epilogue      -- two groups of 4 warps, each taking every other 32-column chunk of the tile:
//                                tcgen05.ld accumulator rows -> registers -> fused epilogue (alpha, residual /
//                                beta*C, bias, activation; or the integer zero-point correction, cast*scale, bias,
//                                residual, activation; optionally the output's min / max) -> 128B-swizzled smem
//                                staging -> cp.async.bulk.tensor store (full-line writes; TMA clips rows/columns
//                                outside the output).  Outputs whose rows are not contiguous fall back to direct
//                                register->global stores.  Runs concurrently with the next tile's main loop thanks
//                                to the second TMEM stage.
// Work decomposition (tile width, pair, split-K, CTA pair ...) is a launch `Plan` (see "Launch plans" below), ranked by
// a cost model and, optionally, measured on the device per problem.
// For Conv the A tile is a TMA box over the NHWC activation tensor at (c0, ox0*sx - pad + kx*dx,
// oy0*sy - pad + ky*dy, b0): padding comes from TMA out-of-bounds zero fill, the stride from the
// tensor map's element strides; the im2col matrix is never materialised.
#include <cuda.h>
#include <cuda_runtime.h>

#include <algorithm>
#include <array>
#include <cmath>
#include <vector>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>

#include "math.cuh"
#include "ptx.cuh"
#include "rowops.h"
#include "umma_gemm.h"
#include "umma_kernel.cuh"  // device side: KParams, the kernels

namespace rtb {

// ------------------------------------------------------------------------------------------
// Host side
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode(rten_ctx* ctx) {
    if (!ctx->encode_tiled) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess ||
            qres != cudaDriverEntryPointSuccess)
            return nullptr;
        ctx->encode_tiled = fn;
    }
    return reinterpret_cast<EncodeTiledFn>(ctx->encode_tiled);
}

bool tma_compatible(const OperandDesc& od, int esize, int rank) {
    if (reinterpret_cast<uintptr_t>(od.base) & 15) return false;
    if (od.strides[0] != 1) return false;
    for (int i = 1; i < rank; i++) {
        if (od.dims[i] > 1) {
            if ((od.strides[i] * esize) % 16 != 0) return false;
            if (od.strides[i] * esize >= (1ll << 40)) return false;
        }
    }
    for (int i = 0; i < rank; i++)
        if (od.dims[i] < 1 || od.dims[i] > 0xFFFFFFFFll) return false;
    return true;
}

bool encode_map(rten_ctx* ctx, CUtensorMap* map, const OperandDesc& od, int esize, bool is_f32,
                const uint32_t box[4], const uint32_t estr[4]) {
    EncodeTiledFn enc = get_encode(ctx);
    if (!enc) return false;
    cuuint64_t dims[4];
    cuuint64_t strides[3];
    cuuint32_t b[4], es[4];
    for (int i = 0; i < 4; i++) {
        dims[i] = (cuuint64_t)od.dims[i];
        b[i] = box[i];
        es[i] = estr[i];
    }
    for (int i = 1; i < 4; i++) {
        long long s = od.strides[i] * esize;
        // size-1 / broadcast dims: any legal multiple of 16 works, the coordinate is always 0
        if (s == 0 || od.dims[i] == 1) s = 16;
        strides[i - 1] = (cuuint64_t)s;
    }
    CUresult r = enc(map, is_f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_UINT8, 4,
                     const_cast<void*>(od.base), dims, strides, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

// Pick the output-pixel box (tw x th x tb <= 128 rows) that wastes the fewest MMA rows.
static void pick_conv_tile(const ConvGeom& g, int& tw, int& th, int& tb) {
    double best = -1.0;
    tw = th = tb = 1;
    for (int w = 1; w <= std::min(g.OW, 128); w++) {
        if (w * g.sx > 256) break;
        for (int h = 1; h <= std::min(g.OH, 128 / w); h++) {
            if (h * g.sy > 256) break;
            int b = std::min(g.B, 128 / (w * h));
            if (b < 1) continue;
            long long tiles = (long long)((g.OW + w - 1) / w) * ((g.OH + h - 1) / h) * ((g.B + b - 1) / b);
            double eff = (double)g.B * g.OH * g.OW / ((double)tiles * 128.0);
            // prefer wider boxes on ties (longer contiguous runs for TMA and the epilogue)
            if (eff > best + 1e-9 || (eff > best - 1e-9 && w > tw)) {
                best = eff;
                tw = w;
                th = h;
                tb = b;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// Launch plans
// ------------------------------------------------------------------------------------------
// A plan fixes the tile shape and the work decomposition of one launch.  Plans come from (a) the cost model below or
// (b) the per-context autotune cache: with rten_b200_set_autotune(ctx, 1) the first launch of every distinct problem
// times the model's best candidates on the device (CUDA events on the context stream) and remembers the winner.
struct Plan {
    int bn = 32, pair = 0, katoms = 1, ksplit = 0, splitk = 1, nbuf = 1, acc1 = 0, cta2 = 0;
};

// Everything about a launch that does not depend on the plan.
struct Prepared {
    KParams p;  // geometry filled in; plan-dependent fields zero
    uint32_t abox[4], aes[4], bbox_k;
    uint32_t a_rows;
    long long batch;
    OperandDesc od, ord;
    uint32_t dbox[4];
    int tma_store, res_tma;  // eligibility
    int step;
    int esize, kelems;
};

constexpr int SK_CNT_INTS = 1 << 16;
// 1 KB alignment slack, 1 KB barriers, column vectors of the plain epilogues (f32: 1 KB, integer kind: 3 KB)
static int smem_budget_for(int n_stg, int kind) { return 227 * 1024 - (kind == 0 ? 3072 : 5120) - n_stg * STG_BYTES; }

struct PlanShape {
    long long tiles_n, units_m, tiles, units;
    int kb_per, atom_bytes, stage_bytes, stages, n_stg;
};

// Derived sizes of a plan; false if the plan cannot run (TMEM columns, shared memory, counters).
static bool plan_shape(const Prepared& q, const Plan& pl, PlanShape& ps) {
    const KParams& p = q.p;
    if (pl.bn < 16 || pl.bn > 256 || pl.bn % q.step) return false;
    if (pl.pair && p.tiles_m < 2) return false;
    if (pl.cta2 && (p.tiles_m < 2 || pl.bn % 32)) return false;
    if (pl.acc1 != ((pl.pair && pl.bn > 128) ? 1 : 0)) return false;
    if (pl.ksplit && (pl.pair || pl.bn > 128 || pl.splitk > 1)) return false;
    ps.tiles_n = (p.N + pl.bn - 1) / pl.bn;
    const int mult = (pl.pair + 1) * (pl.cta2 + 1);
    ps.units_m = (p.tiles_m + mult - 1) / mult;
    ps.tiles = ps.units_m * ps.tiles_n * q.batch;
    ps.units = ps.tiles * pl.splitk;
    if (ps.units > 0x7FFFFFFFll) return false;
    ps.kb_per = (p.k_blocks + pl.splitk - 1) / pl.splitk;
    if (pl.splitk > 1) {
        if (pl.bn % 32 || (long long)(pl.splitk - 1) * ps.kb_per >= p.k_blocks) return false;  // no empty split
        if (ps.tiles * 2 * (pl.cta2 + 1) > SK_CNT_INTS) return false;
    }
    ps.n_stg = 2 * pl.nbuf;
    ps.atom_bytes = (pl.pair ? 2 : 1) * A_STAGE_BYTES + (pl.bn >> pl.cta2) * KBYTES;  // pair mode: half of B per CTA
    if (pl.katoms == 2 && ps.kb_per < 2) return false;
    ps.stage_bytes = ps.atom_bytes * pl.katoms;
    ps.stages = std::min(MAX_STAGES, smem_budget_for(ps.n_stg, q.esize == 4 ? 0 : 1) / ps.stage_bytes);
    if (ps.stages < 2) return false;
    return true;
}

// Cost model in SM clocks.  Constants measured with the in-kernel trace (tools/trace_probe.py,
// profiles/r01_trace_pipeline.txt) and from whole-layer timings:
//   * the operand stream L2 -> shared memory is the first limit: ~7400 B/clk for the whole chip (all SMs loading),
//     at most ~64 B/clk for one SM -> a K block of `atom_bytes` cannot take less than atom_bytes / bw;
//   * the tensor pipe needs bn/2 clk per 128 x bn x 32-byte MMA, the elected thread ~42 clk to issue it;
//   * every pipeline stage costs the issuing warp a fixed ~320 clk (barrier wait, fence, descriptors, commit);
//   * a stage cannot complete faster than TMA latency (~2300 clk under load) / stages in flight;
//   * the epilogue (~350 clk per 32-column chunk, two warp groups) overlaps the next main loop unless acc1.
static double plan_cost(const Prepared& q, const Plan& pl, const PlanShape& ps, int num_sms) {
    const int workers = pl.cta2 ? num_sms / 2 : num_sms;
    const double active = (double)std::min<long long>(ps.units, workers) * (pl.cta2 + 1);
    const double waves = std::ceil((double)ps.units / workers);
    const double bw = std::min(64.0, 7400.0 / active);
    const double mmas = 4.0 * (pl.pair ? 2 : 1);
    const double t_kb = std::max(mmas * std::max(42.0, pl.bn / 2.0), ps.atom_bytes / bw);
    double t_stage = std::max(pl.katoms * t_kb, 320.0 + pl.katoms * mmas * 42.0);
    t_stage = std::max(t_stage, 2300.0 / ps.stages);
    const double mainloop = std::ceil((double)ps.kb_per / pl.katoms) * t_stage;
    const double epi = (pl.pair ? 2 : 1) * (pl.bn / 32.0) * 350.0 / 2.0 + 600.0;
    double unit = pl.acc1 ? mainloop + epi + 1000.0 : std::max(mainloop, epi) + 1500.0;
    double cost = waves * unit + 2500.0;
    if (pl.splitk > 1) cost += epi * (1.0 + 0.25 * pl.splitk) + 1500.0;  // publish + the owner's reduction

    return cost;
}

static void enumerate_plans(const Prepared& q, int num_sms, std::vector<std::pair<double, Plan>>& out) {
    const KParams& p = q.p;
    const int nmax = (p.N + q.step - 1) / q.step * q.step;
    static const int splits[] = {1, 2, 3, 4, 5, 6, 8, 10, 12, 16};
    const bool allow_cta2 = !getenv("RTEN_B200_NO_CTA2");
    for (int cta2 = 0; cta2 <= (allow_cta2 ? 1 : 0); cta2++)
    for (int pair = 0; pair <= 1; pair++)
        for (int bn = q.step; bn <= 256; bn += q.step) {
            if (bn > nmax && bn != q.step) break;
            for (int katoms = 1; katoms <= 2; katoms++)
                for (int sk : splits) {
                    Plan pl;
                    pl.cta2 = cta2;
                    pl.bn = bn;
                    pl.pair = pair;
                    pl.katoms = katoms;
                    pl.splitk = sk;
                    pl.acc1 = (pair && bn > 128) ? 1 : 0;
                    if (sk > 1 && p.k_blocks / sk < 4) continue;
                    pl.ksplit = (!pair && bn <= 128 && sk == 1 && !getenv("RTEN_B200_NO_KSPLIT")) ? 1 : 0;
                    const int kb_per = (p.k_blocks + sk - 1) / sk;
                    pl.nbuf = pl.acc1 ? 1 : ((q.res_tma || kb_per < 24) ? 2 : 1);
                    PlanShape ps;
                    if (pl.nbuf == 2 && !getenv("RTEN_B200_NO_NBUF3")) {
                        // A third staging buffer per group takes the wait for the previous store's shared-memory read (a
                        // 16 KB bulk store drains at the SM's ~32 B/clk write port: ~900 clk) and, with a residual, the
                        // late request of the next residual tile off the chunk's critical path -- as long as the operand
                        // ring keeps three stages (or loses none)
                        PlanShape ps2;
                        const bool ok2 = plan_shape(q, pl, ps2);
                        pl.nbuf = 3;
                        if (!plan_shape(q, pl, ps) || (ps.stages < 3 && !(ok2 && ps.stages == ps2.stages))) pl.nbuf = 2;
                    }
                    if (!plan_shape(q, pl, ps)) continue;
                    if (sk > 1 && ps.tiles * (cta2 + 1) >= 2 * num_sms) continue;  // enough parallelism without splitting K
                    if (ps.stages < 3 && !(katoms == 1 && ps.stages == 2)) continue;
                    out.emplace_back(plan_cost(q, pl, ps, num_sms), pl);
                }
        }
    std::sort(out.begin(), out.end(), [](const std::pair<double, Plan>& x, const std::pair<double, Plan>& y) {
        return x.first < y.first;
    });
}

static rten_status prepare_launch(rten_ctx* ctx, const GemmLaunch& L, Prepared& q) {
    const int esize = L.kind == 0 ? 4 : 1;
    const int kelems = KBYTES / esize;
    if (!tma_compatible(L.a, esize, 4) || !tma_compatible(L.b, esize, 4)) return RTEN_ERR_UNSUPPORTED_VALUE;
    if (L.M <= 0 || L.N <= 0 || L.K <= 0) return RTEN_ERR_UNSUPPORTED_VALUE;
    q.esize = esize;
    q.kelems = kelems;
    KParams& p = q.p;
    memset(&p, 0, sizeof(p));
    p.M = L.M;
    p.N = L.N;
    p.K = L.K;
    p.z0 = L.z0;
    p.z1 = L.z1;
    p.kelems = kelems;
    p.conv = L.conv;
    p.epi = L.epi;
    p.trace = reinterpret_cast<long long*>(ctx->trace);
    p.c_blocks = 1;
    p.kw = 1;
    for (int i = 0; i < 4; i++) q.aes[i] = 1;
    if (L.conv) {
        const ConvGeom& g = L.g;
        pick_conv_tile(g, p.tw, p.th, p.tb);
        p.tiles_x = (g.OW + p.tw - 1) / p.tw;
        p.tiles_y = (g.OH + p.th - 1) / p.th;
        int tiles_b = (g.B + p.tb - 1) / p.tb;
        p.tiles_m = p.tiles_x * p.tiles_y * tiles_b;
        p.OH = g.OH;
        p.OW = g.OW;
        p.Bn = g.B;
        p.sy = g.sy;
        p.sx = g.sx;
        p.dy = g.dy;
        p.dx = g.dx;
        p.pt = g.pt;
        p.pl = g.pl;
        p.kw = g.kw;
        p.c_blocks = (g.C + kelems - 1) / kelems;
        p.k_blocks = g.kh * g.kw * p.c_blocks;
        p.z0 = p.z1 = 1;
        q.abox[0] = kelems;
        q.abox[1] = p.tw * g.sx;
        q.abox[2] = p.th * g.sy;
        q.abox[3] = p.tb;
        q.aes[1] = g.sx;
        q.aes[2] = g.sy;
        q.a_rows = p.tw * p.th * p.tb;
        q.batch = 1;
    } else {
        p.tiles_m = (L.M + BM - 1) / BM;
        p.k_blocks = (L.K + kelems - 1) / kelems;
        q.abox[0] = kelems;
        q.abox[1] = BM;
        q.abox[2] = 1;
        q.abox[3] = 1;
        q.a_rows = BM;
        q.batch = (long long)L.z0 * L.z1;
        p.a_bcast0 = (L.a.dims[2] == 1 && L.z0 > 1) ? 1 : 0;
        p.a_bcast1 = (L.a.dims[3] == 1 && L.z1 > 1) ? 1 : 0;
        p.b_bcast0 = (L.b.dims[2] == 1 && L.z0 > 1) ? 1 : 0;
        p.b_bcast1 = (L.b.dims[3] == 1 && L.z1 > 1) ? 1 : 0;
    }
    // ---- output path: TMA store needs contiguous 4-byte rows at 16-byte aligned pitches
    OperandDesc& od = q.od;
    OperandDesc& ord = q.ord;
    q.dbox[0] = 32;
    q.dbox[1] = q.dbox[2] = q.dbox[3] = 1;
    const EpilogueDesc& e = L.epi;
    od.base = e.d;
    od.dims[0] = L.N;
    od.strides[0] = 1;
    if (L.conv) {
        od.dims[1] = L.g.OW;
        od.dims[2] = L.g.OH;
        od.dims[3] = L.g.B;
        od.strides[1] = e.s_z1;
        od.strides[2] = e.s_row;
        od.strides[3] = e.s_z0;
        q.dbox[1] = p.tw;
        q.dbox[2] = p.th;
        q.dbox[3] = p.tb;
    } else {
        od.dims[1] = L.M;
        od.dims[2] = L.z0;
        od.dims[3] = L.z1;
        od.strides[1] = e.s_row;
        od.strides[2] = e.s_z0;
        od.strides[3] = e.s_z1;
        q.dbox[1] = BM;
    }
    q.tma_store = (e.s_col == 1 && L.N >= 4 && tma_compatible(od, 4, 4)) ? 1 : 0;
    if (getenv("RTEN_B200_NO_TMA_STORE")) q.tma_store = 0;
    // residual prefetched by TMA: same geometry as the output, own strides (fast-path epilogue only)
    ord = od;
    ord.base = e.r;
    if (L.conv) {
        ord.strides[1] = e.r_z1;
        ord.strides[2] = e.r_row;
        ord.strides[3] = e.r_z0;
    } else {
        ord.strides[1] = e.r_row;
        ord.strides[2] = e.r_z0;
        ord.strides[3] = e.r_z1;
    }
    q.res_tma = (q.tma_store && (L.kind == 0 || e.scale) && e.r && e.r_col == 1 && (L.N % 32) == 0 &&
                 (e.bias_kind != 1 || (reinterpret_cast<uintptr_t>(e.bias) & 15) == 0) && tma_compatible(ord, 4, 4))
                    ? 1
                    : 0;
    // a broadcast residual (Gemm's C) has zero strides on real dims: keep the register path for it
    for (int i = 1; i < 4; i++)
        if (ord.dims[i] > 1 && ord.strides[i] == 0) q.res_tma = 0;
    if (getenv("RTEN_B200_NO_RES_TMA")) q.res_tma = 0;
    p.res_tx_bytes = q.a_rows * KBYTES;
    q.step = q.tma_store ? 32 : 16;
    return RTEN_OK;
}

static size_t splitk_ws_bytes(const PlanShape& ps, const Plan& pl) {
    return pl.splitk > 1 ? (size_t)ps.tiles * (pl.cta2 + 1) * 2 * pl.splitk * (pl.bn / 32) * 4096 * 4 : 0;
}

static rten_status ensure_splitk_counters(rten_ctx* ctx) {
    if (!ctx->sk_counters) {
        cudaError_t ce = cudaMalloc(&ctx->sk_counters, SK_CNT_INTS * sizeof(int));
        if (ce != cudaSuccess) return fail_cuda(ctx, ce, "split-K counters");
        ce = cudaMemset(ctx->sk_counters, 0, SK_CNT_INTS * sizeof(int));
        if (ce != cudaSuccess) return fail_cuda(ctx, ce, "split-K counters");
    }
    return RTEN_OK;
}

struct LaunchArgs {
    bool plain = false;  // f32 launch that qualifies for the plain epilogue (kernel variant 3; a subset of variant 1)
    KParams p;
    CUtensorMap maps[5];  // a, b, d, residual, a2 (two-plane 3xTF32: low parts of A)
    size_t smem_bytes;
};

// cls = kind * 3 + epilogue variant
static rten_status launch_single(rten_ctx* ctx, int cls, const LaunchArgs& pl) {
    const KParams& p = pl.p;
    const int grid = p.cta2 ? 2 * std::min(p.units_total, ctx->num_sms / 2) : std::min(p.units_total, ctx->num_sms);
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = pl.smem_bytes;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[2];
    fill_launch_attrs(cfg, attr, p.cta2 != 0);
    auto launch = [&](auto kern) -> cudaError_t {
        cudaError_t e2 = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e2 != cudaSuccess) return e2;
        return cudaLaunchKernelEx(&cfg, kern, pl.maps[0], pl.maps[1], pl.maps[2], pl.maps[3], pl.maps[4], p);
    };
    cudaError_t e;
    if (pl.plain && cls == 1) {
        e = p.cta2 ? launch(umma_gemm_kernel<0, 3, 1>) : launch(umma_gemm_kernel<0, 3, 0>);
    } else if (pl.plain && cls == 2) {
        e = p.cta2 ? launch(umma_gemm_kernel<0, 5, 1>) : launch(umma_gemm_kernel<0, 5, 0>);
    } else if (pl.plain && cls == 5) {
        e = p.cta2 ? launch(umma_gemm_kernel<1, 6, 1>) : launch(umma_gemm_kernel<1, 6, 0>);
    } else if (pl.plain && cls == 4) {
        e = p.cta2 ? launch(umma_gemm_kernel<1, 4, 1>) : launch(umma_gemm_kernel<1, 4, 0>);
    } else
    switch (cls * 2 + (p.cta2 ? 1 : 0)) {
        case 0: e = launch(umma_gemm_kernel<0, 0, 0>); break;
        case 1: e = launch(umma_gemm_kernel<0, 0, 1>); break;
        case 2: e = launch(umma_gemm_kernel<0, 1, 0>); break;
        case 3: e = launch(umma_gemm_kernel<0, 1, 1>); break;
        case 4: e = launch(umma_gemm_kernel<0, 2, 0>); break;
        case 5: e = launch(umma_gemm_kernel<0, 2, 1>); break;
        case 6: e = launch(umma_gemm_kernel<1, 0, 0>); break;
        case 7: e = launch(umma_gemm_kernel<1, 0, 1>); break;
        case 8: e = launch(umma_gemm_kernel<1, 1, 0>); break;
        case 9: e = launch(umma_gemm_kernel<1, 1, 1>); break;
        case 10: e = launch(umma_gemm_kernel<1, 2, 0>); break;
        default: e = launch(umma_gemm_kernel<1, 2, 1>); break;
    }
    if (e != cudaSuccess) return fail_cuda(ctx, e, "umma_gemm launch");
    e = cudaGetLastError();
    if (e != cudaSuccess) return fail_cuda(ctx, e, "umma_gemm launch");
    count_launch(ctx);
    return RTEN_OK;
}

// `ws`: split-K workspace of at least splitk_ws_bytes() (null: taken from the op's temporaries)
static rten_status launch_plan(rten_ctx* ctx, const GemmLaunch& L, const Prepared& q, const Plan& pl, bool verbose, void* ws = nullptr) {
    PlanShape ps;
    if (!plan_shape(q, pl, ps)) return RTEN_ERR_UNSUPPORTED_VALUE;
    KParams p = q.p;
    p.bn = pl.bn;
    p.pair = pl.pair;
    p.katoms = pl.katoms;
    p.ksplit = pl.ksplit;
    p.splitk = pl.splitk;
    p.acc1 = pl.acc1;
    p.cta2 = pl.cta2;
    p.nbuf = pl.nbuf;
    p.tma_store = q.tma_store;
    p.res_tma = q.res_tma ? 1 : 0;
    if (p.res_tma && p.nbuf < 2) p.nbuf = 2;
    p.kb_per = ps.kb_per;
    p.tiles_n = (int)ps.tiles_n;
    p.tiles_total = (int)ps.tiles;
    p.units_total = (int)ps.units;
    p.d_tiles_n.set(p.tiles_n);
    p.d_units_m.set((int)ps.units_m);
    p.d_z0.set(p.z0);
    p.d_tiles_x.set(p.conv ? p.tiles_x : 1);
    p.d_tiles_y.set(p.conv ? p.tiles_y : 1);
    p.d_tiles_total.set(p.tiles_total);
    p.d_c_blocks.set(p.c_blocks);
    p.d_kw.set(p.kw);
    p.d_tw.set(p.conv ? p.tw : 1);
    p.d_th.set(p.conv ? p.th : 1);
    const int n_stg = 2 * p.nbuf;
    p.atom_bytes = ps.atom_bytes;
    p.stage_bytes = ps.stage_bytes;
    p.tx_bytes = (p.pair ? 2 : 1) * q.a_rows * KBYTES + (p.bn >> p.cta2) * KBYTES;  // per 128-byte K block and CTA
    p.stages = std::min(MAX_STAGES, smem_budget_for(n_stg, L.kind) / (int)p.stage_bytes);
    if (p.stages < 2) return RTEN_ERR_UNSUPPORTED_VALUE;
    if (L.kind == 0)
        p.idesc = make_idesc(1 /*F32*/, 2 /*TF32*/, 2, BM << p.cta2, p.bn);
    else
        p.idesc = make_idesc(2 /*S32*/, L.a_signed ? 1 : 0, L.b_signed ? 1 : 0, BM << p.cta2, p.bn);
    if (p.splitk > 1) {
        RTB_TRY(ensure_splitk_counters(ctx));
        if (!ws) RTB_TRY(temp_alloc(ctx, splitk_ws_bytes(ps, pl), &ws));
        p.sk_ws = reinterpret_cast<uint32_t*>(ws);
        p.sk_cnt = reinterpret_cast<int*>(ctx->sk_counters);
    }

    uint32_t bbox[4] = {(uint32_t)q.kelems, (uint32_t)(p.bn >> p.cta2), 1, 1}, bes[4] = {1, 1, 1, 1}, des[4] = {1, 1, 1, 1};
    CUtensorMap map_a, map_b;
    if (!encode_map(ctx, &map_a, L.a, q.esize, L.kind == 0, q.abox, q.aes)) return RTEN_ERR_UNSUPPORTED_VALUE;
    if (!encode_map(ctx, &map_b, L.b, q.esize, L.kind == 0, bbox, bes)) return RTEN_ERR_UNSUPPORTED_VALUE;
    CUtensorMap map_d = map_a, map_r = map_a, map_a2 = map_a;
    p.x3_cb = L.x3_cb;
    if (L.x3_cb && !encode_map(ctx, &map_a2, L.a_lo, q.esize, true, q.abox, q.aes)) return RTEN_ERR_UNSUPPORTED_VALUE;
    if (p.tma_store && !encode_map(ctx, &map_d, q.od, 4, true, q.dbox, des)) {
        p.tma_store = 0;  // direct stores still work for any bn that is a multiple of 16
        p.res_tma = 0;
        map_d = map_a;
    }
    if (p.res_tma && !encode_map(ctx, &map_r, q.ord, 4, true, q.dbox, des)) {
        p.res_tma = 0;
        map_r = map_a;
    }

    if (verbose)
        fprintf(stderr, "[umma_gemm] kind=%d conv=%d M=%d N=%d K=%d kb=%d tiles_m=%d bn=%d pair=%d ksplit=%d katoms=%d splitk=%d acc1=%d cta2=%d units=%d stages=%d tma_store=%d res_tma=%d nbuf=%d box=%dx%dx%d\n",
                L.kind, L.conv, L.M, L.N, L.K, p.k_blocks, p.tiles_m, p.bn, p.pair, p.ksplit, p.katoms, p.splitk, p.acc1, p.cta2,
                p.units_total, p.stages, p.tma_store, p.res_tma, p.nbuf, p.tw, p.th, p.tb);
    const size_t smem_bytes = (size_t)p.stages * p.stage_bytes + n_stg * STG_BYTES + 1024 /*align*/ + 1024 /*barriers*/ + (L.kind == 0 ? 1024 : 3072) /*column vectors*/;
    // specialised epilogue when every chunk qualifies for the register fast path
    const EpilogueDesc& ee = L.epi;
    bool fastk = p.tma_store && (L.N % 32) == 0 && (!ctx->trace || getenv("RTEN_B200_TRACE_FAST")) && !getenv("RTEN_B200_NO_FAST");
    if (L.kind == 0)
        fastk = fastk && ee.bias_kind != 2 && (ee.r == nullptr || p.res_tma) &&
                (ee.bias_kind != 1 || (reinterpret_cast<uintptr_t>(ee.bias) & 15) == 0);
    else  // integer: column vectors must be 128-bit loadable, zero-point / scale vectors per column or scalar
        fastk = fastk && ee.bias_kind != 2 && (ee.r == nullptr || p.res_tma) &&
                (ee.bias_kind != 1 || (reinterpret_cast<uintptr_t>(ee.bias) & 15) == 0) &&
                (!(ee.za || ee.za8) || (reinterpret_cast<uintptr_t>(ee.colsum) & 15) == 0) &&
                (!ee.zb || ee.zb_len == 1 || (ee.zb_len == L.N && (reinterpret_cast<uintptr_t>(ee.zb) & 15) == 0)) &&
                (!ee.scale || ee.scale_len == 1 || (ee.scale_len == L.N && (reinterpret_cast<uintptr_t>(ee.scale) & 15) == 0));
    // the generic epilogue takes a TMA-staged residual only on its register path (f32, act <= Relu)
    if (!fastk && (L.kind == 1 || ee.act > 1)) p.res_tma = 0;
    LaunchArgs args;
    if (L.kind == 0)
        args.plain = fastk && ee.alpha == 1.0f && ee.act <= 3 && !ee.range && (ee.r == nullptr || (p.res_tma && ee.r_scale == 1.0f));
    else  // integer kind: the *ToFloat operators with a scalar (or no) activation zero point and symmetric weights
        args.plain = fastk && ee.scale && !ee.za && !ee.zb && (ee.scale_len == 1 || ee.scale_len == L.N) && ee.act <= 3 && p.splitk == 1 &&
                     (ee.r == nullptr || p.res_tma) && (!ee.za8 || ee.colsum);
    if (getenv("RTEN_B200_NO_PLAIN")) args.plain = false;
    args.p = p;
    args.maps[0] = map_a;
    args.maps[1] = map_b;
    args.maps[2] = map_d;
    args.maps[3] = map_r;
    args.maps[4] = map_a2;
    args.smem_bytes = smem_bytes;
    // kernel class = data kind x epilogue variant (0 generic, 1 specialised, 2 specialised + out-of-line Gelu)
    const int cls = L.kind * 3 + (fastk ? (ee.act > 1 ? 2 : 1) : 0);
    return launch_single(ctx, cls, args);
}

// Problem signature for the autotune cache: everything that changes which plan is fastest.
static std::vector<long long> tune_key(const GemmLaunch& L, const Prepared& q) {
    const EpilogueDesc& e = L.epi;
    std::vector<long long> k = {L.kind, L.conv, L.M, L.N, L.K, L.z0, L.z1, q.tma_store, q.res_tma, e.act, e.bias_kind,
                                e.r != nullptr, (e.za != nullptr || e.za8 != nullptr), e.zb != nullptr, e.scale != nullptr,
                                L.a.strides[1], L.b.strides[1], L.x3_cb};
    if (L.conv) {
        const ConvGeom& g = L.g;
        for (long long v : {g.B, g.H, g.W, g.C, g.OH, g.OW, g.kh, g.kw, g.sy, g.sx, g.dy, g.dx, g.pt, g.pl}) k.push_back(v);
    }
    return k;
}

static Plan plan_from_array(const std::array<int, 8>& a) {
    Plan pl;
    pl.bn = a[0];
    pl.pair = a[1];
    pl.katoms = a[2];
    pl.ksplit = a[3];
    pl.splitk = a[4];
    pl.nbuf = a[5];
    pl.acc1 = a[6];
    pl.cta2 = a[7];
    return pl;
}

// RTEN_F32_TF32X3: run the same kernel over split operands -- K (plain) or C (conv; K order is (ky, kx, c)) tripled:
// A' = [lo | hi | hi], B' = [hi | lo | hi]  =>  lo*hi + hi*lo + hi*hi, small terms first.
//  * B: a constant operand (prepacked weights, `b_x3_slot`) is split ONCE and cached with its owner.
//  * A: kind::tf32 ignores the 13 low mantissa bits, so the ORIGINAL tensor serves as both `hi` segments; only the low
//    parts are written (4 B / element instead of 12) and the kernel's producer switches tensor maps per segment
//    (KParams::x3_cb).  Needs K (C) % 32 == 0 and a TMA-addressable A; otherwise the three-segment copy is built.
static rten_status launch_tf32x3(rten_ctx* ctx, const GemmLaunch& L0) {
    GemmLaunch L = L0;
    const long long d0 = L0.a.dims[0];               // K, or channels per group
    const long long d0p = (d0 + 3) / 4 * 4;          // thirds stay 16-byte aligned for TMA
    auto split = [&](const OperandDesc& src, OperandDesc& dst, int role, void* into) -> rten_status {
        const long long planes = role == 2 ? 1 : 3;
        long long dims[4], strides[4], n = planes * d0p;
        for (int i = 0; i < 4; i++) {
            // broadcast dims (stride 0) are split once and stay broadcast
            dims[i] = (i > 0 && src.strides[i] == 0) ? 1 : src.dims[i];
            strides[i] = src.strides[i];
        }
        for (int i = 1; i < 4; i++) n *= dims[i];
        void* buf = into;
        if (!buf) RTB_TRY(temp_alloc(ctx, (size_t)n * 4, &buf));
        RTB_TRY(launch_tf32x3_split(ctx, (const float*)src.base, (float*)buf, dims, strides, d0p, role));
        dst = src;
        dst.base = buf;
        dst.dims[0] = planes * d0p;
        long long st = planes * d0p;
        for (int i = 1; i < 4; i++) {
            dst.strides[i] = (src.strides[i] == 0 && src.dims[i] > 1) ? 0 : st;
            st *= dims[i];
        }
        return RTEN_OK;
    };
    if (L0.b.dims[0] != d0) return RTEN_ERR_UNSUPPORTED_VALUE;
    // ---- B
    if (L0.b_x3_slot && !getenv("RTEN_B200_X3_NO_CACHE")) {
        if (!*L0.b_x3_slot && !ctx->capturing) {
            long long n = 3 * d0p;
            for (int i = 1; i < 4; i++) n *= (L0.b.strides[i] == 0 ? 1 : L0.b.dims[i]);
            void* buf = nullptr;
            if (cudaMalloc(&buf, (size_t)n * 4) != cudaSuccess) return fail(ctx, RTEN_ERR_CUDA, "cudaMalloc failed for the 3xTF32 copy of a prepacked operand");
            OperandDesc tmp;
            const rten_status st = split(L0.b, tmp, 1, buf);
            if (st != RTEN_OK) {
                cudaFree(buf);
                return st;
            }
            *L0.b_x3_slot = buf;
        }
    }
    if (L0.b_x3_slot && *L0.b_x3_slot && !getenv("RTEN_B200_X3_NO_CACHE")) {
        L.b = L0.b;
        L.b.base = *L0.b_x3_slot;
        L.b.dims[0] = 3 * d0p;
        long long st = 3 * d0p;
        for (int i = 1; i < 4; i++) {
            const long long di = L0.b.strides[i] == 0 ? 1 : L0.b.dims[i];
            L.b.strides[i] = (L0.b.strides[i] == 0 && L0.b.dims[i] > 1) ? 0 : st;
            st *= di;
        }
    } else {
        RTB_TRY(split(L0.b, L.b, 1, nullptr));
    }
    // ---- A
    const bool two_plane = d0 % 32 == 0 && tma_compatible(L0.a, 4, 4) && !getenv("RTEN_B200_X3_THREE_PLANES");
    if (two_plane && L0.a_lo_base) {
        L.a_lo = L0.a;
        L.a_lo.base = L0.a_lo_base;
        L.x3_cb = (int)(d0 / 32);
    } else if (two_plane) {
        RTB_TRY(split(L0.a, L.a_lo, 2, nullptr));
        L.x3_cb = (int)(d0 / 32);
    } else {
        RTB_TRY(split(L0.a, L.a, 0, nullptr));
    }
    if (L.conv)
        L.g.C = (int)(3 * d0p);
    L.K = L.conv ? (int)(L0.K / d0 * 3 * d0p) : (int)(3 * d0p);
    L.b_x3_slot = nullptr;
    L.a_lo_base = nullptr;
    const int saved = ctx->f32_mode;
    ctx->f32_mode = RTEN_F32_TF32;
    const rten_status st = launch_umma_gemm(ctx, L);
    ctx->f32_mode = saved;
    return st;
}

rten_status launch_umma_gemm(rten_ctx* ctx, const GemmLaunch& L) {
    if (L.kind == 0 && ctx->f32_mode == RTEN_F32_TF32X3) return launch_tf32x3(ctx, L);
    // stride-1 windows (the 3x3 layers): the halo-reuse kernel moves the activations into shared memory once per channel
    // block instead of once per filter tap (umma_halo.cu); everything it does not cover falls through
    if (L.conv && L.kind == 0 && L.g.kh * L.g.kw > 1 && (!ctx->trace || getenv("RTEN_B200_TRACE_FAST")) && !L.x3_cb) {
        const rten_status hs = launch_umma_halo_conv(ctx, L);
        if (hs != RTEN_ERR_UNSUPPORTED_VALUE) return hs;
    }
    Prepared q;
    RTB_TRY(prepare_launch(ctx, L, q));
    const bool verbose = getenv("RTEN_B200_VERBOSE") != nullptr;
    const bool forced = getenv("RTEN_B200_FORCE_BN") || getenv("RTEN_B200_FORCE_PAIR") || getenv("RTEN_B200_FORCE_KATOMS") ||
                        getenv("RTEN_B200_FORCE_SPLITK") || getenv("RTEN_B200_FORCE_CTA2");
    if (!forced && !ctx->tune_cache.empty()) {  // measured plan on record: no need to enumerate and rank candidates
        auto hit = ctx->tune_cache.find(tune_key(L, q));
        if (hit != ctx->tune_cache.end()) {
            PlanShape ps;
            if (hit->second[0] < 0) {  // the halo-reuse kernel measured faster: {-1, bn, T}
                const rten_status hs = launch_umma_halo_conv(ctx, L, hit->second[1], hit->second[2]);
                if (hs != RTEN_ERR_UNSUPPORTED_VALUE) return hs;
            } else
            if (plan_shape(q, plan_from_array(hit->second), ps)) return launch_plan(ctx, L, q, plan_from_array(hit->second), verbose);
            // a stale entry (plans file written by another build / geometry): drop it and plan afresh
            if (verbose) fprintf(stderr, "[umma_gemm] recorded plan no longer valid for this problem: re-planning\n");
            ctx->tune_cache.erase(hit);
        }
    }
    std::vector<std::pair<double, Plan>> cands;
    enumerate_plans(q, ctx->num_sms, cands);
    if (cands.empty()) return RTEN_ERR_UNSUPPORTED_VALUE;
    Plan plan = cands[0].second;

    if (forced) {
        // debugging / sweeps: the best-ranked candidate that matches every forced field
        const char* fb = getenv("RTEN_B200_FORCE_BN");
        const char* fp = getenv("RTEN_B200_FORCE_PAIR");
        const char* fk = getenv("RTEN_B200_FORCE_KATOMS");
        const char* fs = getenv("RTEN_B200_FORCE_SPLITK");
        const char* fc = getenv("RTEN_B200_FORCE_CTA2");
        bool found = false;
        for (const auto& c : cands) {
            const Plan& x = c.second;
            if (fb && x.bn != atoi(fb)) continue;
            if (fp && x.pair != (atoi(fp) ? 1 : 0)) continue;
            if (fk && x.katoms != atoi(fk)) continue;
            if (fs && x.splitk != atoi(fs)) continue;
            if (fc && x.cta2 != (atoi(fc) ? 1 : 0)) continue;
            plan = x;
            found = true;
            break;
        }
        // RTEN_B200_FORCE_STRICT=1 (tests): a forced combination that no valid plan satisfies is an error instead of a
        // silent fall-back to the model's choice -- a sweep must exercise what it names
        if (!found) {
            ctx->forced_misses++;
            if (verbose) fprintf(stderr, "[umma_gemm] no valid plan matches the forced fields: using the model's choice\n");
            if (getenv("RTEN_B200_FORCE_STRICT"))
                return fail(ctx, RTEN_ERR_INVALID_VALUE, "no launch plan matches the forced RTEN_B200_FORCE_* fields");
        } else {
            ctx->forced_hits++;
        }
    } else if (ctx->autotune || !ctx->tune_cache.empty()) {
        // measured plans are used whenever they exist; new measurements are only taken while autotuning is on
        const std::vector<long long> key = tune_key(L, q);
        auto it = ctx->tune_cache.find(key);
        PlanShape ps_hit;
        if (it != ctx->tune_cache.end() && it->second[0] < 0) {
            const rten_status hs = launch_umma_halo_conv(ctx, L, it->second[1], it->second[2]);
            if (hs != RTEN_ERR_UNSUPPORTED_VALUE) return hs;
            ctx->tune_cache.erase(it);
        } else if (it != ctx->tune_cache.end() && plan_shape(q, plan_from_array(it->second), ps_hit)) {
            plan = plan_from_array(it->second);
        } else if (ctx->autotune) {
            cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
            cudaStreamIsCapturing(ctx->stream, &cs);
            // re-running the launch must be idempotent: the output may not alias the residual
            const bool safe = !ctx->capturing && cs == cudaStreamCaptureStatusNone && !ctx->trace &&
                              (L.epi.r == nullptr || (const void*)L.epi.r != (const void*)L.epi.d);
            if (safe) {
                cudaEvent_t e0, e1;
                cudaEventCreate(&e0);
                cudaEventCreate(&e1);
                const size_t ncand = std::min<size_t>(cands.size(), 24);
                // one split-K workspace for every candidate (allocating inside the timed launches would time cudaMalloc)
                size_t ws_max = 0;
                for (size_t i = 0; i < ncand; i++) {
                    PlanShape ps;
                    if (plan_shape(q, cands[i].second, ps)) ws_max = std::max(ws_max, splitk_ws_bytes(ps, cands[i].second));
                }
                void* ws = nullptr;
                if (ws_max) {
                    RTB_TRY(ensure_splitk_counters(ctx));
                    RTB_TRY(temp_alloc(ctx, ws_max, &ws));
                    cudaStreamSynchronize(ctx->stream);
                }
                double best_ms = 1e30;
                int reps = 4;  // raised after the first candidate so that every timed window is >= ~150 us (event resolution)
                std::vector<std::pair<double, size_t>> timed;
                auto time_plan = [&](const Plan& x, int n) -> double {
                    if (launch_plan(ctx, L, q, x, false, ws) != RTEN_OK) return -1.0;  // warm-up (also validates the plan)
                    cudaEventRecord(e0, ctx->stream);
                    bool ok = true;
                    for (int r = 0; r < n && ok; r++) ok = launch_plan(ctx, L, q, x, false, ws) == RTEN_OK;
                    cudaEventRecord(e1, ctx->stream);
                    if (cudaEventSynchronize(e1) != cudaSuccess || !ok) return -1.0;
                    float t = 0.f;
                    cudaEventElapsedTime(&t, e0, e1);
                    return (double)t / n;
                };
                for (size_t i = 0; i < ncand; i++) {
                    const Plan& x = cands[i].second;
                    double ms = time_plan(x, reps);
                    if (ms < 0) continue;
                    timed.emplace_back(ms, i);
                    if (verbose)
                        fprintf(stderr, "[autotune] bn=%d pair=%d katoms=%d splitk=%d cta2=%d model=%.0f -> %.2f us\n", x.bn, x.pair,
                                x.katoms, x.splitk, x.cta2, cands[i].first, ms * 1e3);
                    if (ms < best_ms) {
                        best_ms = ms;
                        plan = x;
                    }
                    reps = std::max(4, std::min(32, (int)(0.15 / std::max(best_ms, 1e-3))));
                }
                // second look at the three fastest with longer windows: single measurements of 20-40 us kernels are noisy
                // enough to flip the choice between near-equal plans from run to run
                std::sort(timed.begin(), timed.end());
                best_ms = 1e30;
                for (size_t k = 0; k < std::min<size_t>(3, timed.size()); k++) {
                    const Plan& x = cands[timed[k].second].second;
                    const double again = time_plan(x, 2 * reps);
                    const double ms = again < 0 ? timed[k].first : again;  // the longer window decides
                    if (ms < best_ms) {
                        best_ms = ms;
                        plan = x;
                    }
                }
                // stride-1 windows: the halo-reuse kernel (umma_halo.cu) over a few unit shapes, same timing
                int halo_bn = 0, halo_T = 0;
                if (L.conv && L.kind == 0 && L.g.kh * L.g.kw > 1 && !L.x3_cb && !getenv("RTEN_B200_NO_HALO")) {
                    for (int hbn : {64, 128, 256})
                        for (int hT : {1, 2, 4}) {
                            if (hbn > L.N || hT * hbn > 512) continue;
                            auto time_halo = [&](int n) -> double {
                                if (launch_umma_halo_conv(ctx, L, hbn, hT) != RTEN_OK) return -1.0;
                                cudaEventRecord(e0, ctx->stream);
                                bool ok = true;
                                for (int r = 0; r < n && ok; r++) ok = launch_umma_halo_conv(ctx, L, hbn, hT) == RTEN_OK;
                                cudaEventRecord(e1, ctx->stream);
                                if (cudaEventSynchronize(e1) != cudaSuccess || !ok) return -1.0;
                                float t = 0.f;
                                cudaEventElapsedTime(&t, e0, e1);
                                return (double)t / n;
                            };
                            double ms = time_halo(reps);
                            if (ms > 0 && ms < best_ms * 1.05) ms = time_halo(2 * reps);  // a second, longer look at contenders
                            if (verbose && ms > 0) fprintf(stderr, "[autotune] halo bn=%d T=%d -> %.2f us\n", hbn, hT, ms * 1e3);
                            if (ms > 0 && ms < best_ms * 0.97) {  // must win clearly: the generic kernel is the better-trodden path
                                best_ms = ms;
                                halo_bn = hbn;
                                halo_T = hT;
                            }
                        }
                }
                cudaEventDestroy(e0);
                cudaEventDestroy(e1);
                if (halo_bn) {
                    ctx->tune_cache[key] = {-1, halo_bn, halo_T, 0, 0, 0, 0, 0};
                    return launch_umma_halo_conv(ctx, L, halo_bn, halo_T);
                }
                ctx->tune_cache[key] = {plan.bn, plan.pair, plan.katoms, plan.ksplit, plan.splitk, plan.nbuf, plan.acc1, plan.cta2};
            }
        }
    }
    return launch_plan(ctx, L, q, plan, verbose);
}

}  // namespace rtb
