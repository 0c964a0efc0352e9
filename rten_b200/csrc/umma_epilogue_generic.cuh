// Specialised (FAST = 1 / 2) and generic (FAST = 0) epilogues of the tcgen05 GEMM / conv kernel: every zero-point, scale,
// range, split-K and edge case of the operator family; the plain variants (umma_epilogue_plain.cuh) take the common cases.
// Included by umma_kernel.cuh.
#pragma once

namespace rtb {

template <int KIND, int FAST, int CTA2>
__device__ __forceinline__ void epilogue_fast(const EpiCtx& c) {
    const KParams& p = c.p;
    const SmemLayout& L = c.L;
    uint8_t* const stg_base = c.stg_base;
    const int nbuf = c.nbuf;
    uint64_t* const tmem_full = c.tmem_full;
    uint64_t* const tmem_empty = c.tmem_empty;
    uint64_t* const res_bar = c.res_bar;
    int* const sk_flag = c.sk_flag;
    const CUtensorMap* const tma_d = c.tma_d;
    const CUtensorMap* const tma_r = c.tma_r;
    const uint32_t tmem_base = c.tmem_base;
    const int cta_rank = c.cta_rank, worker = c.worker, n_workers = c.n_workers;
    PipeState& st = c.st;
    const int warp = c.warp, lane = c.lane;
    (void)L; (void)sk_flag; (void)tma_r; (void)cta_rank; (void)res_bar;
    // ===================== epilogue (specialised) =====================
    const EpilogueDesc& e = p.epi;
    const int q = warp & 3;
    const int grp = (warp - 4) >> 2;
    const int r = q * 32 + lane;
    const int sw = r & 7;
    uint8_t* stg0 = stg_base + grp * nbuf * STG_BYTES;
    const bool issuer = (q == 0 && lane == 0);
    const bool has_bias = e.bias_kind == 1;
    const bool do_relu = e.act == 1;  // (no activation: NaNs must pass through, fmaxf would drop them)
    uint32_t ci = 0;
    uint32_t& rphase = st.rphase;
    float rg_lo = __int_as_float(0x7f800000), rg_hi = __int_as_float(0xff800000);  // output range (e.range)
    const bool tr = p.trace && blockIdx.x == 0 && warp == 4 && lane == 0;  // (debug trace, RTEN_B200_TRACE_FAST)
    const int it0 = st.it;
    for (int u = worker; u < p.units_total; u += n_workers, st.it++) {
        int t, ks_u;
        p.d_tiles_total.divmod(u, ks_u, t);
        const int acc = p.acc1 ? 0 : (st.it & 1);
        const uint32_t acc_phase = (st.acc >> acc) & 1;
        st.acc ^= 1u << acc;
        // residual of this tile's first chunk: independent of the accumulator -> requested before waiting for it
        // (split-K: only once this CTA knows that it owns the tile's epilogue)
        auto first_residual = [&]() {
            const TileCoord tc0 = decode_tile(p, t, 0, cta_rank);
            const int b0 = ci % nbuf;
            bulk_wait_read(nbuf - 1);
            uint64_t* rb = &res_bar[grp * 4 + b0];
            mbar_expect_tx(rb, p.res_tx_bytes);
            if (p.conv)
                tma_load_4d(stg0 + b0 * STG_BYTES, tma_r, rb, tc0.n0 + grp * 32, tc0.ox0, tc0.oy0, tc0.b0);
            else
                tma_load_4d(stg0 + b0 * STG_BYTES, tma_r, rb, tc0.n0 + grp * 32, tc0.m0, tc0.z0, tc0.z1);
        };
        if (p.res_tma && p.splitk == 1 && issuer && grp * 32 < p.bn) first_residual();
        mbar_wait(&tmem_full[acc], acc_phase);
        if (tr && st.it - it0 < 2048) p.trace[4096 + st.it - it0] = clock64();
        tc_fence_after();
        bool owner = true;
        if (p.splitk > 1) {
            owner = splitk_publish(p, CTA2 ? 2 * t + cta_rank : t, ks_u, grp, q, lane,
                                   tmem_base + ((uint32_t)(q * 32) << 16) + acc * ACC_STRIDE, &sk_flag[grp]);
            if (owner && p.res_tma && issuer && grp * 32 < p.bn) first_residual();
        }
        for (int sub = 0; owner && sub <= p.pair; sub++) {
            const TileCoord tc = decode_tile(p, t, sub, cta_rank);
            const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + acc * ACC_STRIDE + sub * p.bn;
            // integer zero-point terms of this thread's row:  C = acc - za*colsum[n] - zb[n]*(rowsum - K*za)
            unsigned za_v = 0, t_m = 0;
            bool row_ok = true;
            if ((KIND == 1 && (e.za || e.za8 || e.zb)) || e.range) {
                int m_idx;
                if (p.conv) {
                    int xi, r2, yi, bi;
                    p.d_tw.divmod(r, r2, xi);
                    p.d_th.divmod(r2, bi, yi);
                    const int ox = tc.ox0 + xi, oy = tc.oy0 + yi, b = tc.b0 + bi;
                    row_ok = (bi < p.tb) && (ox < p.OW) && (oy < p.OH) && (b < p.Bn);
                    m_idx = (b * p.OH + oy) * p.OW + ox;
                } else {
                    m_idx = tc.m0 + r;
                    row_ok = m_idx < p.M;
                }
                if (row_ok) {
                    if (e.za) za_v = (unsigned)e.za[m_idx % e.za_len];
                    else if (e.za8) za_v = (unsigned)(e.za8_signed ? (int)(int8_t)__ldg(e.za8) : (int)__ldg(e.za8));
                    if (e.zb) t_m = (unsigned)e.rowsum[m_idx] - (unsigned)p.K * za_v;
                }
            }
            for (int c0 = grp * 32; c0 < p.bn; c0 += 64) {
                uint32_t v[32];
                if (p.splitk > 1)
                    splitk_sum<KIND>(p, CTA2 ? 2 * t + cta_rank : t, sub, c0, r, v);
                else
                    tmem_ld_32x32(t_row + c0, v);
                const int nbase = tc.n0 + c0;
                const int bcur = ci % nbuf;
                uint8_t* stg = stg0 + bcur * STG_BYTES;
                uint8_t* rowp = stg + r * 128;
                if (p.res_tma && issuer) {  // prefetch the next chunk's residual of this tile into the next ring slot
                    int nsub = sub, nc0 = c0 + 64;
                    if (nc0 >= p.bn) {
                        nsub = sub + 1;
                        nc0 = grp * 32;
                    }
                    if (nsub <= p.pair && nc0 < p.bn) {
                        const TileCoord tn = decode_tile(p, t, nsub, cta_rank);
                        const int bnext = (ci + 1) % nbuf;
                        bulk_wait_read(nbuf - 2);
                        uint64_t* rb = &res_bar[grp * 4 + bnext];
                        mbar_expect_tx(rb, p.res_tx_bytes);
                        if (p.conv)
                            tma_load_4d(stg0 + bnext * STG_BYTES, tma_r, rb, tn.n0 + nc0, tn.ox0, tn.oy0, tn.b0);
                        else
                            tma_load_4d(stg0 + bnext * STG_BYTES, tma_r, rb, tn.n0 + nc0, tn.m0, tn.z0, tn.z1);
                    }
                }
                tmem_ld_wait();
                if (p.ksplit) {
#pragma unroll
                    for (int h = 0; h < 2; h++) {
                        uint32_t w[16];
                        tmem_ld_32x16(t_row + p.bn + c0 + h * 16, w);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 16; j++) {
                            if (KIND == 0)
                                v[h * 16 + j] = __float_as_uint(__fadd_rn(__uint_as_float(v[h * 16 + j]), __uint_as_float(w[j])));
                            else
                                v[h * 16 + j] += w[j];
                        }
                    }
                }
                if (p.res_tma) {
                    mbar_wait(&res_bar[grp * 4 + bcur], (rphase >> bcur) & 1);
                    rphase ^= 1u << bcur;
                }
                // a tile may overhang N (N % bn != 0): its last 32-column chunks are then entirely out of range -- the
                // TMA store clips them, and neither the column vectors (bias, sums, scales) nor the range may touch them
                const bool col_ok = nbase < p.N;
                if (!col_ok) {
                } else
                if (KIND == 0) {
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        float4 rr = make_float4(0.f, 0.f, 0.f, 0.f), bb = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (p.res_tma) rr = *reinterpret_cast<const float4*>(rowp + (((j >> 2) ^ sw) << 4));
                        if (has_bias) bb = __ldg(reinterpret_cast<const float4*>(e.bias + nbase + j));
                        const float r4[4] = {rr.x, rr.y, rr.z, rr.w}, b4[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
                        for (int u = 0; u < 4; u++) {
                            float x = __uint_as_float(v[j + u]) * e.alpha;
                            x = fmaf(e.r_scale, r4[u], x);
                            x = x + b4[u];
                            v[j + u] = __float_as_uint(do_relu ? fmaxf(x, 0.0f) : x);
                        }
                        if (FAST == 2 && e.act > 1) {  // (own instantiation: a possible call changes the whole loop's code)
                            const float4 t = act4(make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                                              __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3])), e.act);
                            v[j] = __float_as_uint(t.x);
                            v[j + 1] = __float_as_uint(t.y);
                            v[j + 2] = __float_as_uint(t.z);
                            v[j + 3] = __float_as_uint(t.w);
                        }
                    }
                } else if (e.za || e.za8 || e.zb || e.scale) {
                    // exact i32 arithmetic with wrap-around (unsigned ops), column vectors fetched 128 bits at a time
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        uint4 cs = make_uint4(0u, 0u, 0u, 0u), zb4 = make_uint4(0u, 0u, 0u, 0u);
                        float4 sc = make_float4(1.f, 1.f, 1.f, 1.f);
                        if (e.za || e.za8) cs = __ldg(reinterpret_cast<const uint4*>(e.colsum + nbase + j));
                        if (e.zb) {
                            if (e.zb_len == 1) {
                                const unsigned z = (unsigned)__ldg(e.zb);
                                zb4 = make_uint4(z, z, z, z);
                            } else {
                                zb4 = __ldg(reinterpret_cast<const uint4*>(e.zb + nbase + j));
                            }
                        }
                        if (e.scale) {
                            if (e.scale_len == 1) {
                                const float z = __ldg(e.scale);
                                sc = make_float4(z, z, z, z);
                            } else {
                                sc = __ldg(reinterpret_cast<const float4*>(e.scale + nbase + j));
                            }
                            if (e.scale2) {
                                const float s2 = __ldg(e.scale2);
                                sc = make_float4(__fmul_rn(s2, sc.x), __fmul_rn(s2, sc.y), __fmul_rn(s2, sc.z), __fmul_rn(s2, sc.w));
                            }
                        }
                        float4 rr = make_float4(0.f, 0.f, 0.f, 0.f), bb = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (p.res_tma) rr = *reinterpret_cast<const float4*>(rowp + (((j >> 2) ^ sw) << 4));
                        if (has_bias) bb = __ldg(reinterpret_cast<const float4*>(e.bias + nbase + j));
                        const unsigned c4[4] = {cs.x, cs.y, cs.z, cs.w}, z4[4] = {zb4.x, zb4.y, zb4.z, zb4.w};
                        const float s4[4] = {sc.x, sc.y, sc.z, sc.w}, r4[4] = {rr.x, rr.y, rr.z, rr.w},
                                    b4[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
                        for (int u = 0; u < 4; u++) {
                            const unsigned c = v[j + u] - za_v * c4[u] - z4[u] * t_m;
                            if (e.scale) {
                                // ConvIntegerToFloat / MatMulIntegerToFloat, then the graph's Add(bias), Add(residual),
                                // Relu as separate exactly-rounded f32 operations (no contraction)
                                float x = __fmul_rn(__int2float_rn((int)c), s4[u]);
                                if (has_bias) x = __fadd_rn(x, b4[u]);
                                if (p.res_tma) x = __fadd_rn(x, r4[u]);
                                v[j + u] = __float_as_uint(do_relu ? fmaxf(x, 0.0f) : x);
                            } else {
                                v[j + u] = c;
                            }
                        }
                        if (FAST == 2 && e.scale && e.act > 1) {
                            const float4 t = act4(make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                                              __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3])), e.act);
                            v[j] = __float_as_uint(t.x);
                            v[j + 1] = __float_as_uint(t.y);
                            v[j + 2] = __float_as_uint(t.z);
                            v[j + 3] = __float_as_uint(t.w);
                        }
                    }
                }
                if (e.range && row_ok && col_ok) {
#pragma unroll
                    for (int j = 0; j < 32; j++) {
                        rg_lo = fminf(rg_lo, __uint_as_float(v[j]));
                        rg_hi = fmaxf(rg_hi, __uint_as_float(v[j]));
                    }
                }
                if (nbuf == 1) {  // single staging buffer: the previous store must have been read before it is rewritten
                    if (issuer) bulk_wait_read(0);
                    asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
                }
#pragma unroll
                for (int j = 0; j < 8; j++)
                    *reinterpret_cast<uint4*>(rowp + ((j ^ sw) << 4)) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
                if (issuer && !p.res_tma && nbuf > 1) bulk_wait_read(nbuf - 2);
                fence_proxy_async();
                asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
                if (issuer) {
                    if (p.conv)
                        tma_store_4d(tma_d, stg, nbase, tc.ox0, tc.oy0, tc.b0);
                    else
                        tma_store_4d(tma_d, stg, nbase, tc.m0, tc.z0, tc.z1);
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
                ci++;
            }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
            if (CTA2)
                mbar_arrive_cluster(smem_u32(&tmem_empty[acc]) & PEER_BIT_MASK);  // the leader's MMA warp waits on it
            else
                mbar_arrive(&tmem_empty[acc]);
        }
        if (tr && st.it - it0 < 2048) p.trace[6144 + st.it - it0] = clock64();
    }
    if (e.range) range_commit(e.range, rg_lo, rg_hi);
    // shared memory must stay valid until the last bulk store has READ it; the global writes complete on their own
    // before the grid is considered finished
    if (issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

template <int KIND, int CTA2>
__device__ __forceinline__ void epilogue_generic(const EpiCtx& c) {
    constexpr int FAST = 0;
    (void)FAST;
    const KParams& p = c.p;
    const SmemLayout& L = c.L;
    uint8_t* const stg_base = c.stg_base;
    const int nbuf = c.nbuf;
    uint64_t* const tmem_full = c.tmem_full;
    uint64_t* const tmem_empty = c.tmem_empty;
    uint64_t* const res_bar = c.res_bar;
    int* const sk_flag = c.sk_flag;
    const CUtensorMap* const tma_d = c.tma_d;
    const CUtensorMap* const tma_r = c.tma_r;
    const uint32_t tmem_base = c.tmem_base;
    const int cta_rank = c.cta_rank, worker = c.worker, n_workers = c.n_workers;
    PipeState& st = c.st;
    const int warp = c.warp, lane = c.lane;
    (void)L; (void)sk_flag; (void)tma_r; (void)cta_rank; (void)res_bar;
    // ===================== epilogue (generic) =====================
    const EpilogueDesc& e = p.epi;
    const int q = warp & 3;          // TMEM lane quadrant this warp may access
    const int grp = (warp - 4) >> 2;  // epilogue group: chunks grp, grp+2, ...
    const int r = q * 32 + lane;
    uint8_t* stg0 = stg_base + grp * nbuf * STG_BYTES;
    const bool issuer = (q == 0 && lane == 0);
    uint32_t ci = 0;            // chunks processed by this group so far (selects the staging buffer)
    uint32_t& rphase = st.rphase;  // bit b = phase of res_bar[grp][b]
    float rg_lo = __int_as_float(0x7f800000), rg_hi = __int_as_float(0xff800000);  // output range (e.range)
    const int it0 = st.it;
    for (int u = worker; u < p.units_total; u += n_workers, st.it++) {
        const int it = st.it - it0;
        int t, ks_u;
        p.d_tiles_total.divmod(u, ks_u, t);
        const int acc = p.acc1 ? 0 : (st.it & 1);
        const uint32_t acc_phase = (st.acc >> acc) & 1;
        st.acc ^= 1u << acc;
        auto first_residual = [&]() {
            // residual of this tile's first chunk: independent of the accumulator -> request it before waiting
            const TileCoord tc0 = decode_tile(p, t, 0, cta_rank);
            const int b0 = ci % nbuf;
            bulk_wait_read(nbuf - 1);  // the store that last used buffer b0 (chunk ci - nbuf) has been read
            uint64_t* rb = &res_bar[grp * 4 + b0];
            mbar_expect_tx(rb, p.res_tx_bytes);
            if (p.conv)
                tma_load_4d(stg0 + b0 * STG_BYTES, tma_r, rb, tc0.n0 + grp * 32, tc0.ox0, tc0.oy0, tc0.b0);
            else
                tma_load_4d(stg0 + b0 * STG_BYTES, tma_r, rb, tc0.n0 + grp * 32, tc0.m0, tc0.z0, tc0.z1);
        };
        if (p.res_tma && p.splitk == 1 && issuer && grp * 32 < p.bn) first_residual();
        mbar_wait(&tmem_full[acc], acc_phase);
        if (p.trace && blockIdx.x == 0 && warp == 4 && lane == 0 && it < 2048) p.trace[4096 + it] = clock64();
        tc_fence_after();
        bool owner = true;
        if (p.splitk > 1) {
            owner = splitk_publish(p, CTA2 ? 2 * t + cta_rank : t, ks_u, grp, q, lane,
                                   tmem_base + ((uint32_t)(q * 32) << 16) + acc * ACC_STRIDE, &sk_flag[grp]);
            if (owner && p.res_tma && issuer && grp * 32 < p.bn) first_residual();
        }
        for (int sub = 0; owner && sub <= p.pair; sub++) {
        const TileCoord tc = decode_tile(p, t, sub, cta_rank);
        // ---- row bookkeeping
        bool row_ok;
        long long d_off, r_off;
        int m_idx;
        if (p.conv) {
            int xi, r2, yi, bi;
            p.d_tw.divmod(r, r2, xi);
            p.d_th.divmod(r2, bi, yi);
            const int ox = tc.ox0 + xi, oy = tc.oy0 + yi, b = tc.b0 + bi;
            row_ok = (bi < p.tb) && (ox < p.OW) && (oy < p.OH) && (b < p.Bn);
            d_off = (long long)b * e.s_z0 + (long long)oy * e.s_row + (long long)ox * e.s_z1;
            r_off = (long long)b * e.r_z0 + (long long)oy * e.r_row + (long long)ox * e.r_z1;
            m_idx = (b * p.OH + oy) * p.OW + ox;
        } else {
            const int m = tc.m0 + r;
            row_ok = m < p.M;
            d_off = (long long)tc.z0 * e.s_z0 + (long long)tc.z1 * e.s_z1 + (long long)m * e.s_row;
            r_off = (long long)tc.z0 * e.r_z0 + (long long)tc.z1 * e.r_z1 + (long long)m * e.r_row;
            m_idx = m;
        }
        float row_bias = 0.0f;
        int za_v = 0, rs_v = 0;
        if (row_ok) {
            if (KIND == 0) {
                if (e.bias_kind == 2) row_bias = e.bias[m_idx];
            } else {
                if (e.za) za_v = e.za[m_idx % e.za_len];
                else if (e.za8) za_v = e.za8_signed ? (int)(int8_t)__ldg(e.za8) : (int)__ldg(e.za8);
                if (e.zb) rs_v = e.rowsum[m_idx];
            }
        }
        const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + acc * ACC_STRIDE + sub * p.bn;
        for (int c0 = grp * 32; c0 < p.bn; c0 += 64) {
            const bool tr = p.trace && blockIdx.x == 0 && warp == 4 && lane == 0;
            long long t0 = tr ? clock64() : 0;
            uint32_t v[32];
            const int ncols = (p.bn - c0) >= 32 ? 32 : 16;
            if (p.splitk > 1) {
                splitk_sum<KIND>(p, CTA2 ? 2 * t + cta_rank : t, sub, c0, r, v);
            } else if (ncols == 32) {
                tmem_ld_32x32(t_row + c0, v);
            } else {
                uint32_t w[16];
                tmem_ld_32x16(t_row + c0, w);
#pragma unroll
                for (int j = 0; j < 16; j++) v[j] = w[j];
#pragma unroll
                for (int j = 16; j < 32; j++) v[j] = 0;
            }
            tmem_ld_wait();
            if (tr) { const long long t1 = clock64(); p.trace[6144 + 1024 + 0] += t1 - t0; t0 = t1; }
            if (p.ksplit) {
                // add the second partial accumulator (columns + bn), 16 columns at a time to bound registers
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    if (h * 16 < ncols) {
                        uint32_t w[16];
                        tmem_ld_32x16(t_row + p.bn + c0 + h * 16, w);
                        tmem_ld_wait();
#pragma unroll
                        for (int j = 0; j < 16; j++) {
                            if (KIND == 0)
                                v[h * 16 + j] = __float_as_uint(__fadd_rn(__uint_as_float(v[h * 16 + j]), __uint_as_float(w[j])));
                            else
                                v[h * 16 + j] += w[j];
                        }
                    }
                }
            }
            const int nbase = tc.n0 + c0;
            const int bcur = ci % nbuf;
            uint8_t* stg = stg0 + bcur * STG_BYTES;
            uint8_t* rowp = stg + r * 128;
            const int sw = r & 7;
            if (p.res_tma) {
                // request the next chunk's residual of this tile (other buffer) once the store that last used that
                // buffer has been read, then wait for this chunk's residual to land
                if (issuer) {
                    int nsub = sub, nc0 = c0 + 64;
                    if (nc0 >= p.bn) {
                        nsub = sub + 1;
                        nc0 = grp * 32;
                    }
                    if (nsub <= p.pair && nc0 < p.bn) {
                        const TileCoord tn = decode_tile(p, t, nsub, cta_rank);
                        const int bnext = (ci + 1) % nbuf;
                        bulk_wait_read(nbuf - 2);  // chunk ci + 1 - nbuf's store has been read; newer ones stay in flight
                        uint64_t* rb = &res_bar[grp * 4 + bnext];
                        mbar_expect_tx(rb, p.res_tx_bytes);
                        uint8_t* dst = stg0 + bnext * STG_BYTES;
                        if (p.conv)
                            tma_load_4d(dst, tma_r, rb, tn.n0 + nc0, tn.ox0, tn.oy0, tn.b0);
                        else
                            tma_load_4d(dst, tma_r, rb, tn.n0 + nc0, tn.m0, tn.z0, tn.z1);
                    }
                }
                mbar_wait(&res_bar[grp * 4 + bcur], (rphase >> bcur) & 1);
                rphase ^= 1u << bcur;
            }
            // ---- fast path (registers, fully unrolled): f32, act in {none, relu}, residual / bias absent or
            //      128-bit loadable.  Everything else (gelu, strided residual, N tails, the integer zero-point
            //      math) runs as a ROLLED loop over the staged row: keeps the unrolled code small enough for
            //      the instruction cache.
            const bool full = nbase + 32 <= p.N;
            bool fast = (KIND == 0) ? (e.act <= 1 && full) : !(e.za || e.za8 || e.zb || e.scale);  // raw i32: nothing to do
            if (fast && e.r && !p.res_tma)
                fast = e.r_col == 1 && ((reinterpret_cast<uintptr_t>(e.r + r_off + nbase) & 15) == 0);
            if (fast && e.bias_kind == 1) fast = (reinterpret_cast<uintptr_t>(e.bias + nbase) & 15) == 0;
            fast = __all_sync(0xffffffffu, fast || !row_ok) || p.res_tma;  // (res_tma launches are fast-path only)
            if (KIND == 0 && fast && row_ok) {
                const bool do_relu = e.act == 1;  // (no activation: NaNs must pass through, fmaxf would drop them)
#pragma unroll
                for (int j = 0; j < 32; j += 4) {
                    float4 rr = make_float4(0.f, 0.f, 0.f, 0.f), bb = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (p.res_tma)
                        rr = *reinterpret_cast<const float4*>(rowp + (((j >> 2) ^ sw) << 4));
                    else if (e.r)
                        rr = __ldcg(reinterpret_cast<const float4*>(e.r + r_off + nbase + j));
                    if (e.bias_kind == 1) bb = __ldg(reinterpret_cast<const float4*>(e.bias + nbase + j));
                    const float r4[4] = {rr.x, rr.y, rr.z, rr.w}, b4[4] = {bb.x, bb.y, bb.z, bb.w};
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        float x = __uint_as_float(v[j + u]) * e.alpha;
                        x = fmaf(e.r_scale, r4[u], x);
                        x = x + b4[u] + row_bias;
                        v[j + u] = __float_as_uint(do_relu ? fmaxf(x, 0.0f) : x);
                    }
                }
            }
            if (tr) { const long long t1 = clock64(); p.trace[6144 + 1024 + 1] += t1 - t0; t0 = t1; }
            // ---- stage the row chunk in shared memory (128 B per row, 16-byte chunks XOR-swizzled by r & 7)
            // Buffer reuse: (no residual) the issuer waited, before the previous chunk's barrier, until the store of
            // chunk ci - nbuf had been read; (res_tma) the residual mbarrier of this buffer orders it.
            if (p.tma_store && nbuf == 1) {
                if (issuer) bulk_wait_read(0);
                asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
            }
#pragma unroll
            for (int j = 0; j < 8; j++)
                *reinterpret_cast<uint4*>(rowp + ((j ^ sw) << 4)) = make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
            if (!fast && row_ok) {
                // rolled slow path on this thread's own staged row
#pragma unroll 1
                for (int j = 0; j < ncols; j++) {
                    const int n = nbase + j;
                    if (n >= p.N) break;
                    uint32_t* sp = reinterpret_cast<uint32_t*>(rowp + (((j >> 2) ^ sw) << 4)) + (j & 3);
                    if (KIND == 0) {
                        float x = __uint_as_float(*sp) * e.alpha;
                        if (e.r) x = fmaf(e.r_scale, __ldcg(e.r + r_off + (long long)n * e.r_col), x);
                        if (e.bias_kind == 1) x += e.bias[n];
                        x += row_bias;
                        *sp = __float_as_uint(apply_act(x, e.act));
                    } else {
                        // exact i32 arithmetic with wrap-around (unsigned ops)
                        unsigned c = *sp;
                        if (e.za || e.za8) c -= (unsigned)za_v * (unsigned)e.colsum[n];
                        if (e.zb) {
                            const unsigned zbv = (unsigned)e.zb[n % e.zb_len];
                            c -= zbv * (unsigned)rs_v;
                            if (e.za || e.za8) c += (unsigned)p.K * (unsigned)za_v * zbv;
                        }
                        if (e.scale) {
                            float sv = e.scale[n % e.scale_len];
                            if (e.scale2) sv = __fmul_rn(__ldg(e.scale2), sv);
                            float x = __fmul_rn(__int2float_rn((int)c), sv);
                            if (e.bias_kind == 1) x = __fadd_rn(x, e.bias[n]);
                            if (e.r) x = __fadd_rn(x, __ldcg(e.r + r_off + (long long)n * e.r_col));
                            *sp = __float_as_uint(apply_act(x, e.act));
                        } else {
                            *sp = c;
                        }
                    }
                }
            }
            if (e.range && row_ok) {  // (rolled: the generic epilogue trades speed for size)
#pragma unroll 1
                for (int j = 0; j < ncols; j++) {
                    if (nbase + j >= p.N) break;
                    const float xv = *(reinterpret_cast<const float*>(rowp + (((j >> 2) ^ sw) << 4)) + (j & 3));
                    rg_lo = fminf(rg_lo, xv);
                    rg_hi = fmaxf(rg_hi, xv);
                }
            }
            if (tr) { const long long t1 = clock64(); p.trace[6144 + 1024 + 2] += t1 - t0; t0 = t1; }
            if (p.tma_store) {
                // leave nbuf-1 stores in flight minus the one about to be issued: frees the buffer of chunk ci+1
                if (issuer && !p.res_tma && nbuf > 1) bulk_wait_read(nbuf - 2);
                if (tr) { const long long t1 = clock64(); p.trace[6144 + 1024 + 3] += t1 - t0; t0 = t1; }
                fence_proxy_async();
                if (tr) { const long long t1 = clock64(); p.trace[6144 + 1024 + 4] += t1 - t0; t0 = t1; }
                asm volatile("bar.sync %0, 128;" ::"r"(1 + grp) : "memory");
                if (tr) { const long long t1 = clock64(); p.trace[6144 + 1024 + 5] += t1 - t0; t0 = t1; p.trace[6144 + 1024 + 7] += 1; }
                if (issuer) {
                    if (p.conv)
                        tma_store_4d(tma_d, stg, nbase, tc.ox0, tc.oy0, tc.b0);
                    else
                        tma_store_4d(tma_d, stg, nbase, tc.m0, tc.z0, tc.z1);
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
                if (tr) { const long long t1 = clock64(); p.trace[6144 + 1024 + 6] += t1 - t0; t0 = t1; }
                ci++;
            } else if (row_ok) {
                // direct stores from the staged row (any output strides); consecutive lanes = consecutive rows
                uint32_t* dptr = reinterpret_cast<uint32_t*>(e.d) + d_off;
#pragma unroll 1
                for (int j = 0; j < ncols; j++) {
                    const int n = nbase + j;
                    if (n >= p.N) break;
                    dptr[(long long)n * e.s_col] = *(reinterpret_cast<const uint32_t*>(rowp + (((j >> 2) ^ sw) << 4)) + (j & 3));
                }
            }
            __syncwarp();
        }
        }  // sub
        tc_fence_before();
        __syncwarp();
        if (p.trace && blockIdx.x == 0 && warp == 4 && lane == 0 && it < 2048) p.trace[6144 + it] = clock64();
        if (lane == 0) {
            if (CTA2)
                mbar_arrive_cluster(smem_u32(&tmem_empty[acc]) & PEER_BIT_MASK);  // the leader's MMA warp waits on it
            else
                mbar_arrive(&tmem_empty[acc]);
        }
    }
    // smem must stay valid until the last bulk store has read it
    if (e.range) range_commit(e.range, rg_lo, rg_hi);
    if (p.tma_store && issuer) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

}  // namespace rtb
