// affine_tma.cu — TMA-staged, warp-specialised 3-D rigid/affine registration epoch (sm_100a).
//
// Same contract as affine_moments_kernel<3,*> in affine.cu (reference call sites listed there),
// re-organised around what bounds it on B200: 8 B/voxel of HBM traffic against ~60 fp32
// pipe operations per voxel.  Design:
//   * persistent CTAs (one per SM) of 16 warps; there is no dedicated producer warp: the LAST warp
//     to finish a tile (shared-memory arrival counter) computes and issues the TMA loads that
//     refill that stage, so no warp ever waits for a slot to drain;
//   * work unit = a z-run of ZC output tiles of 32x16x8 voxels; lane <-> x, warp <-> y, so a
//     thread keeps its x and y base coordinates for the whole unit and steps along z;
//   * the producer maps each output tile through theta, takes the bounding box of its source
//     footprint and, if it fits the fixed TMA box (BX x BY x BZ incl. halo), fetches that box of the
//     moving volume and the target tile with two cp.async.bulk.tensor loads into a 4-stage smem
//     ring (mbarrier "full" per stage).  TMA's out-of-bounds zero fill IS grid_sample's zeros padding.
//     Tiles whose footprint does not fit (large rotations) are gathered from global memory with
//     explicit bounds checks instead — same arithmetic, slower, always correct;
//   * consumers process two voxels (z, z+1) per thread with packed f32x2 arithmetic
//     (FFMA2/FADD2): half the issue slots for the same fp32 pipe work; floor() is a round-down
//     add of 1.5*2^23 (FADD.RM) instead of FRND/F2I (those run at 16 lanes/clk/SM on the XU pipe,
//     profiles/r01_microbench_issue_rates.txt); the smem index is formed in fp32 and extracted
//     from the mantissa, so the only integer work per voxel is one subtract and one LEA;
//   * moments are kept per thread over a unit (x,y constant -> only the z-weighted sums need a
//     per-voxel FMA), folded with x,y once per unit, reduced per CTA, and finished by the last
//     CTA exactly like the non-TMA kernel (same epilogue code).
#define TRB_TIMING_OWNER 1
#include "affine_tile.cuh"

namespace trb {


constexpr int kRedLd = TRB_MOMENTS + 3;

// ---- grid-level reduction of the per-CTA partial sums -------------------------------------------------
// Every CTA owns slot blockIdx.x of every pair (zeros for pairs it never touches).  CTAs are grouped by 16;
// the CTA that completes a (pair, group) ticket adds the group's 16 slots in index order into the group
// slot — this happens DURING the launch, off the critical path.  The last CTA to finish all its tiles then
// only has ceil(G/16) group slots per pair to add (fixed order) before the epilogue, so the serial tail of
// a launch is a few microseconds however many SMs contributed.  All orders are fixed => bit-reproducible.
constexpr int kGroup = 16;
constexpr int kTicketsPerPair = 128;          // [0..63] group tickets; [126] CTAs-done (pair 0); [127] direct kernel

__device__ __forceinline__ double *slot_ptr(const TmaParams &p, int pair, int slot)
{
    return p.a.partials + ((size_t)pair * kMaxSlots + slot) * TRB_MOMENTS;
}

// add slots [s0, s1) of `pair` in index order; lane l returns moments l (x) and l+32 (y, valid for l < 9)
__device__ __forceinline__ double2 warp_fold_slots(const TmaParams &p, int pair, int s0, int s1, int lane)
{
    const int v1 = min(lane + 32, TRB_MOMENTS - 1);
    double r0 = 0.0, r1 = 0.0;
    for (int b0 = s0; b0 < s1; b0 += kGroup) {
        // issue all 32 loads of the pass before touching any result: written as `acc += __ldcg(...)` the
        // compiler emitted load-pair / add / load-pair / add with two registers, i.e. one L2 round trip per
        // slot (tools/_lat microbenchmark: 6.4k cycles for 16 slots)
        double x0[kGroup], x1[kGroup];
#pragma unroll
        for (int j = 0; j < kGroup; ++j) {
            const double *row = slot_ptr(p, pair, (b0 + j < s1) ? b0 + j : s0);
            asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(x0[j]) : "l"(row + lane));
            asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(x1[j]) : "l"(row + v1));
        }
#pragma unroll
        for (int j = 0; j < kGroup; ++j) {              // index order
            const bool ok = b0 + j < s1;
            r0 += ok ? x0[j] : 0.0;
            r1 += ok ? x1[j] : 0.0;
        }
    }
    return make_double2(r0, r1);
}

// one warp: CTA blockIdx.x has deposited its slot of `pair`; arrive on the group ticket, fold if last
__device__ void warp_arrive_group(const TmaParams &p, int pair, int G, int lane)
{
    __threadfence();
    __syncwarp();
    const int g = blockIdx.x / kGroup;
    const int gsize = min(kGroup, G - g * kGroup);
    unsigned *tk = p.a.tickets + (size_t)pair * kTicketsPerPair + g;
    unsigned t = 0;
    if (lane == 0) t = atomicAdd(tk, 1u);
    t = __shfl_sync(kFull, t, 0);
    if (t != (unsigned)gsize - 1u) return;
    __threadfence();
    const double2 r = warp_fold_slots(p, pair, g * kGroup, g * kGroup + gsize, lane);
    double *dst = slot_ptr(p, pair, G + g);
    __stcg(dst + lane, r.x);
    if (lane + 32 < TRB_MOMENTS) __stcg(dst + lane + 32, r.y);
    if (lane == 0) *tk = 0u;
    __threadfence();
}

// Warp-level hand-over of a pair's sums (no CTA barrier: warps never wait for each other).  Each warp
// deposits its 41 totals in red[warp]; the LAST warp of the CTA to arrive adds the 16 rows in fixed
// order, writes the CTA partial (fp64) to its slot and arrives on the group ticket.
__device__ void warp_publish_pair(const float (&acc)[TRB_MOMENTS], float *red /*[16][kRedLd]*/, unsigned *cnt,
                                  const TmaParams &p, int pair, int G, int warp, int lane)
{
    warp_reduce_moments(acc, red + warp * kRedLd, lane);
    __syncwarp();
    unsigned old = 0;
    if (lane == 0)
        asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(smem_u32(cnt)) : "memory");
    old = __shfl_sync(kFull, old, 0);
    if (old != kConsumerWarps - 1) return;
    // lane 0's acq_rel atomic synchronises with the other warps' (release) arrivals; __syncwarp extends that
    // ordering to the remaining lanes before they read the 16 rows.  (compute-sanitizer racecheck flags these
    // reads because it only models barriers, not atomics-based hand-over.)
    __syncwarp();
    if (lane == 0) *cnt = 0u;
    double *mine = slot_ptr(p, pair, blockIdx.x);
    for (int v = lane; v < TRB_MOMENTS; v += 32) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < kConsumerWarps; ++w) s += (double)red[w * kRedLd + v];
        __stcg(mine + v, s);
    }
    // the group arrival (fence + global ticket + possibly a 16-slot fold: 2-5 us of round trips) is NOT done here: the
    // warp that does it would finish its next tile late, and a stage is only refilled when the slowest warp is through —
    // measured as a 4-5 us bubble of the TMA ring after every pair switch.  The kernel arrives for all its pairs after
    // the main loop.
}

// Run by the LAST CTA to complete its tiles (all 16 warps): per pair, add the group slots in index order
// and run the epilogue (FUSED) or publish the moments.  Pairs are spread over the warps.
template <bool FUSED>
__device__ void final_phase(const TmaParams &p, double *fin_s /*[16][TRB_MOMENTS + 1] smem*/, int G, int warp, int lane)
{
    constexpr int LD = TRB_MOMENTS + 1;
    if (p.use_groups) {
        const int n_groups = (G + kGroup - 1) / kGroup;
        for (int pair = warp; pair < p.n_pairs; pair += kConsumerWarps) {
            const double2 r = warp_fold_slots(p, pair, G, G + n_groups, lane);
            double *row = fin_s + warp * LD;
            row[lane] = r.x;
            if (lane + 32 < TRB_MOMENTS) row[lane + 32] = r.y;
            __syncwarp();
            if (FUSED) {
                if (lane == 0) affine_epilogue<3>(row, p.a, pair);
            } else {
                for (int v = lane; v < TRB_MOMENTS; v += 32) p.a.moments_out[(size_t)pair * TRB_MOMENTS + v] = row[v];
            }
            __syncwarp();
        }
        return;
    }
    // one or two pairs: no group stage — every warp folds a contiguous range of one pair's G slots
    // (one round trip), the ranges are combined in index order, one warp per pair runs the epilogue
    const int np = p.n_pairs;
    const int wpp = kConsumerWarps / np;                     // warps per pair
    const int pl = warp / wpp, part = warp - pl * wpp;
    if (pl < np) {
        const double2 r = warp_fold_slots(p, pl, G * part / wpp, G * (part + 1) / wpp, lane);
        fin_s[warp * LD + lane] = r.x;
        if (lane + 32 < TRB_MOMENTS) fin_s[warp * LD + lane + 32] = r.y;
    }
    __syncthreads();
    if (warp < np) {
        double *row = fin_s + (warp * wpp) * LD;
        for (int v = lane; v < TRB_MOMENTS; v += 32) {
            double t = row[v];
            for (int q = 1; q < wpp; ++q) t += row[q * LD + v];
            row[v] = t;
        }
        __syncwarp();
        if (FUSED) {
            if (p.a.peer.world > 1) peer_allreduce(row, TRB_MOMENTS, p.a.peer, lane);
            if (lane == 0) affine_epilogue<3>(row, p.a, warp);
        } else {
            for (int v = lane; v < TRB_MOMENTS; v += 32) p.a.moments_out[(size_t)warp * TRB_MOMENTS + v] = row[v];
        }
    }
}

template <int BX, int BY, int BZ, int NSTAGE, bool FUSED, bool MSE_ONLY>
__global__ void __launch_bounds__(kTmaThreads, 1)
affine3d_tma_kernel(const TmaParams p, const __grid_constant__ CUtensorMap map_mov, const __grid_constant__ CUtensorMap map_tgt)
{
    using L = SmemLayout<BX, BY, BZ>;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem_raw + (size_t)NSTAGE * L::kStageBytes);
    unsigned *done_cnt = reinterpret_cast<unsigned *>(full_bar + NSTAGE);
    TileMeta *meta = reinterpret_cast<TileMeta *>(done_cnt + NSTAGE);
    __shared__ __align__(16) float red[2][kConsumerWarps * kRedLd];     // double-buffered by the parity of the flush count;
                                                                         // re-used (as doubles) by final_phase
    __shared__ unsigned pair_cnt[2];
    __shared__ float coef_s[kMaxCachedPairs * 12];

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int W = p.a.W, H = p.a.H, D = p.a.D;
    const int G = gridDim.x, b = blockIdx.x;
    const float inv_d2 = 2.f / (float)D, zoff = 1.f / (float)D - 1.f;      // zv(z) = (2z+1)/D - 1

    // Programmatic dependent launch: let the next epoch's grid be scheduled as SMs drain (its CTAs get as far
    // as this point — smem carve-up, barrier init — while our stragglers and final phase finish), and do not
    // read theta / touch the workspace until the previous epoch's grid has completed and flushed.
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (threadIdx.x == 0) {
        pair_cnt[0] = pair_cnt[1] = 0u;
        for (int i = 0; i < NSTAGE; ++i) { mbar_init(full_bar + i, 1); done_cnt[i] = 0u; }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");

    // coordinate maps of all pairs -> smem (theta was written by the previous epoch's epilogue)
    if (p.n_pairs <= kMaxCachedPairs) {
        for (int pr = threadIdx.x; pr < p.n_pairs; pr += kTmaThreads) {
            const float *st = p.a.state + (size_t)pr * TRB_STATE_FLOATS + TRB_STATE_THETA;
            float th[12];
#pragma unroll
            for (int i = 0; i < 12; ++i) th[i] = __ldcg(st + i);
            const Coef k = make_coef(th, D, H, W);
#pragma unroll
            for (int r = 0; r < 3; ++r) {
#pragma unroll
                for (int j = 0; j < 3; ++j) coef_s[pr * 12 + r * 4 + j] = k.A[r][j];
                coef_s[pr * 12 + r * 4 + 3] = k.C[r];
            }
        }
    }
    if (threadIdx.x == 0) {
        pair_cnt[0] = pair_cnt[1] = 0u;
        for (int i = 0; i < NSTAGE; ++i) { mbar_init(full_bar + i, 1); done_cnt[i] = 0u; }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    TRB_T(0);
    TileIter cur, ahead;
    iter_begin(cur, p, b, G);
    ahead = cur;
    // pairs this CTA never touches still owe their (zero) slot to the grid reduction: settle that now,
    // off the critical path.  Thread 0 walks the work list (a few columns) to mark the touched pairs.
    __shared__ unsigned touched[kMaxTmaPairs / 32];
    for (int i = threadIdx.x; i < kMaxTmaPairs / 32; i += kTmaThreads) touched[i] = 0u;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int r = 0; r < p.full_rounds; ++r) {
            const int pr = (r * G + b) / p.cols_per_pair;
            touched[pr >> 5] |= 1u << (pr & 31);
        }
        const long long t0 = p.tail_tiles * (long long)b / G, t1 = p.tail_tiles * (long long)(b + 1) / G;
        if (t1 > t0) {
            const int c0 = p.full_rounds * G + (int)(t0 / p.tiles_z), c1 = p.full_rounds * G + (int)((t1 - 1) / p.tiles_z);
            for (int pr = c0 / p.cols_per_pair; pr <= c1 / p.cols_per_pair; ++pr) touched[pr >> 5] |= 1u << (pr & 31);
        }
    }
    __syncthreads();
    // zero slots of the untouched pairs: plain stores now, their group arrivals with everybody else's after the main
    // loop (an arrival is a fence + a global atomic: ~1.5 us that used to sit in front of the first TMA issue)
    for (int pr = warp; pr < p.n_pairs; pr += kConsumerWarps) {
        if (touched[pr >> 5] & (1u << (pr & 31))) continue;
        double *mine = slot_ptr(p, pr, b);
        for (int v = lane; v < TRB_MOMENTS; v += 32) __stcg(mine + v, 0.0);
    }
    __shared__ ColConst colc[kConsumerWarps];   // each warp's copy of the footprint constants of `ahead`'s column
    if (threadIdx.x == 0) {                     // prologue: fill the ring
        TileIter t = cur;
        ColConst c;
        compute_col(c, t, p, coef_s, inv_d2, zoff);
        for (int i = 0; i < NSTAGE && t.phase != 2; ++i) {
            issue_tile<BX, BY, BZ>(t.tz_i, c, p, smem_raw + (size_t)i * L::kStageBytes, full_bar + i, meta + i, &map_mov, &map_tgt);
            if (iter_next(t, p, b, G) && t.phase != 2) compute_col(c, t, p, coef_s, inv_d2, zoff);
        }
    }
    for (int i = 0; i < NSTAGE && ahead.phase != 2; ++i) iter_next(ahead, p, b, G);   // ahead = cur + NSTAGE tiles
    if (lane == 0 && ahead.phase != 2) compute_col(colc[warp], ahead, p, coef_s, inv_d2, zoff);
    __syncwarp();

    // per-pair totals of this thread, folded with its x,y,z base coordinates.  Touched once per column
    // only: kept in local memory (volatile) so the 41 values do not occupy registers in the hot loop.
    float Tmem[TRB_MOMENTS];
    volatile float *T = Tmem;
#pragma unroll
    for (int i = 0; i < TRB_MOMENTS; ++i) T[i] = 0.f;
    int n_flush = 0;
    bool t_dirty = false;                       // T holds sums of earlier columns of the current pair

    int it = 0;
    while (cur.phase != 2) {
        // ---- column setup: this thread's x, y and the coordinate map of the pair ------------------------
        const int pair = cur.cg / p.cols_per_pair;
        const int col = cur.cg - pair * p.cols_per_pair;
        const int ty_i = col / p.tiles_x;
        const int x = (col - ty_i * p.tiles_x) * TX + lane, y = ty_i * TY + warp;
        const bool valid = (x < W) && (y < H);
        const float xv = __ldg(p.a.xb + min(x, W - 1)), yv = __ldg(p.a.yb + min(y, H - 1));
        float pxy[3], sz[3];
        {
            const Coef k = load_coef(coef_s, p, pair);
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                pxy[r] = fmaf(k.A[r][0], xv, fmaf(k.A[r][1], yv, fmaf(k.A[r][2], zoff, k.C[r])));
                sz[r] = k.A[r][2] * inv_d2;
            }
        }
        const float *__restrict__ mov = p.a.moving + (size_t)pair * p.a.pair_stride;
        // unfused pass: the warped samples are a by-product the caller may want (default-loss loop: the NMI term)
        const size_t HWs = (size_t)H * W;
        float *wcol = (!FUSED && p.a.warped_out && valid) ? p.a.warped_out + (size_t)pair * HWs * D + (size_t)y * W + x : nullptr;
        Acc A;
#pragma unroll
        for (int i = 0; i < 5; ++i) A.s[i] = f2(0.f);
#pragma unroll
        for (int kk = 0; kk < 3; ++kk)
#pragma unroll
            for (int r = 0; r < 3; ++r) A.P[kk][r] = A.Q[kk][r] = f2(0.f);

        bool col_done = false;
        while (!col_done) {
            const int stage = it % NSTAGE;
            const unsigned phase = (unsigned)(it / NSTAGE) & 1u;
#ifdef TRB_TIMING
            const unsigned long long tw0 = gtime();
#endif
            mbar_wait(full_bar + stage, phase);
#ifdef TRB_TIMING
            if (warp == 0 && lane == 0) { g_dbg[blockIdx.x * 16 + 7] += gtime() - tw0; g_dbg[blockIdx.x * 16 + 8] += 1ull; }
            if (blockIdx.x == 5 && lane == 0 && (warp == 0 || warp == 15) && it < 1000) { g_dbg[4096 + it * 4 + (warp == 15 ? 2 : 0)] = tw0; g_dbg[4096 + it * 4 + (warp == 15 ? 3 : 1)] = gtime(); }
#endif
            const TileMeta m = meta[stage];
            unsigned char *stg = smem_raw + (size_t)stage * L::kStageBytes;
            const uint32_t box_addr = smem_u32(stg);
            const uint32_t tg = box_addr + L::kBoxFloats * 4 + (uint32_t)(warp * TX + lane) * 4u;
            const int z0 = p.a.s_begin + cur.tz_i * TZ;
            const int nz = min(TZ, p.a.s_end - z0);
            if (valid) {
                if (m.fits) {
                    // index magic: 2.0 + rel * 2^-22 has bit pattern 0x40000000 + rel, and (bits << 2) wraps to 4*rel
                    const float Mrel = 2.f - kIdxScale * (float)(m.ox + BX * m.oy + BX * BY * m.oz);
                    const float zf0 = (float)z0;
                    if (nz == TZ) {
                        float2 zf = make_float2(zf0, zf0 + 1.f);
                        static_for<0, TZ / 2>([&](auto J) {
                            constexpr int j = decltype(J)::value;
                            const float2 ix = __ffma2_rn(f2(sz[0]), zf, f2(pxy[0]));
                            const float2 iy = __ffma2_rn(f2(sz[1]), zf, f2(pxy[1]));
                            const float2 iz = __ffma2_rn(f2(sz[2]), zf, f2(pxy[2]));
                            // immediates: the target tile advances TX*TY*4 bytes per z
                            const float2 t = make_float2(lds_f<(2 * j) * TX * TY * 4>(tg), lds_f<(2 * j + 1) * TX * TY * 4>(tg));
                            const float2 wv = pair_step<BX, BY, true, MSE_ONLY>(box_addr, Mrel, ix, iy, iz, t, zf, A);
                            if (!FUSED && wcol) { __stcs(wcol + (size_t)(z0 + 2 * j) * HWs, wv.x); __stcs(wcol + (size_t)(z0 + 2 * j + 1) * HWs, wv.y); }
                            zf = __fadd2_rn(zf, f2(2.f));
                        });
                    } else {
                        for (int zz = 0; zz < nz; zz += 2) {
                            const bool second = zz + 1 < nz;
                            const float za = zf0 + (float)zz;
                            const float2 zf = make_float2(za, second ? za + 1.f : za);
                            const float2 ix = __ffma2_rn(f2(sz[0]), zf, f2(pxy[0]));
                            const float2 iy = __ffma2_rn(f2(sz[1]), zf, f2(pxy[1]));
                            const float2 iz = __ffma2_rn(f2(sz[2]), zf, f2(pxy[2]));
                            const float2 t = make_float2(lds_f_dyn(tg + zz * (TX * TY * 4)),
                                                         lds_f_dyn(tg + (second ? zz + 1 : zz) * (TX * TY * 4)));
                            const float2 wv = second ? pair_step<BX, BY, true, MSE_ONLY>(box_addr, Mrel, ix, iy, iz, t, zf, A)
                                                     : pair_step<BX, BY, false, MSE_ONLY>(box_addr, Mrel, ix, iy, iz, t, zf, A);
                            if (!FUSED && wcol) {
                                __stcs(wcol + (size_t)(z0 + zz) * HWs, wv.x);
                                if (second) __stcs(wcol + (size_t)(z0 + zz + 1) * HWs, wv.y);
                            }
                        }
                    }
                } else {
                    for (int zz = 0; zz < nz; ++zz) {
                        const float zf = (float)(z0 + zz);
                        const float wv = voxel_direct<MSE_ONLY>(mov, D, H, W, fmaf(sz[0], zf, pxy[0]), fmaf(sz[1], zf, pxy[1]),
                                                                fmaf(sz[2], zf, pxy[2]), lds_f_dyn(tg + zz * (TX * TY * 4)), zf, A);
                        if (!FUSED && wcol) __stcs(wcol + (size_t)(z0 + zz) * HWs, wv);
                    }
                }
            }
            // ---- release the stage; the last warp to finish refills it with the tile NSTAGE ahead --------
            __syncwarp();
            if (lane == 0) {
                unsigned old;
                asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], 1;" : "=r"(old) : "r"(smem_u32(done_cnt + stage)) : "memory");
                if (old == kConsumerWarps - 1) {
                    done_cnt[stage] = 0u;
                    if (ahead.phase != 2)
                        issue_tile<BX, BY, BZ>(ahead.tz_i, colc[warp], p, stg, full_bar + stage, meta + stage, &map_mov, &map_tgt);
                }
            }
            ++it;
            if (ahead.phase != 2) {
                const bool moved = iter_next(ahead, p, b, G);
                if (moved && ahead.phase != 2 && lane == 0)
                    compute_col(colc[warp], ahead, p, coef_s, inv_d2, zoff);      // once per column, per warp
            }
            __syncwarp();
            col_done = iter_next(cur, p, b, G);
        }

        // ---- fold the column's sums with this thread's base coordinates (x, y constant over the column) --
        // The totals live in local memory, and with 219 KB of the SM given to the TMA ring the L1 left over (~28 KB)
        // cannot hold 512 x 164 B of them: every access is an L2 round trip.  `T[i] += v` on a volatile is load ->
        // add -> store per element, 41 SERIALISED round trips (measured: 13 us per column, a quarter of a 24-tile
        // column).  All loads first, then the arithmetic, then all stores: one round trip.
        const bool pair_done = cur.phase == 2 || cur.cg / p.cols_per_pair != pair;
        float acc[TRB_MOMENTS];
        if (t_dirty) {
#pragma unroll
            for (int i = 0; i < TRB_MOMENTS; ++i) acc[i] = T[i];
        } else {                                // first column of the pair in this CTA: nothing to load
#pragma unroll
            for (int i = 0; i < TRB_MOMENTS; ++i) acc[i] = 0.f;
        }
        if (valid) {
#pragma unroll
            for (int i = 0; i < 5; ++i) acc[i] += A.s[i].x + A.s[i].y;
#pragma unroll
            for (int kk = 0; kk < 3; ++kk)
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    const float pp = A.P[kk][r].x + A.P[kk][r].y, qq = A.Q[kk][r].x + A.Q[kk][r].y;
                    const int bi = 5 + kk * 12 + r * 4;
                    acc[bi + 0] = fmaf(xv, pp, acc[bi + 0]);
                    acc[bi + 1] = fmaf(yv, pp, acc[bi + 1]);
                    acc[bi + 2] += fmaf(inv_d2, qq, zoff * pp);
                    acc[bi + 3] += pp;
                }
        }
        if (!pair_done) {
#pragma unroll
            for (int i = 0; i < TRB_MOMENTS; ++i) T[i] = acc[i];
        }
        t_dirty = !pair_done;
        // ---- pair finished (for this CTA): hand its totals to the grid-level reduction ----------------
        if (pair_done) {
            // a warp can be at most one flush ahead of the slowest warp of its CTA (the TMA ring holds fewer
            // tiles than a pair has), so two scratch buffers alternate safely
#ifdef TRB_TIMING
            const unsigned long long tp0 = gtime();
#endif
            warp_publish_pair(acc, red[n_flush & 1], pair_cnt + (n_flush & 1), p, pair, G, warp, lane);
#ifdef TRB_TIMING
            if (warp == 0 && lane == 0) { g_dbg[blockIdx.x * 16 + 9] += gtime() - tp0; g_dbg[blockIdx.x * 16 + 10] += 1ull; }
#endif
            ++n_flush;
        }
    }
    // ---- deferred group arrivals of the pairs this CTA published (see warp_publish_pair) -----------
    __syncthreads();                            // every slot of this CTA has been written
    if (p.use_groups)
        for (int pr = warp; pr < p.n_pairs; pr += kConsumerWarps) warp_arrive_group(p, pr, G, lane);   // touched or zero
    TRB_T(1);
    // ---- the last CTA to get here finishes every pair ------------------------------------------------
    __shared__ int is_last_cta;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const unsigned done = atomicAdd(p.a.tickets + 126, 1u);
        is_last_cta = (done == (unsigned)G - 1u) ? 1 : 0;
    }
    __syncthreads();
    if (!is_last_cta) return;
    TRB_T(3);
    __threadfence();
    TRB_T(4);
    final_phase<FUSED>(p, reinterpret_cast<double *>(&red[0][0]), G, warp, lane);
    if (threadIdx.x == 0) p.a.tickets[126] = 0u;
    TRB_T(2);
}



bool tma_path_eligible(int ndim, const AffineParams &a, int n_pairs)
{
    if (ndim != 3) return false;
    if (a.W % 4 != 0 || a.W < TX || a.H < TY || (a.s_end - a.s_begin) < 1) return false;
    if (((uintptr_t)a.moving & 15) || ((uintptr_t)a.target & 15)) return false;
    if (n_pairs > 1 && (a.pair_stride % 4 != 0)) return false;
    if (n_pairs > kMaxTmaPairs) return false;
    // fp32 index trick range: |x + BX*y + BX*BY*z| < 2^22 with some headroom.  It also keeps every axis far below
    // kMaxFastFloorAxis, which the kMagic floor of the staged and clamped samples needs
    if ((double)a.W + (double)kBX * a.H + (double)kBX * kBY * a.D > 1.8e6) return false;
    {   // the pair-parity double buffer assumes a pair spans more tiles than the ring holds
        const long long tpp = (long long)((a.W + TX - 1) / TX) * ((a.H + TY - 1) / TY) * ((a.s_end - a.s_begin + TZ - 1) / TZ);
        if (n_pairs > 1 && tpp < 4 * kStages) return false;   // (tiles per pair; chunks only group them)
    }
    return encode_fn() != nullptr;
}

// Enqueue n_launch epochs (FUSED) or one moments pass (!FUSED) of the TMA kernel.
int launch_affine3d_tma(AffineParams a, int n_pairs, bool fused, int epoch0, int n_launch, cudaStream_t stream)
{
    using L = SmemLayout<kBX, kBY, kBZ>;
    CUtensorMap map_mov, map_tgt;
    int rc = make_map(&map_mov, a.moving, n_pairs, a.pair_stride, a.D, a.H, a.W, kBX, kBY, kBZ);
    if (rc) return rc;
    rc = make_map(&map_tgt, a.target, n_pairs, a.pair_stride, a.D, a.H, a.W, TX, TY, TZ);
    if (rc) return rc;
    TmaParams p;
    p.a = a;
    p.n_pairs = n_pairs;
    p.tiles_x = (a.W + TX - 1) / TX;
    p.tiles_y = (a.H + TY - 1) / TY;
    p.tiles_z = (a.s_end - a.s_begin + TZ - 1) / TZ;
    int sms, dev = 0;
    if ((rc = sm_count(sms))) return rc;
    cudaGetDevice(&dev);
    p.cols_per_pair = p.tiles_x * p.tiles_y;
    const long long total_cols = (long long)n_pairs * p.cols_per_pair;
    long long grid_ll = sms;
    if (grid_ll > total_cols * p.tiles_z) grid_ll = total_cols * p.tiles_z;
    if (grid_ll > kMaxSlots - 64) grid_ll = kMaxSlots - 64;       // slots G.. hold the group sums
    const int grid = (int)grid_ll;
    p.use_groups = n_pairs > 2 ? 1 : 0;        // measured: the direct fold only pays for one or two pairs
    p.full_rounds = (int)(total_cols / grid);
    p.tail_tiles = (total_cols - (long long)p.full_rounds * grid) * p.tiles_z;
    const size_t smem = (size_t)kStages * L::kStageBytes + 2 * kStages * sizeof(uint64_t) + kStages * sizeof(TileMeta);
    // MSE-only steps (w_ncc == 0: the reference's "criterion given" branch, warpings.py:38-40,125-127) need one
    // weighted moment family instead of three; the sharded (unfused) form always produces the full moment set
    const bool mse_only = fused && a.w_ncc == 0.f;
    auto kf = mse_only ? affine3d_tma_kernel<kBX, kBY, kBZ, kStages, true, true> : affine3d_tma_kernel<kBX, kBY, kBZ, kStages, true, false>;
    auto ku = affine3d_tma_kernel<kBX, kBY, kBZ, kStages, false, false>;
    // the attribute is per device: keep one flag per device ordinal (a process may drive several GPUs)
    static bool attr_set_dev[64] = {};
    bool &attr_set = attr_set_dev[dev & 63];
    if (!attr_set) {
        cudaError_t e = cudaFuncSetAttribute(affine3d_tma_kernel<kBX, kBY, kBZ, kStages, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(affine3d_tma_kernel<kBX, kBY, kBZ, kStages, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) e = cudaFuncSetAttribute(ku, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(tma kernel)");
        attr_set = true;
    }
    const unsigned long long seq0 = a.peer.seq;
    if (a.peer.world > 1 && (n_pairs != 1 || !fused)) { set_error("peer exchange is for ONE pair in the fused epoch kernel"); return TRB_ERR_ARG; }
    for (int e = 0; e < n_launch; ++e) {
        p.a.epoch = epoch0 + e;
        p.a.peer.seq = seq0 + (unsigned long long)e;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kTmaThreads); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        cudaError_t le = fused ? cudaLaunchKernelEx(&cfg, kf, p, map_mov, map_tgt) : cudaLaunchKernelEx(&cfg, ku, p, map_mov, map_tgt);
        if (le != cudaSuccess) return check_cuda(le, "cudaLaunchKernelEx(affine3d_tma)");
    }
    return check_cuda(cudaGetLastError(), "affine3d_tma");
}

}  // namespace trb
#ifdef TRB_TIMING
extern "C" int trb_debug_read(unsigned long long *out, int n) { return (int)cudaMemcpyFromSymbol(out, trb::g_dbg, sizeof(unsigned long long) * n); }
extern "C" int trb_debug_clear() { static unsigned long long z[1024 * 16]; return (int)cudaMemcpyToSymbol(trb::g_dbg, z, sizeof(z)); }
#endif
