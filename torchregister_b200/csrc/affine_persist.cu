// affine_persist.cu — persistent, warp-specialised 3-D rigid/affine registration: ALL epochs of a call in one
// cooperative launch (sm_100a).  Replaces the per-epoch launches of affine_tma.cu for the fused optimisation loop
// (reference loop bodies warpings.py:67-93 (affine) and :138-159 (rigid): F.affine_grid + F.grid_sample (:24-25),
// MSELoss / NCCLoss (utils.py:197-205), backward (:80,146), SGD.step (:81,147), best/loss bookkeeping (:83-93,149-159)).
//
// Why: with one launch per epoch the kernel paid, per epoch, a prologue (tensor maps, barrier init, ring fill), a
// column-end hand-over done by the compute warps themselves and a serial last-CTA reduction — 23 % of the batch epoch
// and 40 % of a 256^3 epoch (profiles/r01_notes.md).  Here:
//   * one CTA per SM lives for the whole optimisation; 16 CONSUMER warps (setmaxnreg 112) do nothing but
//     shared-memory loads and packed fp32 arithmetic on staged tiles — no global memory access, no atomics, no iteration
//     logic: they follow a stream of tile descriptors;
//   * a PRODUCER warp walks the CTA's tile list (the same column-cyclic decomposition as affine_tma.cu, repeated per
//     epoch), bounds each tile's source footprint under the current theta and issues the two TMA loads into a 4-stage
//     full/empty mbarrier ring;
//   * a REDUCER warp sums the 16 warp rows a column leaves in shared memory (fp64) and, when the CTA's run of tiles
//     of one pair ends, adds the 41 sums to the pair's accumulator in global memory with integer atomics
//     (fixed point, four 40-bit limbs per value: integer addition is associative, so the result is bit-reproducible
//     whatever the arrival order).  Every accumulator word carries its own contribution COUNT in its low 12 bits, so a
//     reader knows a word is complete without any fence, flag or ticket;
//   * theta of the next epoch is obtained by PULL: the producer of every CTA that needs pair p polls the pair's
//     accumulator of the previous epoch until all words are complete and runs the epilogue (loss, d theta, rigid
//     chain, SGD/Adam) itself on a private copy of the optimiser state in shared memory.  The epilogue is
//     deterministic, so all CTAs hold identical state; one designated CTA per pair writes loss log and final state.
//     There is no grid barrier and no "last block": with several pairs in the batch a CTA that needs theta of
//     (epoch e+1, pair p) finds epoch e of that pair completed long ago (other pairs' tiles were in between), so the
//     tile stream never stalls; with a single pair the hand-over is one atomic flight + one poll + the epilogue.
#include "affine_tile.cuh"
#include <cooperative_groups.h>
#include <vector>
#include <stdio.h>

namespace trb {

constexpr int kHelperWarps = 4;                                   // one warpgroup: setmaxnreg works on warpgroups
constexpr int kPersistThreads = kTmaThreads + kHelperWarps * 32;  // 640
constexpr int kConsumerRegs = 104, kHelperRegs = 64;               // 512*104 + 128*64 = 61440 = 640*96 (launch allocation)
constexpr int kColSlots = 8;
constexpr int kCoefSlots = 4;                                     // theta warp -> producer hand-over ring (segments)
constexpr int kStateSlots = 16;                                   // private optimiser-state copies (pairs a CTA touches)
constexpr int kLimbs = 4;
constexpr int kAccNan = kLimbs * TRB_MOMENTS;                     // word 164: count of non-finite contributions
constexpr int kAccWords = 168;                                    // per (epoch, pair): 4 x 41 limbs + nan word, padded
constexpr int kCountBits = 12;                                    // low bits of every word: contributions received
constexpr int kRedLdP = 44;
constexpr int kTargetWord = 100;                                  // tickets[pair*kTicketStride + 100]: contributions per epoch
constexpr int kTsumWord = 104;                                    // tickets[pair*kTicketStride + 104..119]: sum t, sum t^2 (2 x 4 limbs, u64)
constexpr int kTsumBlocks = 64;

enum { kFits = 1, kNewCol = 2, kEndCol = 4, kEnd = 8 };

#ifdef TRB_TIMING
__device__ unsigned long long g_pdbg[1024 * 32];
#define PT_NOW() gtime()
#define PT_ADD(slot, t0) do { if (lane == 0) g_pdbg[blockIdx.x * 32 + (slot)] += gtime() - (t0); } while (0)
#define PT_INC(slot) do { if (lane == 0) g_pdbg[blockIdx.x * 32 + (slot)] += 1ull; } while (0)
#define PT_SET(slot) do { if (lane == 0) g_pdbg[blockIdx.x * 32 + (slot)] = gtime(); } while (0)
#else
#define PT_NOW() 0ull
#define PT_ADD(slot, t0) do { (void)(t0); } while (0)
#define PT_INC(slot) do { } while (0)
#define PT_SET(slot) do { } while (0)
#endif

struct __align__(16) PTile { int ox, oy, oz, flags; float Mrel, zf0; int nz, colslot; };
struct __align__(16) PCol { int x0, y0, pair, pad; float coef[12]; };

struct PersistParams {
    TmaParams t;
    int tsum_blocks;                 // blocks per pair of target_sums_kernel (= count field of its words); 0: no target sums
    int moments_only;                // 1: ONE pass at the theta in `state`, the 41 moments go to a.moments_out, no update
    int n_epochs;                    // epochs in this launch (<= chunk capacity of the accumulator region)
    unsigned long long *acc;         // [n_epochs][n_pairs][kAccWords], zeroed before the launch
    const unsigned *targets;         // tickets region; word [pair*kTicketStride + kTargetWord]
    const unsigned long long *pairs_slot;   // gather variant: device word holding the address of the pair volume (or 0)
    int pair0;                       // first pair of this launch within the batch (sub-batches)
};

using PL = SmemLayout<kBX, kBY, kBZ>;
// the small arrays come first, the TMA ring last: its stage size depends on the kernel variant
constexpr size_t kOffBars = 0;
constexpr size_t kOffTiles = kOffBars + 24 * sizeof(uint64_t);
constexpr size_t kOffCols = kOffTiles + kStages * sizeof(PTile);
constexpr size_t kOffRed = kOffCols + kColSlots * sizeof(PCol);
constexpr size_t kOffState = kOffRed + 2 * kConsumerWarps * kRedLdP * sizeof(float);
constexpr size_t kOffAccw = kOffState + kStateSlots * TRB_STATE_FLOATS * sizeof(float);
constexpr size_t kOffMrow = kOffAccw + kAccWords * sizeof(unsigned long long);
constexpr size_t kOffCoefq = kOffMrow + 48 * sizeof(double);
constexpr size_t kOffStages = (kOffCoefq + kCoefSlots * 12 * sizeof(float) + 127) / 128 * 128;    // TMA destinations: 128-byte aligned
// ROT = false: a stage is the staged box of the moving volume + the target tile (TMA-staged variant);
// ROT = true : the target tile only — the moving volume is gathered through L1 (large-rotation variant, below)
template <bool ROT> struct Ring {
    static constexpr size_t kTgtOff = ROT ? 0 : (size_t)PL::kBoxFloats * 4;
    static constexpr size_t kStageBytes = ROT ? (size_t)PL::kTgtFloats * 4 : (size_t)PL::kStageBytes;
    static constexpr size_t kSmem = kOffStages + kStages * kStageBytes;
};
static_assert(Ring<false>::kSmem + 640 <= 232448, "persistent kernel: dynamic + static shared memory must stay within 227 KB");

__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long *p)
{
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_add_u64(unsigned long long *p, unsigned long long v)
{
    asm volatile("red.relaxed.gpu.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// helper warps wait for microseconds at a time: let the hardware suspend them (suspend-time hint) and back off between
// tries, so that they do not take issue slots from the consumer warps of their sub-partition (the first version's spin
// loops were 4 % of all executed instructions, ncu)
__device__ __forceinline__ void mbar_wait_sleepy(uint64_t *bar, unsigned parity)
{
    unsigned ok;
    for (;;) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(20000u) : "memory");
        if (ok) return;
        __nanosleep(200);
    }
}

// ---- fixed-point accumulators -----------------------------------------------------------------------------------
// x = q0*2^40 + q1 + q2*2^-40 + q3*2^-80 (+ a residual below 2^-80 that is dropped), |q1..3| < 2^40, |q0| < 2^39 for
// |x| < 2^79.  All steps are exact in fp64, so the decomposition does not depend on anything but x.
__device__ __forceinline__ void to_limbs(double x, long long (&q)[kLimbs])
{
    double r = x;
    q[0] = __double2ll_rz(r * 0x1p-40);
    r -= (double)q[0] * 0x1p40;
    q[1] = __double2ll_rz(r);
    r -= (double)q[1];
    q[2] = __double2ll_rz(r * 0x1p40);
    r -= (double)q[2] * 0x1p-40;
    q[3] = __double2ll_rz(r * 0x1p80);
}
__device__ __forceinline__ double from_limbs(const unsigned long long *w /*smem, stride TRB_MOMENTS*/, unsigned count)
{
    double q[kLimbs];
#pragma unroll
    for (int l = 0; l < kLimbs; ++l)
        q[l] = (double)((long long)(w[l * TRB_MOMENTS] - (unsigned long long)count) >> kCountBits);
    return (q[0] * 0x1p40 + q[1]) + (q[2] * 0x1p-40 + q[3] * 0x1p-80);
}


// sum t and sum t^2 of every pair's slab [s_begin, s_end): independent of theta, so computed once per launch instead
// of once per voxel and epoch.  fp64 per thread, fixed-point atomics across blocks (order independent, see to_limbs).
__global__ void __launch_bounds__(256) target_sums_kernel(const float *__restrict__ target, long long pair_stride, long long begin,
                                                          long long count, unsigned *tickets)
{
    const int pair = blockIdx.y;
    const float4 *src = reinterpret_cast<const float4 *>(target + (size_t)pair * pair_stride + begin);
    const long long n4 = count >> 2;
    double s = 0.0, ss = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (long long)gridDim.x * blockDim.x) {
        const float4 v = __ldg(src + i);
        s += ((double)v.x + (double)v.y) + ((double)v.z + (double)v.w);
        ss += ((double)v.x * v.x + (double)v.y * v.y) + ((double)v.z * v.z + (double)v.w * v.w);
    }
    s = warp_sum(s); ss = warp_sum(ss);
    __shared__ double sh[2][8];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { sh[0][warp] = s; sh[1][warp] = ss; }
    __syncthreads();
    if (threadIdx.x < 2) {
        double t = 0.0;
        for (int w = 0; w < 8; ++w) t += sh[threadIdx.x][w];
        unsigned long long *dst = reinterpret_cast<unsigned long long *>(tickets + (size_t)pair * kTicketStride + kTsumWord) + threadIdx.x * kLimbs;
        long long q[kLimbs];
        const bool fin = isfinite(t) && fabs(t) < 0x1p78;
        to_limbs(fin ? t : 0.0, q);
#pragma unroll
        for (int l = 0; l < kLimbs; ++l) red_add_u64(dst + l, ((unsigned long long)q[l] << kCountBits) + (fin ? 1ull : 0ull));
    }
}
__device__ __forceinline__ double tsum_read(const unsigned *tickets, int pair, int which, unsigned count)
{
    const unsigned long long *w = reinterpret_cast<const unsigned long long *>(tickets + (size_t)pair * kTicketStride + kTsumWord) + which * kLimbs;
    double q[kLimbs];
    bool ok = true;
#pragma unroll
    for (int l = 0; l < kLimbs; ++l) {
        const unsigned long long v = __ldcg(w + l);
        ok = ok && ((unsigned)(v & ((1ull << kCountBits) - 1ull)) == count);      // a non-finite block sum leaves the count short
        q[l] = (double)((long long)(v - (unsigned long long)(v & ((1ull << kCountBits) - 1ull))) >> kCountBits);
    }
    return ok ? (q[0] * 0x1p40 + q[1]) + (q[2] * 0x1p-40 + q[3] * 0x1p-80) : __longlong_as_double(0x7ff8000000000000ll);
}

// footprint constants of one column under the coordinate map k (compute_col of affine_tile.cuh without its smem cache)
__device__ __forceinline__ void compute_col_k(ColConst &c, const Coef &k, int pair, int col, const TmaParams &p,
                                              float inv_d2, float zoff)
{
    const int W = p.a.W, H = p.a.H;
    const int ty_i = col / p.tiles_x;
    const int x0 = (col - ty_i * p.tiles_x) * TX, y0 = ty_i * TY;
    const float xa = __ldg(p.a.xb + x0), xe = __ldg(p.a.xb + min(x0 + TX - 1, W - 1));
    const float ya = __ldg(p.a.yb + y0), ye = __ldg(p.a.yb + min(y0 + TY - 1, H - 1));
    const float za0 = fmaf(inv_d2, (float)p.a.s_begin, zoff);
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const float base = k.A[r][0] * xa + k.A[r][1] * ya + k.A[r][2] * za0 + k.C[r];
        const float dx = k.A[r][0] * (xe - xa), dy = k.A[r][1] * (ye - ya), dz = k.A[r][2] * inv_d2 * (float)(TZ - 1);
        c.lo[r] = base + fminf(dx, 0.f) + fminf(dy, 0.f) + fminf(dz, 0.f) - 0.03f;
        c.hi[r] = base + fmaxf(dx, 0.f) + fmaxf(dy, 0.f) + fmaxf(dz, 0.f) + 0.03f;
        c.step[r] = k.A[r][2] * inv_d2 * (float)TZ;
    }
    c.pair = pair; c.x0 = x0; c.y0 = y0;
}

// d params[j] of the 3-D rigid parametrisation (rigid_chain<3> of affine_shared.cuh, one component per call so that
// six lanes can work side by side).  g: d loss / d theta (12 doubles, shared memory).
__device__ double rigid_chain_component(const float *p, const double *g, int j)
{
    if (j >= 3) {
        const double t = tanh((double)p[j]);
        return g[3 + 4 * (j - 3)] * 0.25 * (1.0 - t * t);
    }
    double sps, cps, sth, cth, sph, cph;
    sincos((double)p[0], &sps, &cps);
    sincos((double)p[1], &sth, &cth);
    sincos((double)p[2], &sph, &cph);
    if (j == 0)
        return g[0] * (-sps * cth) + g[1] * (sph * cps * cth) + g[2] * (cph * cps * cth)
             + g[4] * (-sps * sth) + g[5] * (sph * cps * sth) + g[6] * (cph * cps * sth)
             - g[8] * cps - g[9] * (sph * sps) - g[10] * (cph * sps);
    if (j == 1)
        return -g[0] * (cps * sth) - g[1] * (sph * sps * sth + cph * cth) + g[2] * (sph * cth - cph * sps * sth)
             + g[4] * (cps * cth) + g[5] * (sph * sps * cth - cph * sth) + g[6] * (cph * sps * cth + sph * sth);
    return g[1] * (cph * sps * cth + sph * sth) + g[2] * (cph * sth - sph * sps * cth)
         + g[5] * (cph * sps * sth - sph * cth) - g[6] * (sph * sps * sth + cph * cth)
         + g[9] * (cph * cps) - g[10] * (sph * cps);
}

// Warp-cooperative form of affine_epilogue_core<3, true>: lane i owns entry i of theta / params, so nothing lives in
// per-thread arrays (the helper warps run on 64 registers and local memory is an L2 round trip here: the serial form
// took 5 us, most of it spill traffic).  Same expression per entry as the serial form.  st, gs: shared memory.
// (force-inlined: a call would pass the kernel parameters by address, i.e. copy all of them to local memory at kernel entry)
__device__ __forceinline__ float affine_epilogue_warp(const double *M, const AffineParams &p, int epoch, float *st, double *gs, int lane)
{
    const double n = (double)p.D * (double)p.H * (double)p.W;
    const LossCoef lc = loss_coefficients(n, M[0], M[1], M[2], M[3], M[4], (double)p.w_mse, (double)p.w_ncc);
    const float loss = (float)lc.loss;
    const bool improved = (epoch == 0 || loss < st[TRB_STATE_BEST_LOSS]);
    const bool rigid = p.mode == TRB_MODE_RIGID;
    const int np = rigid ? 6 : 12;
    float par = 0.f, th_cur = 0.f;
    if (lane < 12) {
        par = st[TRB_STATE_PARAMS + lane];
        th_cur = st[TRB_STATE_THETA + lane];
        const int r = lane >> 2;
        const double scale = r == 0 ? 0.5 * p.W : (r == 1 ? 0.5 * p.H : 0.5 * p.D);
        gs[lane] = (lc.cw * M[29 + lane] + lc.ct * M[17 + lane] + lc.c0 * M[5 + lane]) * scale;
    }
    __syncwarp();
    if (improved && lane < 12) st[TRB_STATE_BEST_THETA + lane] = th_cur;
    if (lane == 0) {
        if (improved) st[TRB_STATE_BEST_LOSS] = loss;
        st[TRB_STATE_LAST_LOSS] = loss;
    }
    if (lane < np) {
        const double dp = rigid ? rigid_chain_component(st + TRB_STATE_PARAMS, gs, lane) : gs[lane];
        const float g = (float)dp;
        float v = par;
        if (p.optimiser == TRB_OPT_SGD) {
            v = v - p.lr * g;
        } else {
            const float t = (float)(epoch + 1);
            float m = st[TRB_STATE_ADAM_M + lane], sq = st[TRB_STATE_ADAM_V + lane];
            m = p.beta1 * m + (1.f - p.beta1) * g;
            sq = p.beta2 * sq + (1.f - p.beta2) * g * g;
            st[TRB_STATE_ADAM_M + lane] = m;
            st[TRB_STATE_ADAM_V + lane] = sq;
            const float bc1 = 1.f - powf(p.beta1, t), bc2 = 1.f - powf(p.beta2, t);
            v = v - (p.lr / bc1) * (m / (sqrtf(sq) / sqrtf(bc2) + p.adam_eps));
        }
        par = v;
    }
    __syncwarp();                                   // every lane has read the old params (rigid chain) before they change
    if (lane < np) st[TRB_STATE_PARAMS + lane] = par;
    __syncwarp();
    if (rigid) {
        if (lane == 0) {
            float th[12];
            rigid_theta<3>(st + TRB_STATE_PARAMS, th);
#pragma unroll
            for (int i = 0; i < 12; ++i) st[TRB_STATE_THETA + i] = th[i];
        }
    } else if (lane < 12) {
        st[TRB_STATE_THETA + lane] = par;
    }
    __syncwarp();
    return loss;
}

// ---- theta warp: theta of (epoch e_rel, pair) into the CTA's private state slot ---------------------------------
// e_rel == 0: the state loaded at kernel start is current.  Otherwise wait for the pair's accumulator of epoch
// e_rel-1 to be complete (every word's count field == contributions per epoch), rebuild the 41 moments and run the
// epilogue on the private state.  All 32 lanes take part.
__device__ __forceinline__ void acquire_theta(const PersistParams &pp, int e_rel, int pair, float *st, bool writer, unsigned target,
                              const double *tsum /* sum t, sum t^2 of the pair, or NULL (MSE only) */,
                              unsigned long long *accw, double *mrow, int lane)
{
    if (e_rel == 0) return;
    const AffineParams &a = pp.t.a;
    const unsigned long long *A = pp.acc + ((size_t)(e_rel - 1) * pp.t.n_pairs + pair) * kAccWords;
    const unsigned long long cmask = (1ull << kCountBits) - 1ull;
    const unsigned long long tq0 = PT_NOW();
    unsigned backoff = 32;
    const unsigned backoff_max = pp.t.n_pairs <= 2 ? 96u : 1024u;   // few pairs: every CTA waits for this hand-over
    for (;;) {
        // cheap probe first: one word (the one the contributors add last), then the full check
        unsigned long long probe = 0ull;
        if (lane == 0) probe = ld_relaxed_u64(A + kAccNan);
        probe = __shfl_sync(kFull, probe, 0);
        if ((unsigned)(probe & cmask) == target) {
            bool ok = true;
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                const int i = lane + 32 * j;
                if (i <= kAccNan) {
                    const unsigned long long v = ld_relaxed_u64(A + i);
                    accw[i] = v;
                    ok = ok && ((unsigned)(v & cmask) == target);
                }
            }
            if (__all_sync(kFull, ok)) break;
        }
        PT_INC(16);
        __nanosleep(backoff);                      // 32 ns .. 1 us: short while the hand-over is imminent (few pairs), cheap otherwise
        if (backoff < backoff_max) backoff += backoff >> 1;
    }
    PT_ADD(2, tq0);
    const unsigned long long te0 = PT_NOW();
    __syncwarp();
    const bool bad = (accw[kAccNan] >> kCountBits) != 0ull;
    for (int v = lane; v < TRB_MOMENTS; v += 32)
        mrow[v] = bad ? __longlong_as_double(0x7ff8000000000000ll) : from_limbs(accw + v, target);
    __syncwarp();
    if (tsum && lane == 0 && !bad) { mrow[0] = tsum[0]; mrow[2] = tsum[1]; }
    __syncwarp();
    if (pp.moments_only) {                       // unfused pass (sharded NCCL form, NMI path, vjp): hand the sums out
        if (writer)
            for (int v = lane; v < TRB_MOMENTS; v += 32) a.moments_out[(size_t)pair * TRB_MOMENTS + v] = mrow[v];
        __syncwarp();
        return;
    }
    if (a.peer.world > 1) {
        // one volume sharded into z-slabs over the GPUs of the box: the designated CTA of every rank pushes this
        // rank's 41 sums into every rank's mailbox over NVLink (peer.cuh), EVERY CTA of a rank then reads its own
        // rank's mailbox (local memory) and adds the contributions in rank order, so all CTAs of all ranks continue
        // with identical moments.  Two parities of slots suffice: a rank can push epoch e+2 only after every rank
        // pushed e+1, i.e. after all their CTAs finished reading epoch e.
        const PeerExchange &x = a.peer;
        const unsigned long long seq = x.seq + (unsigned long long)(e_rel - 1);
        const size_t par = (size_t)(seq & 1ull) * 8 * kMailSlot;
        if (writer) {
            for (int r = 0; r < x.world; ++r) {
                volatile double *dst = x.mailbox[r] + par + (size_t)x.rank * kMailSlot;
                for (int v = lane; v < TRB_MOMENTS; v += 32) dst[v] = mrow[v];
            }
            __threadfence_system();
            __syncwarp();
            if (lane < x.world) {
                unsigned long long *flag = reinterpret_cast<unsigned long long *>(x.mailbox[lane] + par + (size_t)x.rank * kMailSlot + (kMailSlot - 1));
                asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(flag), "l"(seq) : "memory");
            }
        }
        double *mine = x.mailbox[x.rank] + par;
        volatile unsigned long long *poison = reinterpret_cast<volatile unsigned long long *>(x.mailbox[x.rank] + kMailPoison);
        bool ok = *poison == 0ull;
        if (ok && lane < x.world) {
            const unsigned long long *flag = reinterpret_cast<const unsigned long long *>(mine + (size_t)lane * kMailSlot + (kMailSlot - 1));
            unsigned long long got = 0;
            long long spins = 0;
            do {
                asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(got) : "l"(flag) : "memory");
                if (got != seq) __nanosleep(40);
            } while (got != seq && ++spins < (1ll << 24));
            ok = got == seq;
        }
        ok = __all_sync(kFull, ok);
        if (!ok && lane == 0) *poison = 1ull;
        for (int v = lane; v < TRB_MOMENTS; v += 32) {
            double t = 0.0;
            for (int r = 0; r < x.world; ++r) t += reinterpret_cast<volatile const double *>(mine)[(size_t)r * kMailSlot + v];
            mrow[v] = ok ? t : __longlong_as_double(0x7ff8000000000000ll);
        }
        __syncwarp();
    }
    const int epoch = a.epoch + e_rel - 1;
    const float loss = affine_epilogue_warp(mrow, a, epoch, st, reinterpret_cast<double *>(accw) /* words are consumed: scratch */, lane);
    if (lane == 0 && writer && a.loss_log) a.loss_log[(size_t)pair * a.log_stride + epoch] = loss;
    __syncwarp();
    PT_ADD(3, te0);
}

// ROT (large rotations, e.g. the reference's own torch.rand(6) start, utils.py:317): the source footprint of a 32x16x8
// tile is a rotated box whose axis-aligned hull is 4-9x the tile, so staging it by TMA does not pay (the TMA variant
// then falls back to uncached global gathers, 5.5x slower).  This variant stages only the target tile (64 KB of shared
// memory instead of 219 KB, which leaves ~128 KB of L1), maps a warp onto an 8x4 (x,y) patch instead of a 32-voxel row —
// the 8 corner loads of a patch touch a compact source region — and gathers the moving volume through L1.
// STORE (unfused one-pass mode only): the staged path also leaves the warped samples in a.warped_out (the gather
// variant decides that at run time)
// PAIRS (gather variant only): the moving volume is read through the pair volume whose address sits in the workspace
// (trb_affine_attach_pairs; the caller says so with TRB_FLAG_PAIR_VOLUME) — a separate instantiation, so that the scalar
// gather loop keeps its registers and its unrolling
template <bool MSE_ONLY, bool ROT, bool STORE = false, int PAIRS = 0>     // PAIRS: 0 scalar gathers, 1 pair volume, 2 quad volume
__global__ void __launch_bounds__(kPersistThreads, 1)
affine3d_persist_kernel(const PersistParams pp, const __grid_constant__ CUtensorMap map_mov,
                        const __grid_constant__ CUtensorMap map_tgt)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + kOffBars);
    uint64_t *full_bar = bars, *empty_bar = bars + kStages, *red_full = bars + 2 * kStages, *red_empty = red_full + 2;
    uint64_t *coef_full = red_empty + 2, *coef_empty = coef_full + kCoefSlots;
    float *coefq = reinterpret_cast<float *>(smem_raw + kOffCoefq);                 // [kCoefSlots][12]
    PTile *tiles = reinterpret_cast<PTile *>(smem_raw + kOffTiles);
    PCol *cols = reinterpret_cast<PCol *>(smem_raw + kOffCols);
    float *red = reinterpret_cast<float *>(smem_raw + kOffRed);                 // [2][16][kRedLdP]
    float *state_s = reinterpret_cast<float *>(smem_raw + kOffState);           // [kStateSlots][TRB_STATE_FLOATS]
    unsigned long long *accw = reinterpret_cast<unsigned long long *>(smem_raw + kOffAccw);
    double *mrow = reinterpret_cast<double *>(smem_raw + kOffMrow);

    const TmaParams &p = pp.t;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int W = p.a.W, H = p.a.H, D = p.a.D;
    const int G = gridDim.x, b = blockIdx.x;
    const float inv_d2 = 2.f / (float)D, zoff = 1.f / (float)D - 1.f;      // zv(z) = (2z+1)/D - 1

    if (threadIdx.x == 0) {
        for (int i = 0; i < kStages; ++i) { mbar_init(full_bar + i, 1); mbar_init(empty_bar + i, kConsumerWarps); }
        for (int i = 0; i < 2; ++i) { mbar_init(red_full + i, kConsumerWarps); mbar_init(red_empty + i, 1); }
        for (int i = 0; i < kCoefSlots; ++i) { mbar_init(coef_full + i, 1); mbar_init(coef_empty + i, 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp >= kConsumerWarps) {
        // =================================== helper warpgroup =====================================================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kHelperRegs));
        const int h = warp - kConsumerWarps;
        if (h == 0) {
            // ------------------------------- producer ---------------------------------------------------------
            PT_SET(6);
            int it = 0, k = 0, seg = 0;
            for (int e_rel = 0; e_rel < pp.n_epochs; ++e_rel) {
                TileIter t;
                iter_begin(t, p, b, G);
                int cur_pair = -1;
                bool newcol = true;
                ColConst c;
                Coef kf;
                while (t.phase != 2) {
                    if (newcol) {
                        const unsigned long long tc0 = PT_NOW();
                        const int pair = t.cg / p.cols_per_pair;
                        if (pair != cur_pair) {
                            // coordinate map of this run of tiles: produced ahead of time by the theta warp
                            const unsigned long long ta0 = PT_NOW();
                            PT_INC(1);
                            cur_pair = pair;
                            const int cs = seg % kCoefSlots;
                            mbar_wait_sleepy(coef_full + cs, (unsigned)(seg / kCoefSlots) & 1u);
                            const float *cq = coefq + cs * 12;
#pragma unroll
                            for (int r = 0; r < 3; ++r) {
#pragma unroll
                                for (int j = 0; j < 3; ++j) kf.A[r][j] = cq[r * 4 + j];
                                kf.C[r] = cq[r * 4 + 3];
                            }
                            __syncwarp();
                            if (lane == 0) mbar_arrive(coef_empty + cs);
                            ++seg;
                            PT_ADD(0, ta0);
                        }
                        compute_col_k(c, kf, pair, t.cg - pair * p.cols_per_pair, p, inv_d2, zoff);
                        if (lane == 0) {
                            PCol &pc = cols[k % kColSlots];
                            pc.x0 = c.x0; pc.y0 = c.y0; pc.pair = pair; pc.pad = 0;
#pragma unroll
                            for (int r = 0; r < 3; ++r) {
#pragma unroll
                                for (int j = 0; j < 3; ++j) pc.coef[r * 4 + j] = kf.A[r][j];
                                pc.coef[r * 4 + 3] = kf.C[r];
                            }
                        }
                        PT_ADD(5, tc0);
                    }
                    const int stage = it % kStages;
                    const unsigned long long tw0 = PT_NOW();
                    if (it >= kStages) mbar_wait_sleepy(empty_bar + stage, (unsigned)((it / kStages) - 1) & 1u);
                    PT_ADD(4, tw0);
                    TileIter nx = t;
                    const bool moved = iter_next(nx, p, b, G);
                    if (lane == 0) {
                        // footprint of this tile -> box origin / fits (issue_tile of affine_tile.cuh with the extra stream fields)
                        int o[3];
                        bool fits = !ROT;
                        const int B[3] = {kBX, kBY, kBZ};
                        const float kfz = (float)t.tz_i;
#pragma unroll
                        for (int r = 0; r < 3; ++r) {
                            const float lo = fmaf(kfz, c.step[r], c.lo[r]), hi = fmaf(kfz, c.step[r], c.hi[r]);
                            const float loc = fminf(fmaxf(lo, -1.0e6f), 1.0e6f), hic = fminf(fmaxf(hi, -1.0e6f), 1.0e6f);
                            o[r] = r == 0 ? 4 * (int)floorf(loc * 0.25f) : (int)floorf(loc);
                            fits = fits && ((int)floorf(hic) + 1 <= o[r] + B[r] - 1);
                        }
                        fits = fits && (fabsf((float)o[0]) + kBX * fabsf((float)o[1]) + (float)(kBX * kBY) * fabsf((float)o[2]) < 1.9e6f);
                        const int z0 = p.a.s_begin + t.tz_i * TZ;
                        PTile m;
                        m.ox = o[0]; m.oy = o[1]; m.oz = o[2];
                        m.flags = (fits ? kFits : 0) | (newcol ? kNewCol : 0) | (moved ? kEndCol : 0);
                        m.Mrel = 2.f - kIdxScale * (float)(o[0] + kBX * o[1] + kBX * kBY * o[2]);
                        m.zf0 = (float)z0;
                        m.nz = min(TZ, p.a.s_end - z0);
                        m.colslot = k % kColSlots;
                        tiles[stage] = m;
                        unsigned char *stg = smem_raw + kOffStages + (size_t)stage * Ring<ROT>::kStageBytes;
                        const unsigned tgt_bytes = PL::kTgtFloats * 4, box_bytes = PL::kBoxFloats * 4;
                        mbar_arrive_expect_tx(full_bar + stage, fits ? (tgt_bytes + box_bytes) : tgt_bytes);
                        if (fits) tma_load_4d(stg, &map_mov, full_bar + stage, o[0], o[1], o[2], c.pair);
                        tma_load_4d(stg + Ring<ROT>::kTgtOff, &map_tgt, full_bar + stage, c.x0, c.y0, z0, c.pair);
                    }
                    __syncwarp();
                    if (moved) ++k;
                    newcol = moved;
                    t = nx;
                    ++it;
                }
            }
            PT_SET(7);
            {   // end of stream
                const int stage = it % kStages;
                if (it >= kStages) mbar_wait_sleepy(empty_bar + stage, (unsigned)((it / kStages) - 1) & 1u);
                if (lane == 0) {
                    PTile m = {};
                    m.flags = kEnd;
                    tiles[stage] = m;
                    mbar_arrive(full_bar + stage);
                }
            }
        } else if (h == 1) {
            // ------------------------------- reducer ----------------------------------------------------------
            int k = 0;
            for (int e_rel = 0; e_rel < pp.n_epochs; ++e_rel) {
                TileIter t;
                iter_begin(t, p, b, G);
                double s0 = 0.0, s1 = 0.0;
                while (t.phase != 2) {
                    const int pair = t.cg / p.cols_per_pair;
                    if (!iter_next(t, p, b, G)) continue;                // walk to the end of the column piece
                    const int cbuf = k & 1;
                    const unsigned long long tr0 = PT_NOW();
                    mbar_wait_sleepy(red_full + cbuf, (unsigned)(k >> 1) & 1u);
                    PT_ADD(14, tr0);
                    const unsigned long long tp0 = PT_NOW();
                    const float *rows = red + cbuf * (kConsumerWarps * kRedLdP);
                    const int v1 = min(lane + 32, TRB_MOMENTS - 1);
                    double a0 = 0.0, a1 = 0.0;
#pragma unroll
                    for (int w = 0; w < kConsumerWarps; ++w) { a0 += (double)rows[w * kRedLdP + lane]; a1 += (double)rows[w * kRedLdP + v1]; }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(red_empty + cbuf);
                    s0 += a0; s1 += a1;
                    ++k;
                    const bool seg_end = t.phase == 2 || t.cg / p.cols_per_pair != pair;
                    if (seg_end) {
                        unsigned long long *A = pp.acc + ((size_t)e_rel * p.n_pairs + pair) * kAccWords;
                        const bool fin0 = isfinite(s0) && fabs(s0) < 0x1p78, fin1 = lane + 32 >= TRB_MOMENTS || (isfinite(s1) && fabs(s1) < 0x1p78);
                        const unsigned badm = __ballot_sync(kFull, !(fin0 && fin1));
                        long long q[kLimbs];
                        to_limbs(fin0 ? s0 : 0.0, q);
#pragma unroll
                        for (int l = 0; l < kLimbs; ++l) red_add_u64(A + l * TRB_MOMENTS + lane, ((unsigned long long)q[l] << kCountBits) + 1ull);
                        if (lane + 32 < TRB_MOMENTS) {
                            to_limbs(fin1 ? s1 : 0.0, q);
#pragma unroll
                            for (int l = 0; l < kLimbs; ++l) red_add_u64(A + l * TRB_MOMENTS + lane + 32, ((unsigned long long)q[l] << kCountBits) + 1ull);
                        }
                        // the probe word goes last (acquire_theta looks at it first)
                        if (lane == 0) red_add_u64(A + kAccNan, ((unsigned long long)(badm ? 1 : 0) << kCountBits) + 1ull);
                        s0 = s1 = 0.0;
                    }
                    PT_ADD(15, tp0);
                }
            }
        } else if (h == 2) {
            // ------------------------------- theta warp -------------------------------------------------------
            // private optimiser state of the pairs this CTA touches, in stream order (pairs are non-decreasing along
            // the stream, so "slot" is simply the index of the run of equal pairs); then, run after run and epoch after
            // epoch, the coordinate map the producer needs next
            __shared__ int slot_pair[kStateSlots];
            __shared__ unsigned slot_target[kStateSlots];
            __shared__ int slot_writer[kStateSlots];
            __shared__ double slot_tsum[kStateSlots][2];
            const bool need_tsum = !MSE_ONLY;
            int n_slots = 0;
            {
                TileIter t;
                iter_begin(t, p, b, G);
                int last = -1;
                bool newcol = true;
                while (t.phase != 2) {
                    const int pair = t.cg / p.cols_per_pair;
                    if (newcol && pair != last) {
                        if (n_slots < kStateSlots) {
                            if (lane == 0) {
                                slot_pair[n_slots] = pair;
                                slot_target[n_slots] = pp.targets[(size_t)pair * kTicketStride + kTargetWord];
                                slot_writer[n_slots] = (t.cg == pair * p.cols_per_pair && t.tz_i == 0) ? 1 : 0;
                            }
                            if (need_tsum && lane < 2) slot_tsum[n_slots][lane] = pp.tsum_blocks > 0 ? tsum_read(pp.targets, pair, lane, (unsigned)pp.tsum_blocks) : 0.0;
                            const float *src = p.a.state + (size_t)pair * TRB_STATE_FLOATS;
                            if (pp.moments_only) {          // only theta is read (the caller may pass a bare theta rebased by -12)
                                if (lane < 12) state_s[n_slots * TRB_STATE_FLOATS + TRB_STATE_THETA + lane] = __ldcg(src + TRB_STATE_THETA + lane);
                            } else {
                                state_s[n_slots * TRB_STATE_FLOATS + lane] = __ldcg(src + lane);
                                state_s[n_slots * TRB_STATE_FLOATS + 32 + lane] = __ldcg(src + 32 + lane);
                            }
                        }
                        ++n_slots;
                        last = pair;
                    }
                    newcol = iter_next(t, p, b, G);
                }
                if (n_slots > kStateSlots) n_slots = kStateSlots;      // (the host never launches such a decomposition)
            }
            __syncwarp();
            int seg = 0;
            for (int e_rel = 0; e_rel < pp.n_epochs; ++e_rel) {
                for (int sl = 0; sl < n_slots; ++sl, ++seg) {
                    float *st = state_s + sl * TRB_STATE_FLOATS;
                    acquire_theta(pp, e_rel, slot_pair[sl], st, slot_writer[sl] != 0, slot_target[sl], need_tsum ? slot_tsum[sl] : nullptr, accw, mrow, lane);
                    const int cs = seg % kCoefSlots;
                    if (seg >= kCoefSlots) mbar_wait_sleepy(coef_empty + cs, (unsigned)((seg / kCoefSlots) - 1) & 1u);
                    if (lane < 12) {
                        // make_coef of affine_tile.cuh, one entry per lane
                        const int r = lane >> 2, cidx = lane & 3;
                        const float hr = r == 0 ? 0.5f * W : (r == 1 ? 0.5f * H : 0.5f * D);
                        const float th = st[TRB_STATE_THETA + lane];
                        coefq[cs * 12 + lane] = cidx < 3 ? th * hr : fmaf(th + 1.f, hr, -0.5f);
                    }
                    __syncwarp();
                    if (lane == 0) mbar_arrive(coef_full + cs);
                }
            }
            // the designated CTA of every pair finishes the last epoch and writes the state back
            for (int sl = 0; sl < n_slots; ++sl) {
                if (!slot_writer[sl]) continue;
                float *st = state_s + sl * TRB_STATE_FLOATS;
                acquire_theta(pp, pp.n_epochs, slot_pair[sl], st, true, slot_target[sl], need_tsum ? slot_tsum[sl] : nullptr, accw, mrow, lane);
                if (pp.moments_only) continue;
                float *dst = p.a.state + (size_t)slot_pair[sl] * TRB_STATE_FLOATS;
                dst[lane] = st[lane];
                dst[32 + lane] = st[32 + lane];
            }
        }
        return;
    }

    // ======================================= consumers ============================================================
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kConsumerRegs));
    int x = 0, y = 0;
    bool valid = false;
    float xv = 0.f, yv = 0.f, pxy[3] = {0.f, 0.f, 0.f}, sz[3] = {0.f, 0.f, 0.f};
    const float *__restrict__ mov = p.a.moving;
    // gather variant: the pair volume (trb_affine_attach_pairs), if the caller built one
    const char *pairs_all = PAIRS ? reinterpret_cast<const char *>(__ldcg(pp.pairs_slot)) : nullptr;
    const char *pairs = nullptr;
    float *wcol0 = nullptr;              // STORE: this thread's column of the warped output
    Acc2 A;
    int kcol = 0;
    for (int it = 0;; ++it) {
        const int stage = it % kStages;
#ifdef TRB_TIMING
        const unsigned long long tf0 = gtime();
#endif
        mbar_wait(full_bar + stage, (unsigned)(it / kStages) & 1u);
#ifdef TRB_TIMING
        if (lane == 0 && warp == 0) { g_pdbg[blockIdx.x * 32 + 8] += gtime() - tf0; g_pdbg[blockIdx.x * 32 + 9] += 1ull; }
        if (lane == 0 && warp == 15) { g_pdbg[blockIdx.x * 32 + 13] += gtime() - tf0; }
        if (blockIdx.x == 5 && lane == 0 && warp == 0 && it < 600) { g_pdbg[8192 + it * 2] = tf0; g_pdbg[8192 + it * 2 + 1] = gtime(); }
        const unsigned long long ts0 = gtime();
#endif
        const PTile m = tiles[stage];
        if (m.flags & kEnd) break;
        if (m.flags & kNewCol) {
            const PCol &pc = cols[m.colslot];
            x = pc.x0 + (ROT ? 8 * (warp & 3) + (lane & 7) : lane);
            y = pc.y0 + (ROT ? 4 * (warp >> 2) + (lane >> 3) : warp);
            valid = (x < W) && (y < H);
            xv = __ldg(p.a.xb + min(x, W - 1)); yv = __ldg(p.a.yb + min(y, H - 1));
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                pxy[r] = fmaf(pc.coef[r * 4 + 0], xv, fmaf(pc.coef[r * 4 + 1], yv, fmaf(pc.coef[r * 4 + 2], zoff, pc.coef[r * 4 + 3])));
                sz[r] = pc.coef[r * 4 + 2] * inv_d2;
            }
            mov = p.a.moving + (size_t)pc.pair * p.a.pair_stride;
            if constexpr (PAIRS == 1) pairs = pairs_all + (size_t)(pp.pair0 + pc.pair) * ((size_t)D * H * (W + kPairPad)) * sizeof(float2);
            if constexpr (PAIRS == 2) pairs = pairs_all + (size_t)(pp.pair0 + pc.pair) * ((size_t)D * (H + kPairPad) * (W + kPairPad)) * sizeof(float4);
            if constexpr (STORE) wcol0 = p.a.warped_out + (size_t)pc.pair * p.a.pair_stride + (size_t)y * W + x;
#pragma unroll
            for (int i = 0; i < 12; ++i) A.a[i] = f2(0.f);
#ifdef TRB_TIMING
            if (lane == 0 && warp == 0) { g_pdbg[blockIdx.x * 32 + 12] += gtime() - ts0; }
#endif
        }
        unsigned char *stg = smem_raw + kOffStages + (size_t)stage * Ring<ROT>::kStageBytes;
        const uint32_t box_addr = smem_u32(stg);
        const uint32_t tg = box_addr + (uint32_t)Ring<ROT>::kTgtOff +
                            (uint32_t)(ROT ? (4 * (warp >> 2) + (lane >> 3)) * TX + 8 * (warp & 3) + (lane & 7) : warp * TX + lane) * 4u;
        const int nz = m.nz;
        if (valid) {
            if (!ROT && (m.flags & kFits)) {
                const float Mrel = m.Mrel;
                const float zf0 = m.zf0;
                // full tiles (and half tiles: volumes whose depth is a multiple of TZ/2) run unrolled with immediate offsets
                auto run_steps = [&](auto NS) {
                    float2 zf = make_float2(zf0, zf0 + 1.f);
                    static_for<0, decltype(NS)::value>([&](auto J) {
                        constexpr int j = decltype(J)::value;
                        const float2 ix = __ffma2_rn(f2(sz[0]), zf, f2(pxy[0]));
                        const float2 iy = __ffma2_rn(f2(sz[1]), zf, f2(pxy[1]));
                        const float2 iz = __ffma2_rn(f2(sz[2]), zf, f2(pxy[2]));
                        // immediates: the target tile advances TX*TY*4 bytes per z
                        const float2 t = make_float2(lds_f<(2 * j) * TX * TY * 4>(tg), lds_f<(2 * j + 1) * TX * TY * 4>(tg));
                        const float2 wv = pair_step2<kBX, kBY, true, MSE_ONLY>(box_addr, Mrel, ix, iy, iz, t, zf, A);
                        if constexpr (STORE) {
                            const size_t HWs = (size_t)H * W;
                            float *wz = wcol0 + (size_t)(int)zf0 * HWs;
                            __stcs(wz + (size_t)(2 * j) * HWs, wv.x);
                            __stcs(wz + (size_t)(2 * j + 1) * HWs, wv.y);
                        }
                        zf = __fadd2_rn(zf, f2(2.f));
                    });
                };
                if (nz == TZ) run_steps(std::integral_constant<int, TZ / 2>{});
                else if (TZ >= 16 && nz == TZ / 2) run_steps(std::integral_constant<int, TZ / 4>{});
                else {
                    for (int zz = 0; zz < nz; zz += 2) {
                        const bool second = zz + 1 < nz;
                        const float za = zf0 + (float)zz;
                        const float2 zf = make_float2(za, second ? za + 1.f : za);
                        const float2 ix = __ffma2_rn(f2(sz[0]), zf, f2(pxy[0]));
                        const float2 iy = __ffma2_rn(f2(sz[1]), zf, f2(pxy[1]));
                        const float2 iz = __ffma2_rn(f2(sz[2]), zf, f2(pxy[2]));
                        const float2 t = make_float2(lds_f_dyn(tg + zz * (TX * TY * 4)),
                                                     lds_f_dyn(tg + (second ? zz + 1 : zz) * (TX * TY * 4)));
                        const float2 wv = second ? pair_step2<kBX, kBY, true, MSE_ONLY>(box_addr, Mrel, ix, iy, iz, t, zf, A)
                                                 : pair_step2<kBX, kBY, false, MSE_ONLY>(box_addr, Mrel, ix, iy, iz, t, zf, A);
                        if constexpr (STORE) {
                            const size_t HWs = (size_t)H * W;
                            float *wz = wcol0 + (size_t)(int)zf0 * HWs;
                            __stcs(wz + (size_t)zz * HWs, wv.x);
                            if (second) __stcs(wz + (size_t)(zz + 1) * HWs, wv.y);
                        }
                    }
                }
            } else if (ROT) {
                // gathers through L1; several z steps in flight per thread.  The unfused pass also leaves the warped samples
                // (default-loss loop: the NMI term needs them)
                float *wcol = (pp.moments_only && p.a.warped_out)
                                  ? p.a.warped_out + (size_t)(mov - p.a.moving) + ((size_t)(int)m.zf0 * H + y) * W + x : nullptr;
#pragma unroll 4
                for (int zz = 0; zz < nz; ++zz) {
                    const float zf = m.zf0 + (float)zz;
                    float wv;
                    if constexpr (PAIRS == 1)
                        wv = voxel_direct2p<MSE_ONLY>(reinterpret_cast<const float2 *>(pairs), D, H, W, fmaf(sz[0], zf, pxy[0]),
                                                      fmaf(sz[1], zf, pxy[1]), fmaf(sz[2], zf, pxy[2]), lds_f_dyn(tg + zz * (TX * TY * 4)), zf, A);
                    else if constexpr (PAIRS == 2)
                        wv = voxel_direct2q<MSE_ONLY>(reinterpret_cast<const float4 *>(pairs), D, H, W, fmaf(sz[0], zf, pxy[0]),
                                                      fmaf(sz[1], zf, pxy[1]), fmaf(sz[2], zf, pxy[2]), lds_f_dyn(tg + zz * (TX * TY * 4)), zf, A);
                    else
                        wv = voxel_direct2<MSE_ONLY>(mov, D, H, W, fmaf(sz[0], zf, pxy[0]), fmaf(sz[1], zf, pxy[1]), fmaf(sz[2], zf, pxy[2]),
                                                     lds_f_dyn(tg + zz * (TX * TY * 4)), zf, A);
                    if (wcol) __stcs(wcol + (size_t)zz * H * W, wv);
                }
            } else {
                for (int zz = 0; zz < nz; ++zz) {
                    const float zf = m.zf0 + (float)zz;
                    const float wv = voxel_direct2<MSE_ONLY>(mov, D, H, W, fmaf(sz[0], zf, pxy[0]), fmaf(sz[1], zf, pxy[1]),
                                                             fmaf(sz[2], zf, pxy[2]), lds_f_dyn(tg + zz * (TX * TY * 4)), zf, A);
                    if constexpr (STORE) __stcs(wcol0 + ((size_t)(int)m.zf0 + zz) * H * W, wv);
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty_bar + stage);
        if (m.flags & kEndCol) {
#ifdef TRB_TIMING
            const unsigned long long te0 = gtime();
#endif
            // fold the column's sums with this thread's base coordinates (x, y constant over the column), reduce over the
            // warp and leave the 41 totals in this warp's row for the reducer warp
            float acc[TRB_MOMENTS];
#pragma unroll
            for (int i = 0; i < TRB_MOMENTS; ++i) acc[i] = 0.f;
            if (valid) {
                // Acc2 layout (affine_tile.cuh): family f in {1, t, w, z, tz, wz} -> a[2f] = (k G0, k G1), a[2f+1] = (k G2, k w);
                // MSE only: families {d, d z} with (d G2, d^2) in a[1].  sum t / sum t^2 are not accumulated (target_sums_kernel).
                if (MSE_ONLY) {
                    acc[2] = A.a[1].y;                                  // sum d^2 rides in the sum t^2 slot
                    const float Pr[3] = {A.a[0].x, A.a[0].y, A.a[1].x}, Qr[3] = {A.a[2].x, A.a[2].y, A.a[3].x};
#pragma unroll
                    for (int r = 0; r < 3; ++r) {
                        const int bi = 5 + 2 * 12 + r * 4;              // the "w" family: the epilogue turns it into gm * sum d J
                        acc[bi + 0] = xv * Pr[r];
                        acc[bi + 1] = yv * Pr[r];
                        acc[bi + 2] = fmaf(inv_d2, Qr[r], zoff * Pr[r]);
                        acc[bi + 3] = Pr[r];
                    }
                } else {
                    acc[1] = A.a[1].y; acc[3] = A.a[5].y; acc[4] = A.a[3].y;
#pragma unroll
                    for (int kk = 0; kk < 3; ++kk) {
                        const float Pr[3] = {A.a[2 * kk].x, A.a[2 * kk].y, A.a[2 * kk + 1].x};
                        const float Qr[3] = {A.a[2 * (kk + 3)].x, A.a[2 * (kk + 3)].y, A.a[2 * (kk + 3) + 1].x};
#pragma unroll
                        for (int r = 0; r < 3; ++r) {
                            const int bi = 5 + kk * 12 + r * 4;
                            acc[bi + 0] = xv * Pr[r];
                            acc[bi + 1] = yv * Pr[r];
                            acc[bi + 2] = fmaf(inv_d2, Qr[r], zoff * Pr[r]);
                            acc[bi + 3] = Pr[r];
                        }
                    }
                }
            }
            const int cbuf = kcol & 1, use = kcol >> 1;
            if (use > 0) mbar_wait(red_empty + cbuf, (unsigned)(use - 1) & 1u);
            warp_reduce_moments2(acc, red + (cbuf * kConsumerWarps + warp) * kRedLdP, lane);
            __syncwarp();
            if (lane == 0) mbar_arrive(red_full + cbuf);
            ++kcol;
#ifdef TRB_TIMING
            if (lane == 0 && warp == 0) { g_pdbg[blockIdx.x * 32 + 10] += gtime() - te0; g_pdbg[blockIdx.x * 32 + 11] += 1ull; }
#endif
        }
    }
}

// ---- host side -----------------------------------------------------------------------------------------------------
// contributions (runs of tiles of one pair in a CTA's per-epoch stream) per pair, for the decomposition in `p`
static void count_contributions(const TmaParams &p, int G, std::vector<unsigned> &out, int &max_touched)
{
    out.assign((size_t)p.n_pairs, 0u);
    max_touched = 0;
    for (int b = 0; b < G; ++b) {
        int last = -1, touched = 0;
        auto visit = [&](long long col) {
            const int pair = (int)(col / p.cols_per_pair);
            if (pair != last) { ++out[(size_t)pair]; ++touched; last = pair; }
        };
        for (int r = 0; r < p.full_rounds; ++r) visit((long long)r * G + b);
        const long long t0 = p.tail_tiles * (long long)b / G, t1 = p.tail_tiles * (long long)(b + 1) / G;
        if (t1 > t0) {
            const long long c0 = (long long)p.full_rounds * G + t0 / p.tiles_z, c1 = (long long)p.full_rounds * G + (t1 - 1) / p.tiles_z;
            for (long long c = c0; c <= c1; ++c) visit(c);
        }
        if (touched > max_touched) max_touched = touched;
    }
}

static bool g_no_persist = false;
void set_no_persist(bool v) { g_no_persist = v; }
static thread_local char g_persist_status[256] = "never called";
#define PERSIST_REFUSE(...) do { snprintf(g_persist_status, sizeof(g_persist_status), __VA_ARGS__); return TRB_ERR_UNSUPPORTED; } while (0)

struct ContribBlock { static constexpr int kPairs = 256; unsigned v[kPairs]; };
__global__ void set_contributions_kernel(unsigned *tickets, int n, const ContribBlock b)
{
    if ((int)threadIdx.x < n) tickets[(size_t)threadIdx.x * kTicketStride + kTargetWord] = b.v[threadIdx.x];
}

// Enqueue n_epochs fused epochs for n_pairs pairs with the persistent kernel.  Returns TRB_ERR_UNSUPPORTED (without
// enqueuing anything) when the configuration does not fit it; the caller then takes the per-epoch kernel.
int launch_affine3d_persist(AffineParams a, int n_pairs, int epoch0, int n_epochs, cudaStream_t stream, int moments_mode)
{
    // moments_mode: 0 = fused epochs; 1 = one unfused pass (moments to a.moments_out); 2 = the same without target sums;
    // 3 = as 1, the target sums of an earlier mode-1 call on this workspace and these targets are still valid
    const bool moments_only = moments_mode != 0;
    if (moments_only) n_epochs = 1;
    if (g_no_persist || a.extra) PERSIST_REFUSE("disabled (kernel path / extra term)");
    if (a.peer.world > 1 && n_pairs != 1) PERSIST_REFUSE("peer exchange needs one pair");
    int dev = 0, sms = 0, coop = 0;
    if (int rc = sm_count(sms)) return rc;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev);
    if (!coop) PERSIST_REFUSE("no cooperative launch");
    const bool mse_only = !moments_only && a.w_ncc == 0.f;
    const bool rot = a.gather != 0;
    const bool store = moments_only && !rot && a.warped_out != nullptr;
    const bool pairs = rot && a.gather >= 2;
    auto kern = rot ? (a.gather == 3 ? (mse_only ? affine3d_persist_kernel<true, true, false, 2> : affine3d_persist_kernel<false, true, false, 2>)
                       : a.gather == 2 ? (mse_only ? affine3d_persist_kernel<true, true, false, 1> : affine3d_persist_kernel<false, true, false, 1>)
                                       : (mse_only ? affine3d_persist_kernel<true, true> : affine3d_persist_kernel<false, true>))
                    : (mse_only ? affine3d_persist_kernel<true, false>
                                : (store ? affine3d_persist_kernel<false, false, true> : affine3d_persist_kernel<false, false>));
    const size_t kPersistSmem = rot ? Ring<true>::kSmem : Ring<false>::kSmem;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPersistSmem);
    if (e != cudaSuccess) { cudaGetLastError(); PERSIST_REFUSE("cudaFuncSetAttribute(smem %zu): %s", kPersistSmem, cudaGetErrorString(e)); }
    int occ = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kPersistThreads, kPersistSmem);
    if (e != cudaSuccess || occ < 1) {
        cudaGetLastError();
        PERSIST_REFUSE("occupancy %d (%s)", occ, cudaGetErrorString(e));
    }
    const int tiles_x = (a.W + TX - 1) / TX, tiles_y = (a.H + TY - 1) / TY, tiles_z = (a.s_end - a.s_begin + TZ - 1) / TZ;
    const int cpp = tiles_x * tiles_y;
    // sub-batches: a CTA keeps a private copy of the optimiser state of every pair it touches (kStateSlots of them), so
    // a launch covers at most as many pairs as give every CTA <= kStateSlots - 2 whole columns; pairs are independent,
    // so the sub-batches simply run one after the other (each over all epochs)
    int sub = (int)(((long long)(kStateSlots - 2) * sms) / cpp);
    if (sub < 1) sub = 1;
    if (sub > n_pairs) sub = n_pairs;
    // accumulator region = the per-epoch kernels' partial-sum slots: chunk of epochs per launch
    const size_t region_words = (size_t)kMaxSlots * TRB_MOMENTS;          // 8-byte words per pair
    const int chunk_cap = (int)(region_words / kAccWords);
    static thread_local std::vector<unsigned> contrib;
    for (int p0 = 0; p0 < n_pairs; p0 += sub) {
        const int np = min(sub, n_pairs - p0);
        AffineParams as = a;
        as.moving = a.moving + (size_t)p0 * a.pair_stride;
        as.target = a.target + (size_t)p0 * a.pair_stride;
        as.state = a.state + (size_t)p0 * TRB_STATE_FLOATS;
        as.partials = a.partials + (size_t)p0 * region_words;
        as.tickets = a.tickets + (size_t)p0 * kTicketStride;
        if (a.loss_log) as.loss_log = a.loss_log + (size_t)p0 * a.log_stride;
        as.extra = nullptr;
        if (a.warped_out) as.warped_out = a.warped_out + (size_t)p0 * a.pair_stride;
        CUtensorMap map_mov, map_tgt;
        int rc = make_map(&map_mov, as.moving, np, as.pair_stride, as.D, as.H, as.W, kBX, kBY, kBZ);
        if (rc) return rc;
        rc = make_map(&map_tgt, as.target, np, as.pair_stride, as.D, as.H, as.W, TX, TY, TZ);
        if (rc) return rc;
        PersistParams pp;
        pp.t.a = as;
        pp.t.n_pairs = np;
        pp.t.tiles_x = tiles_x; pp.t.tiles_y = tiles_y; pp.t.tiles_z = tiles_z;
        pp.t.cols_per_pair = cpp;
        const long long total_cols = (long long)np * cpp;
        long long grid_ll = sms;
        if (grid_ll > total_cols * tiles_z) grid_ll = total_cols * tiles_z;
        const int grid = (int)grid_ll;
        pp.t.use_groups = 0;
        pp.t.full_rounds = (int)(total_cols / grid);
        pp.t.tail_tiles = (total_cols - (long long)pp.t.full_rounds * grid) * tiles_z;
        int max_touched = 0;
        count_contributions(pp.t, grid, contrib, max_touched);
        unsigned cmax = 0;
        for (unsigned c : contrib) cmax = c > cmax ? c : cmax;
        if (max_touched > kStateSlots || cmax >= (1u << kCountBits)) {
            if (p0 == 0) PERSIST_REFUSE("decomposition: %d pairs per CTA, %u contributions", max_touched, cmax);
            set_error("persistent kernel: inconsistent sub-batch decomposition");
            return TRB_ERR_ARG;
        }
        // contribution counts go up as kernel arguments: a pageable cudaMemcpyAsync would block the host until the work
        // already queued on the stream (e.g. the previous stage's epochs) has drained
        for (int c0 = 0; c0 < np; c0 += ContribBlock::kPairs) {
            ContribBlock cb{};
            const int n = min(ContribBlock::kPairs, np - c0);
            for (int i = 0; i < n; ++i) cb.v[i] = contrib[c0 + i];
            set_contributions_kernel<<<1, ContribBlock::kPairs, 0, stream>>>(as.tickets + (size_t)c0 * kTicketStride, n, cb);
        }
        pp.acc = reinterpret_cast<unsigned long long *>(as.partials);
        pp.pairs_slot = reinterpret_cast<const unsigned long long *>(a.tickets + kPairsWord);     // slot of the WHOLE batch
        pp.pair0 = p0;
        pp.targets = as.tickets;
        pp.tsum_blocks = (mse_only || moments_mode == 2) ? 0 : kTsumBlocks;
        pp.moments_only = moments_only ? 1 : 0;
        if (moments_only) pp.t.a.moments_out = a.moments_out + (size_t)p0 * TRB_MOMENTS;
        if (pp.tsum_blocks > 0 && moments_mode != 3) {
            e = cudaMemset2DAsync(as.tickets + kTsumWord, kTicketStride * sizeof(unsigned), 0, 2 * kLimbs * sizeof(unsigned long long), (size_t)np, stream);
            if (e != cudaSuccess) return check_cuda(e, "cudaMemset2DAsync(target sums)");
            const long long slab = (long long)as.H * as.W;
            target_sums_kernel<<<dim3(kTsumBlocks, np), 256, 0, stream>>>(as.target, as.pair_stride, (long long)as.s_begin * slab,
                                                                        (long long)(as.s_end - as.s_begin) * slab, as.tickets);
        }
        for (int done = 0; done < n_epochs;) {
            const int ne = min(chunk_cap, n_epochs - done);
            pp.n_epochs = ne;
            pp.t.a.epoch = epoch0 + done;
            pp.t.a.peer.seq = a.peer.seq + (unsigned long long)done;
            e = cudaMemsetAsync(pp.acc, 0, (size_t)ne * np * kAccWords * sizeof(unsigned long long), stream);
            if (e != cudaSuccess) return check_cuda(e, "cudaMemsetAsync(accumulators)");
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(grid); cfg.blockDim = dim3(kPersistThreads); cfg.dynamicSmemBytes = kPersistSmem; cfg.stream = stream;
            cudaLaunchAttribute attr[1];
            attr[0].id = cudaLaunchAttributeCooperative;
            attr[0].val.cooperative = 1;
            cfg.attrs = attr; cfg.numAttrs = 1;
            e = cudaLaunchKernelEx(&cfg, kern, pp, map_mov, map_tgt);
            if (e != cudaSuccess) return check_cuda(e, "cudaLaunchKernelEx(affine3d_persist)");
            done += ne;
        }
    }
    snprintf(g_persist_status, sizeof(g_persist_status), "launched: grid %d, %d SMs, %s variant, sub-batches of %d pair(s)",
             (int)(sms < (long long)n_pairs * cpp * tiles_z ? sms : (long long)n_pairs * cpp * tiles_z), sms, rot ? (a.gather == 3 ? "gather (quad volume)" : pairs ? "gather (pair volume)" : "gather") : "tma", sub);
    return check_cuda(cudaGetLastError(), "affine3d_persist");
}
const char *persist_status() { return g_persist_status; }

}  // namespace trb
#ifdef TRB_TIMING
extern "C" int trb_pdebug_read(unsigned long long *out, int n) { return (int)cudaMemcpyFromSymbol(out, trb::g_pdbg, sizeof(unsigned long long) * n); }
extern "C" int trb_pdebug_clear() { static unsigned long long z[1024 * 32]; return (int)cudaMemcpyToSymbol(trb::g_pdbg, z, sizeof(z)); }
#endif
