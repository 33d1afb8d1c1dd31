// affine_shared.cuh — pieces shared by the direct (affine.cu) and TMA-staged (affine_tma.cu)
// rigid/affine kernels: parameters, Theta parametrisation + chain rule, the per-pair epilogue
// (loss, d theta, optimiser step, best tracking) and the CTA -> grid reduction that feeds it.
#pragma once
#include "common.cuh"
#include <math.h>

#include "peer.cuh"

namespace trb {

constexpr int kTicketStride = 128;  // unsigned counters per pair in the workspace (direct kernel uses [127])
constexpr int kPairsWord = 120;     // tickets[120..121] of pair 0: address of the pair volume (trb_affine_attach_pairs) or 0
constexpr int kMaxSlots = 1024;      // partial-sum slots per pair in the workspace (>= CTAs contributing to a pair)

struct AffineParams;
bool tma_path_eligible(int ndim, const AffineParams &a, int n_pairs);
int launch_affine3d_tma(AffineParams a, int n_pairs, bool fused, int epoch0, int n_launch, cudaStream_t stream);
// moments of slices [s_begin, s_end) for all pairs (trb_affine_moments_ex); warped_out (optional, 3-D): the warped volumes
// as a by-product when a TMA-tile kernel takes the pass — *wrote_warped says whether it did; target_sums: 0 not needed,
// 1 compute, 3 compute and keep, 2 still valid from an earlier call with 3 on the same workspace and targets
int affine_moments_impl(int ndim, const float *moving_dev, const float *target_dev, long long pair_stride, int n_pairs, int D, int H,
                        int W, int s_begin, int s_end, const float *xb_dev, const float *yb_dev, const float *zb_dev,
                        const float *state_dev, double *moments_dev, int flags, int target_sums, float *warped_out,
                        bool *wrote_warped, void *workspace_dev, size_t workspace_bytes, void *stream);
// persistent multi-epoch kernel (affine_persist.cu); TRB_ERR_UNSUPPORTED = nothing enqueued, take the per-epoch kernel
int launch_affine3d_persist(AffineParams a, int n_pairs, int epoch0, int n_epochs, cudaStream_t stream, int moments_mode = 0);
void set_no_persist(bool v);
const char *persist_status();
// TMA-staged forward warp (warp_tma.cu)
bool warp_tma_eligible(const float *moving, const float *out, int n_items, long long vol, int D, int H, int W);
int launch_warp_affine_tma(const float *moving, float *out, int n_pairs, int n_channels, int D, int H, int W,
                           const float *theta_dev, const float *xb, const float *yb, bool nearest, cudaStream_t stream);

struct AffineParams {
    const float *moving, *target;
    long long pair_stride;
    int D, H, W;
    int s_begin, s_end;          // slab of output slices (z for 3-D, y for 2-D)
    const float *xb, *yb, *zb;   // base coordinates per axis
    float *state;                // [n_pairs][TRB_STATE_FLOATS]
    double *partials;            // [n_pairs][gridDim.x][TRB_MOMENTS]
    unsigned *tickets;           // [n_pairs]
    double *moments_out;         // unfused: [n_pairs][TRB_MOMENTS]
    float *loss_log;
    int log_stride, epoch;
    float w_mse, w_ncc, lr;
    int mode, optimiser;
    float beta1, beta2, adam_eps;
    float *warped_out;           // optional [n_pairs][D][H][W]: the unfused 3-D TMA moments pass also stores the warped volume
    const double *extra;         // optional [n_pairs][13]: extra loss term and its d/dtheta (e.g. the NMI term), or NULL
    int extra_pair;              // row of `extra` (set by the epilogue wrappers)
    int gather;                  // 1: large-rotation variant of the persistent kernel (L1 gathers instead of TMA-staged boxes);
                                 // 2: the same, reading the pair volume attached to the workspace
    PeerExchange peer;
};

// ---- Theta.forward (utils.py:287-310), fp32 like the reference ------------------
template <int NDIM>
__device__ void rigid_theta(const float *p, float *th)
{
    if (NDIM == 3) {
        float sps, cps, sth, cth, sph, cph;
        sincosf(p[0], &sps, &cps);
        sincosf(p[1], &sth, &cth);
        sincosf(p[2], &sph, &cph);
        th[0] = cps * cth;  th[1] = sph * sps * cth - cph * sth;  th[2] = cph * sps * cth + sph * sth;
        th[3] = 0.25f * tanhf(p[3]);
        th[4] = cps * sth;  th[5] = sph * sps * sth + cph * cth;  th[6] = cph * sps * sth - sph * cth;
        th[7] = 0.25f * tanhf(p[4]);
        th[8] = -sps;       th[9] = sph * cps;                     th[10] = cph * cps;
        th[11] = 0.25f * tanhf(p[5]);
    } else {
        float s, c;
        sincosf(p[0], &s, &c);
        th[0] = c; th[1] = -s; th[2] = p[1];
        th[3] = s; th[4] = c;  th[5] = p[2];
    }
}

// Jacobian-transpose product d theta -> d params of the map above.
template <int NDIM>
__device__ void rigid_chain(const float *p, const double *g, double *dp)
{
    if (NDIM == 3) {
        double sps, cps, sth, cth, sph, cph;
        sincos((double)p[0], &sps, &cps);
        sincos((double)p[1], &sth, &cth);
        sincos((double)p[2], &sph, &cph);
        dp[0] = g[0] * (-sps * cth) + g[1] * (sph * cps * cth) + g[2] * (cph * cps * cth)
              + g[4] * (-sps * sth) + g[5] * (sph * cps * sth) + g[6] * (cph * cps * sth)
              - g[8] * cps - g[9] * (sph * sps) - g[10] * (cph * sps);
        dp[1] = -g[0] * (cps * sth) - g[1] * (sph * sps * sth + cph * cth) + g[2] * (sph * cth - cph * sps * sth)
              + g[4] * (cps * cth) + g[5] * (sph * sps * cth - cph * sth) + g[6] * (cph * sps * cth + sph * sth);
        dp[2] = g[1] * (cph * sps * cth + sph * sth) + g[2] * (cph * sth - sph * sps * cth)
              + g[5] * (cph * sps * sth - sph * cth) - g[6] * (sph * sps * sth + cph * cth)
              + g[9] * (cph * cps) - g[10] * (sph * cps);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            double t = tanh((double)p[3 + k]);
            dp[3 + k] = g[3 + 4 * k] * 0.25 * (1.0 - t * t);
        }
    } else {
        double s, c;
        sincos((double)p[0], &s, &c);
        dp[0] = -g[0] * s - g[1] * c + g[3] * c - g[4] * s;
        dp[1] = g[2];
        dp[2] = g[5];
    }
}

// ---- epilogue: moments -> loss, d theta, chain, optimiser step, bookkeeping ---------
// Runs in ONE thread per pair (O(100) flops).  M holds the TRB_MOMENTS sums with the
// UN-scaled interpolant derivative; the grid_sample un-normalisation factor S_r/2 is
// applied here.
// `st` is the pair's TRB_STATE_FLOATS block: in global memory (LOCAL = false; __ldcg loads: another CTA wrote it in the
// previous epoch) or a private copy in shared memory (LOCAL = true; the persistent kernel keeps one per CTA and pair).
// Returns the loss of the pre-step theta; *improved says whether this epoch became the best so far.
template <int NDIM, bool LOCAL>
__device__ float affine_epilogue_core(const double *M, const AffineParams &p, int epoch, float *st, bool *improved)
{
    constexpr int NC = NDIM + 1, NT = NDIM * NC;
    auto ld = [&](int i) -> float { return LOCAL ? st[i] : __ldcg(st + i); };
    // read everything first (independent loads, one round trip), compute, then write
    float par[12], th_cur[12], am[12], av[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) { par[i] = ld(TRB_STATE_PARAMS + i); th_cur[i] = ld(TRB_STATE_THETA + i); }
    const float best_prev = ld(TRB_STATE_BEST_LOSS);
    if (p.optimiser != TRB_OPT_SGD) {
#pragma unroll
        for (int i = 0; i < 12; ++i) { am[i] = ld(TRB_STATE_ADAM_M + i); av[i] = ld(TRB_STATE_ADAM_V + i); }
    }
    const double n = (double)(NDIM == 3 ? p.D : 1) * (double)p.H * (double)p.W;
    const LossCoef lc = loss_coefficients(n, M[0], M[1], M[2], M[3], M[4], (double)p.w_mse, (double)p.w_ncc);
    const double scale[3] = {0.5 * p.W, 0.5 * p.H, 0.5 * p.D};
    double dth[12];
#pragma unroll
    for (int r = 0; r < NDIM; ++r)
#pragma unroll
        for (int c = 0; c < NC; ++c) {
            const int i = r * NC + c;
            dth[i] = (lc.cw * M[29 + i] + lc.ct * M[17 + i] + lc.c0 * M[5 + i]) * scale[r];
        }
    double loss_d = lc.loss;
    if (p.extra) {                                  // externally evaluated term (already in theta units)
        const double *ex = p.extra + (size_t)(p.extra_pair) * 13;
        loss_d += ex[0];
#pragma unroll
        for (int i = 0; i < NT; ++i) dth[i] += ex[1 + i];
    }
    const float loss = (float)loss_d;
    // best tracking on the pre-step theta (warpings.py:85-93,151-159: strictly lower)
    *improved = (epoch == 0 || loss < best_prev);
    if (*improved) {
        st[TRB_STATE_BEST_LOSS] = loss;
#pragma unroll
        for (int i = 0; i < NT; ++i) st[TRB_STATE_BEST_THETA + i] = th_cur[i];
    }
    st[TRB_STATE_LAST_LOSS] = loss;

    double dp[12];
    int np;
    if (p.mode == TRB_MODE_RIGID) {
        rigid_chain<NDIM>(par, dth, dp);
        np = NDIM == 3 ? 6 : 3;
    } else {
#pragma unroll
        for (int i = 0; i < NT; ++i) dp[i] = dth[i];
        np = NT;
    }
#pragma unroll
    for (int i = 0; i < 12; ++i) {
        if (i < np) {
            const float g = (float)dp[i];
            float v = par[i];
            if (p.optimiser == TRB_OPT_SGD) {
                v = v - p.lr * g;                      // torch.optim.SGD, no momentum / decay
            } else {                                   // torch.optim.Adam semantics (extension)
                const float t = (float)(epoch + 1);
                float m = am[i], s = av[i];
                m = p.beta1 * m + (1.f - p.beta1) * g;
                s = p.beta2 * s + (1.f - p.beta2) * g * g;
                st[TRB_STATE_ADAM_M + i] = m;
                st[TRB_STATE_ADAM_V + i] = s;
                const float bc1 = 1.f - powf(p.beta1, t), bc2 = 1.f - powf(p.beta2, t);
                v = v - (p.lr / bc1) * (m / (sqrtf(s) / sqrtf(bc2) + p.adam_eps));
            }
            par[i] = v;
            st[TRB_STATE_PARAMS + i] = v;
        }
    }
    if (p.mode == TRB_MODE_RIGID) {
        float th[12];
        rigid_theta<NDIM>(par, th);
#pragma unroll
        for (int i = 0; i < NT; ++i) st[TRB_STATE_THETA + i] = th[i];
    } else {
#pragma unroll
        for (int i = 0; i < NT; ++i) st[TRB_STATE_THETA + i] = par[i];
    }
    return loss;
}

template <int NDIM>
__device__ void affine_epilogue(const double *M, AffineParams p, int pair)
{
    bool improved;
    p.extra_pair = pair;
    const float loss = affine_epilogue_core<NDIM, false>(M, p, p.epoch, p.state + (size_t)pair * TRB_STATE_FLOATS, &improved);
    if (p.loss_log) p.loss_log[(size_t)pair * p.log_stride + p.epoch] = loss;
}

// second half of the CTA reduction: `red` holds one row of TRB_MOMENTS warp totals per warp
// (row stride `ld` floats).  Must be called by all NWARPS*32 threads of the CTA after a barrier.
template <int NDIM, bool FUSED, int NWARPS>
__device__ void finish_from_warp_sums(const float *red, int ld, const AffineParams &p, int pair, int slot, int n_slots,
                                      int first_slot, int count, int tid)
{
    constexpr int kSlices = NWARPS * 32 / 64;
    __shared__ double fin[kSlices][TRB_MOMENTS + 1];
    __shared__ int is_last;
    if (tid < TRB_MOMENTS) {
        double s = 0.0;
#pragma unroll
        for (int w = 0; w < NWARPS; ++w) s += (double)red[w * ld + tid];
        __stcg(p.partials + ((size_t)pair * n_slots + slot) * TRB_MOMENTS + tid, s);
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) {
        const unsigned t = atomicAdd(p.tickets + (size_t)pair * kTicketStride + 127, 1u);
        is_last = (t == (unsigned)count - 1u) ? 1 : 0;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    {
        const int v = tid & 63, slice = tid >> 6;
        if (v < TRB_MOMENTS) {
            double *src = p.partials + (size_t)pair * n_slots * TRB_MOMENTS + v;
            double a = 0.0;
            for (int j = slice; j < count; j += kSlices) {
                int sl = first_slot + j;
                if (sl >= n_slots) sl -= n_slots;
                a += __ldcg(src + (size_t)sl * TRB_MOMENTS);
                __stcg(src + (size_t)sl * TRB_MOMENTS, 0.0);      // leave the workspace zeroed (the TMA kernel relies on it)
            }
            fin[slice][v] = a;
        }
    }
    __syncthreads();
    if (tid < TRB_MOMENTS) {
        double a = 0.0;
#pragma unroll
        for (int sidx = 0; sidx < kSlices; ++sidx) a += fin[sidx][tid];
        fin[0][tid] = a;
    }
    __syncthreads();
    if (FUSED) {
        if (tid == 0) {
            affine_epilogue<NDIM>(fin[0], p, pair);
            p.tickets[(size_t)pair * kTicketStride + 127] = 0u;
        }
    } else {
        if (tid < TRB_MOMENTS) p.moments_out[(size_t)pair * TRB_MOMENTS + tid] = fin[0][tid];
        if (tid == 0) p.tickets[(size_t)pair * kTicketStride + 127] = 0u;
    }
}

template <int NDIM, bool FUSED, int NWARPS>
__device__ void reduce_and_finish(float (&acc)[TRB_MOMENTS], const AffineParams &p, int pair, int slot, int n_slots,
                                  int first_slot, int count, int tid)
{
    __shared__ float red[NWARPS][TRB_MOMENTS + 1];
    const int lane = tid & 31, warp = tid >> 5;
    __syncthreads();               // previous use of the scratch is over
#pragma unroll
    for (int i = 0; i < TRB_MOMENTS; ++i) {
        const float v = warp_sum(acc[i]);
        if (lane == 0) red[warp][i] = v;
    }
    __syncthreads();
    finish_from_warp_sums<NDIM, FUSED, NWARPS>(&red[0][0], TRB_MOMENTS + 1, p, pair, slot, n_slots, first_slot, count, tid);
}

}  // namespace trb
