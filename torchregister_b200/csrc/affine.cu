// affine.cu — fused rigid/affine registration epoch for B200 (sm_100a).
//
// One launch per epoch.  Per pair of volumes it replaces, from the reference
// (paths relative to /root/reference/src/TorchRegister/):
//   F.affine_grid + F.grid_sample (align_corners=False, zeros)   warpings.py:24-25
//   nn.MSELoss / NCCLoss.forward                                  warpings.py:37,124; utils.py:197-205
//   error.backward() down to theta and to Regressor.reg           warpings.py:80,146; utils.py:287-310
//   torch.optim.SGD.step, best-theta tracking, loss log           warpings.py:81-93,147-159
// No sampling grid is materialised: coordinates are rebuilt from theta and three
// per-axis base-coordinate tables; the warped volume is never written.
//
// Data layout: moving/target fp32 [D][H][W] per pair (x = W fastest).  A warp owns
// one output row (fixed z,y), lanes run along x, so target loads are fully coalesced
// and the 8 gathered corners of neighbouring lanes fall in the same 128-B lines for
// near-identity transforms.  Algorithmic traffic: 8 B per voxel-warp (moving 4 +
// target 4), everything else is O(1) per pair.
#include "common.cuh"
#include "affine_shared.cuh"
#include "affine_tile.cuh"
#include <math.h>

namespace trb {

// ---- the fused pass ------------------------------------------------------------------
template <int NDIM, bool FUSED>
__global__ void __launch_bounds__(kThreads, 2) affine_moments_kernel(const AffineParams p)
{
    constexpr int NC = NDIM + 1, NT = NDIM * NC;
    const int pair = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float *__restrict__ mov = p.moving + (size_t)pair * p.pair_stride;
    const float *__restrict__ tgt = p.target + (size_t)pair * p.pair_stride;
    const int W = p.W, H = p.H, D = (NDIM == 3 ? p.D : 1);
    const size_t HW = (size_t)H * W;

    float th[NT];
    {
        const float *st = p.state + (size_t)pair * TRB_STATE_FLOATS + TRB_STATE_THETA;
#pragma unroll
        for (int i = 0; i < NT; ++i) th[i] = __ldcg(st + i);
    }
    const float hw = 0.5f * W, hh = 0.5f * H, hd = 0.5f * D;
    const bool mse_only = FUSED && p.w_ncc == 0.f;
    // i_r(x) = a_r * xb[x] + b_r(row): affine_grid, then ((g+1)*S-1)/2 folded in
    const float ax = th[0] * hw, ay = th[NC] * hh, az = NDIM == 3 ? th[2 * NC] * hd : 0.f;

    // accumulators (k: 0 -> weight 1, 1 -> t, 2 -> w ; r: sampling coordinate)
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f, s4 = 0.f;
    float Q[3][NDIM], T1[3][NDIM], Ty[3][NDIM], Tz[3][NDIM];
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int r = 0; r < NDIM; ++r) Q[k][r] = T1[k][r] = Ty[k][r] = Tz[k][r] = 0.f;

    const int rows = (p.s_end - p.s_begin) * (NDIM == 3 ? H : 1);
    for (int row0 = blockIdx.x * kWarps; row0 < rows; row0 += gridDim.x * kWarps) {
        const int row = row0 + warp;
        if (row >= rows) break;
        int z = 0, y;
        if (NDIM == 3) { z = p.s_begin + row / H; y = row - (row / H) * H; }
        else y = p.s_begin + row;
        const float yv = __ldg(p.yb + y);
        const float zv = NDIM == 3 ? __ldg(p.zb + z) : 0.f;
        float bx, by, bz = 0.f;
        if (NDIM == 3) {
            bx = fmaf(th[1] * yv + th[2] * zv + th[3] + 1.f, hw, -0.5f);
            by = fmaf(th[5] * yv + th[6] * zv + th[7] + 1.f, hh, -0.5f);
            bz = fmaf(th[9] * yv + th[10] * zv + th[11] + 1.f, hd, -0.5f);
        } else {
            bx = fmaf(th[1] * yv + th[2] + 1.f, hw, -0.5f);
            by = fmaf(th[4] * yv + th[5] + 1.f, hh, -0.5f);
        }
        const float *__restrict__ trow = tgt + ((size_t)z * H + y) * W;
        float P[3][NDIM];
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int r = 0; r < NDIM; ++r) P[k][r] = 0.f;

        for (int xs = 0; xs < W; xs += 32) {
            const int xi = xs + lane;
            const bool act = xi < W;
            const int xc = act ? xi : W - 1;
            const float xv = __ldg(p.xb + xc);
            const float t = act ? ld_stream_f(trow + xc) : 0.f;
            const float ix = fmaf(ax, xv, bx), iy = fmaf(ay, xv, by);
            const float fx = floorf(ix), fy = floorf(iy);
            const float tx = ix - fx, ty = iy - fy;
            const int x0 = (int)fx, y0 = (int)fy;
            Sample<NDIM> s;
            if constexpr (NDIM == 3) {
                const float iz = fmaf(az, xv, bz);
                const float fz = floorf(iz);
                const float tz = iz - fz;
                const int z0 = (int)fz;
                const bool inb = (x0 >= 0) & (x0 < W - 1) & (y0 >= 0) & (y0 < H - 1) & (z0 >= 0) & (z0 < D - 1);
                // named corners rather than k.c filled in both branches: the array would renumber the PTX registers, and
                // ptxas would schedule this loop differently
                float c000, c001, c010, c011, c100, c101, c110, c111;
                if (__all_sync(kFull, inb)) {
                    const float *q = mov + ((size_t)z0 * H + y0) * W + x0;
                    c000 = __ldg(q);          c001 = __ldg(q + 1);
                    c010 = __ldg(q + W);      c011 = __ldg(q + W + 1);
                    c100 = __ldg(q + HW);     c101 = __ldg(q + HW + 1);
                    c110 = __ldg(q + HW + W); c111 = __ldg(q + HW + W + 1);
                } else {
                    float b[8];
                    load_cell3(mov, D, H, W, x0, y0, z0, b);
                    c000 = b[0]; c001 = b[1]; c010 = b[2]; c011 = b[3]; c100 = b[4]; c101 = b[5]; c110 = b[6]; c111 = b[7];
                }
                s = blend_cell3<true>(Cell3{{c000, c001, c010, c011, c100, c101, c110, c111}, tx, ty, tz});
            } else {
                const bool inb = (x0 >= 0) & (x0 < W - 1) & (y0 >= 0) & (y0 < H - 1);
                float c00, c01, c10, c11;
                if (__all_sync(kFull, inb)) {
                    const float *q = mov + (size_t)y0 * W + x0;
                    c00 = __ldg(q); c01 = __ldg(q + 1); c10 = __ldg(q + W); c11 = __ldg(q + W + 1);
                } else {
                    float b[4];
                    load_cell2(mov, H, W, x0, y0, b);
                    c00 = b[0]; c01 = b[1]; c10 = b[2]; c11 = b[3];
                }
                s = blend_cell2<true>(Cell2{{c00, c01, c10, c11}, tx, ty});
            }
            float val = s.val;
            const float *G = s.g;
            if (act) {
                // w_ncc == 0 (the reference's "criterion given -> MSE" branch): accumulate d = w - t instead of t and w.
                // MSE = sum d^2 / n then needs no (sum t^2 - 2 sum t w + sum w^2) cancellation, which costs 3 digits once
                // the images agree to 1e-3 (500-epoch golden); the epilogue sees (t, w) = (0, d): loss and gradient are
                // the same expressions.
                const float tt = mse_only ? 0.f : t;
                if (mse_only) val -= t;
                const float t = tt;
                s0 += t; s1 += val;
                s2 = fmaf(t, t, s2); s3 = fmaf(val, val, s3); s4 = fmaf(t, val, s4);
#pragma unroll
                for (int r = 0; r < NDIM; ++r) {
                    const float g = G[r], tg = t * g, wg = val * g;
                    P[0][r] += g;  P[1][r] += tg;  P[2][r] += wg;
                    Q[0][r] = fmaf(g, xv, Q[0][r]);
                    Q[1][r] = fmaf(tg, xv, Q[1][r]);
                    Q[2][r] = fmaf(wg, xv, Q[2][r]);
                }
            }
        }
        // y and z are constant along the row: fold the row partials once
#pragma unroll
        for (int k = 0; k < 3; ++k)
#pragma unroll
            for (int r = 0; r < NDIM; ++r) {
                T1[k][r] += P[k][r];
                Ty[k][r] = fmaf(yv, P[k][r], Ty[k][r]);
                if (NDIM == 3) Tz[k][r] = fmaf(zv, P[k][r], Tz[k][r]);
            }
    }

    // ---- CTA reduction + last-CTA epilogue ---------------------------------------------------
    float acc[TRB_MOMENTS];
    acc[0] = s0; acc[1] = s1; acc[2] = s2; acc[3] = s3; acc[4] = s4;
#pragma unroll
    for (int i = 5; i < TRB_MOMENTS; ++i) acc[i] = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
        for (int r = 0; r < NDIM; ++r) {
            const int b = 5 + k * 12 + r * NC;
            acc[b + 0] = Q[k][r];
            acc[b + 1] = Ty[k][r];
            if (NDIM == 3) acc[b + 2] = Tz[k][r];
            acc[b + NDIM] = T1[k][r];
        }
    reduce_and_finish<NDIM, FUSED, kWarps>(acc, p, pair, blockIdx.x, gridDim.x, 0, gridDim.x, threadIdx.x);
}

template <int NDIM>
__global__ void affine_apply_kernel(const AffineParams p, const double *moments)
{
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair < (int)p.pair_stride) affine_epilogue<NDIM>(moments + (size_t)pair * TRB_MOMENTS, p, pair);
}

template <int NDIM>
__global__ void affine_init_state_kernel(float *state, int n_pairs, int mode)
{
    constexpr int NT = NDIM * (NDIM + 1);
    const int pair = blockIdx.x * blockDim.x + threadIdx.x;
    if (pair >= n_pairs) return;
    float *st = state + (size_t)pair * TRB_STATE_FLOATS;
    float th[12];
    if (mode == TRB_MODE_RIGID) rigid_theta<NDIM>(st + TRB_STATE_PARAMS, th);
    else
        for (int i = 0; i < NT; ++i) th[i] = st[TRB_STATE_PARAMS + i];
    for (int i = 0; i < NT; ++i) { st[TRB_STATE_THETA + i] = th[i]; st[TRB_STATE_BEST_THETA + i] = th[i]; }
    st[TRB_STATE_BEST_LOSS] = 0.f;
    st[TRB_STATE_LAST_LOSS] = 0.f;
    for (int i = 0; i < 12; ++i) { st[TRB_STATE_ADAM_M + i] = 0.f; st[TRB_STATE_ADAM_V + i] = 0.f; }
}

// ---- forward-only warp (get_affine_warp, warpings.py:18-26) ------------------------------
// NEAREST: grid_sample(mode='nearest'): the source coordinate rounded half to even, one predicated load per channel
template <int NDIM, bool NEAREST>
__device__ __forceinline__ void warp_affine_body(const float *__restrict__ moving, float *__restrict__ out,
                                                 int n_channels, int D, int H, int W,
                                                 const float *__restrict__ theta,
                                                 const float *__restrict__ xb, const float *__restrict__ yb,
                                                 const float *__restrict__ zb)
{
    constexpr int NC = NDIM + 1, NT = NDIM * NC;
    const size_t HW = (size_t)H * W, vol = HW * (NDIM == 3 ? D : 1);
    // blockIdx.y: pair of a batch (its own theta, its own n_channels volumes)
    theta += (size_t)blockIdx.y * NT;
    moving += (size_t)blockIdx.y * n_channels * vol;
    out += (size_t)blockIdx.y * n_channels * vol;
    float th[NT];
#pragma unroll
    for (int i = 0; i < NT; ++i) th[i] = __ldg(theta + i);
    const float hw = 0.5f * W, hh = 0.5f * H, hd = 0.5f * D;
    for_each_voxel<2>(NDIM == 3 ? D : 1, H, W, [&](size_t idx, int x, int y, int z) {
        const float xv = __ldg(xb + x), yv = __ldg(yb + y);
        if (NDIM == 3) {
            const float zv = __ldg(zb + z);
            const float ix = fmaf(th[0] * hw, xv, fmaf(th[1] * yv + th[2] * zv + th[3] + 1.f, hw, -0.5f));
            const float iy = fmaf(th[4] * hh, xv, fmaf(th[5] * yv + th[6] * zv + th[7] + 1.f, hh, -0.5f));
            const float iz = fmaf(th[8] * hd, xv, fmaf(th[9] * yv + th[10] * zv + th[11] + 1.f, hd, -0.5f));
            if constexpr (NEAREST) {
                long long o;
                const bool v = nearest_offset(D, H, W, ix, iy, iz, o);
                for (int c = 0; c < n_channels; ++c) out[(size_t)c * vol + idx] = v ? __ldg(moving + (size_t)c * vol + o) : 0.f;
                return;
            }
            const float fx = floorf(ix), fy = floorf(iy), fz = floorf(iz);
            Cell3 k;
            k.tx = ix - fx; k.ty = iy - fy; k.tz = iz - fz;
            const int x0 = (int)fx, y0 = (int)fy, z0 = (int)fz;
            // load_cell3's predicates and offset, hoisted out of the channel loop by hand: calling load_cell3 per channel
            // made the 2-channel 256^3 warp 5 % slower (B200, 1000 W: 234 against 223 us)
            const bool vx0 = (unsigned)x0 < (unsigned)W, vx1 = (unsigned)(x0 + 1) < (unsigned)W;
            const bool vy0 = (unsigned)y0 < (unsigned)H, vy1 = (unsigned)(y0 + 1) < (unsigned)H;
            const bool vz0 = (unsigned)z0 < (unsigned)D, vz1 = (unsigned)(z0 + 1) < (unsigned)D;
            const long long o = ((long long)z0 * H + y0) * W + x0;
            for (int c = 0; c < n_channels; ++c) {
                const float *m = moving + (size_t)c * vol;
                k.c[0] = (vz0 & vy0 & vx0) ? __ldg(m + o) : 0.f;
                k.c[1] = (vz0 & vy0 & vx1) ? __ldg(m + o + 1) : 0.f;
                k.c[2] = (vz0 & vy1 & vx0) ? __ldg(m + o + W) : 0.f;
                k.c[3] = (vz0 & vy1 & vx1) ? __ldg(m + o + W + 1) : 0.f;
                k.c[4] = (vz1 & vy0 & vx0) ? __ldg(m + o + (long long)HW) : 0.f;
                k.c[5] = (vz1 & vy0 & vx1) ? __ldg(m + o + (long long)HW + 1) : 0.f;
                k.c[6] = (vz1 & vy1 & vx0) ? __ldg(m + o + (long long)HW + W) : 0.f;
                k.c[7] = (vz1 & vy1 & vx1) ? __ldg(m + o + (long long)HW + W + 1) : 0.f;
                out[(size_t)c * vol + idx] = blend_cell3<false>(k).val;
            }
        } else {
            const float ix = fmaf(th[0] * hw, xv, fmaf(th[1] * yv + th[2] + 1.f, hw, -0.5f));
            const float iy = fmaf(th[3] * hh, xv, fmaf(th[4] * yv + th[5] + 1.f, hh, -0.5f));
            if constexpr (NEAREST) {
                long long o;
                const bool v = nearest_offset(1, H, W, ix, iy, 0.f, o);
                for (int c = 0; c < n_channels; ++c) out[(size_t)c * vol + idx] = v ? __ldg(moving + (size_t)c * vol + o) : 0.f;
                return;
            }
            const float fx = floorf(ix), fy = floorf(iy);
            Cell2 k;
            k.tx = ix - fx; k.ty = iy - fy;
            const int x0 = (int)fx, y0 = (int)fy;
            // load_cell2's flags and offset, hoisted out of the channel loop by hand as in the 3-D branch
            const bool vx0 = (unsigned)x0 < (unsigned)W, vx1 = (unsigned)(x0 + 1) < (unsigned)W;
            const bool vy0 = (unsigned)y0 < (unsigned)H, vy1 = (unsigned)(y0 + 1) < (unsigned)H;
            const long long o = (long long)y0 * W + x0;
            for (int c = 0; c < n_channels; ++c) {
                const float *m = moving + (size_t)c * vol;
                k.c[0] = (vy0 & vx0) ? __ldg(m + o) : 0.f;
                k.c[1] = (vy0 & vx1) ? __ldg(m + o + 1) : 0.f;
                k.c[2] = (vy1 & vx0) ? __ldg(m + o + W) : 0.f;
                k.c[3] = (vy1 & vx1) ? __ldg(m + o + W + 1) : 0.f;
                out[(size_t)c * vol + idx] = blend_cell2<false>(k).val;
            }
        }
    });
}
template <int NDIM>
__global__ void __launch_bounds__(256) warp_affine_kernel(const float *__restrict__ moving, float *__restrict__ out,
                                                           int n_channels, int D, int H, int W,
                                                           const float *__restrict__ theta,
                                                           const float *__restrict__ xb, const float *__restrict__ yb,
                                                           const float *__restrict__ zb)
{
    warp_affine_body<NDIM, false>(moving, out, n_channels, D, H, W, theta, xb, yb, zb);
}
template <int NDIM>
__global__ void __launch_bounds__(256) warp_affine_nearest_kernel(const float *__restrict__ moving, float *__restrict__ out,
                                                                   int n_channels, int D, int H, int W,
                                                                   const float *__restrict__ theta,
                                                                   const float *__restrict__ xb, const float *__restrict__ yb,
                                                                   const float *__restrict__ zb)
{
    warp_affine_body<NDIM, true>(moving, out, n_channels, D, H, W, theta, xb, yb, zb);
}

__global__ void vjp_extract_kernel(const double *moments, double *dtheta, int ndim, int D, int H, int W)
{
    const int i = threadIdx.x;
    const int nc = ndim + 1;
    if (i >= ndim * nc) return;
    const int r = i / nc;
    const double scale = r == 0 ? 0.5 * W : (r == 1 ? 0.5 * H : 0.5 * D);
    dtheta[i] = moments[17 + i] * scale;      // sum_v gout_v * J_v (gout rides in the "target" slot)
}

// start parameters handed over as kernel ARGUMENTS: an upload that neither needs pinned memory nor blocks the host behind
// the work already queued on the stream (a pageable cudaMemcpy does)
struct ParamBlock { static constexpr int kPairs = 64; float v[kPairs * 12]; };
__global__ void affine_set_params_kernel(float *state, int n, int n_params, const ParamBlock b)
{
    const int i = threadIdx.x / 12, j = threadIdx.x % 12;
    if (i < n && j < n_params) state[(size_t)i * TRB_STATE_FLOATS + TRB_STATE_PARAMS + j] = b.v[i * 12 + j];
}

// ---- host side ---------------------------------------------------------------------------
static bool g_force_direct = false;   // test hook: trb_set_kernel_path(1) pins the non-TMA kernel

constexpr int kMaxBlocksPerPair = kMaxSlots;

static size_t affine_ws_bytes(int n_pairs)
{
    return (size_t)n_pairs * kMaxBlocksPerPair * TRB_MOMENTS * sizeof(double) + (size_t)n_pairs * kTicketStride * sizeof(unsigned);
}

static int blocks_per_pair(int rows, int n_pairs, int sms)
{
    const int groups = (rows + kWarps - 1) / kWarps;
    // two resident CTAs per SM; whole waves across the batch
    int per = (2 * sms + n_pairs - 1) / n_pairs;
    if (per > groups) per = groups;
    if (per > kMaxBlocksPerPair) per = kMaxBlocksPerPair;
    if (per < 1) per = 1;
    return per;
}

}  // namespace trb

using namespace trb;

extern "C" int trb_sm_count(void)
{
    int n = 0;
    return sm_count(n) ? -1 : n;
}

extern "C" int trb_set_kernel_path(int path)
{
    if (path < 0 || path > 2) { set_error("path must be 0 (auto), 1 (direct) or 2 (per-epoch TMA kernel)"); return TRB_ERR_ARG; }
    g_force_direct = (path == 1);
    set_no_persist(path == 2);
    return TRB_OK;
}

extern "C" const char *trb_affine_kernel_status(void) { return persist_status(); }

extern "C" size_t trb_affine_workspace_bytes(int n_pairs) { return affine_ws_bytes(n_pairs); }

static int validate_common(int ndim, int n_pairs, int D, int H, int W)
{
    if (ndim != 2 && ndim != 3) { set_error("ndim must be 2 or 3 (got %d)", ndim); return TRB_ERR_ARG; }
    if (n_pairs < 1) { set_error("n_pairs must be >= 1"); return TRB_ERR_ARG; }
    if (H < 1 || W < 1 || (ndim == 3 && D < 1)) { set_error("bad volume shape %dx%dx%d", D, H, W); return TRB_ERR_ARG; }
    if ((long long)(ndim == 3 ? D : 1) * H * W >= (1ll << 31)) { set_error("volume too large for 32-bit row indexing"); return TRB_ERR_UNSUPPORTED; }
    return TRB_OK;
}

// ---- pair volume for the large-rotation (gather) variant --------------------------------------------------------------
__global__ void __launch_bounds__(256) affine_build_pairs_kernel(const float *__restrict__ mov, float2 *__restrict__ P, long long rows, int W)
{
    const int Wp = W + 3;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < rows * Wp; i += (long long)gridDim.x * 256) {
        const long long r = i / Wp;
        const int xr = (int)(i - r * Wp);
        const float *row = mov + r * W;
        const int xa = xr - 2, xb = xr - 1;
        P[i] = make_float2((unsigned)xa < (unsigned)W ? __ldg(row + xa) : 0.f, (unsigned)xb < (unsigned)W ? __ldg(row + xb) : 0.f);
    }
}
__global__ void affine_attach_pairs_kernel(unsigned *tickets, unsigned long long addr)
{
    if (threadIdx.x == 0) *reinterpret_cast<unsigned long long *>(tickets + kPairsWord) = addr;
}

__global__ void __launch_bounds__(256) affine_build_quads_kernel(const float *__restrict__ mov, float4 *__restrict__ Q, long long slices,
                                                                 int H, int W)
{
    const int Wp = W + 3, Hp = H + 3;
    const long long per = (long long)Hp * Wp;
    for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < slices * per; i += (long long)gridDim.x * 256) {
        const long long sl = i / per;
        const int r = (int)(i - sl * per), yr = r / Wp, xr = r - yr * Wp;
        const int x = xr - 2, y = yr - 2;
        const float *pl = mov + sl * H * W;
        auto at = [&](int yy, int xx) { return ((unsigned)yy < (unsigned)H && (unsigned)xx < (unsigned)W) ? __ldg(pl + (long long)yy * W + xx) : 0.f; };
        Q[i] = make_float4(at(y, x), at(y, x + 1), at(y + 1, x), at(y + 1, x + 1));
    }
}

extern "C" size_t trb_affine_quads_bytes(int n_pairs, int D, int H, int W)
{
    if (n_pairs < 1 || D < 1 || H < 1 || W < 1) return 0;
    return (size_t)n_pairs * D * (H + 3) * (W + 3) * sizeof(float4);
}

extern "C" int trb_affine_build_quads(const float *moving_dev, float *quads_dev, int n_pairs, int D, int H, int W, void *stream)
{
    int rc = validate_common(3, n_pairs, D, H, W);
    if (rc) return rc;
    if (!moving_dev || !quads_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    const long long slices = (long long)n_pairs * D;
    long long nb = (slices * (H + 3) * (W + 3) + 255) / 256;
    if (nb > 148 * 32) nb = 148 * 32;
    affine_build_quads_kernel<<<(unsigned)nb, 256, 0, (cudaStream_t)stream>>>(moving_dev, reinterpret_cast<float4 *>(quads_dev), slices, H, W);
    return check_cuda(cudaGetLastError(), "affine_build_quads");
}

extern "C" size_t trb_affine_pairs_bytes(int n_pairs, int D, int H, int W)
{
    if (n_pairs < 1 || D < 1 || H < 1 || W < 1) return 0;
    return (size_t)n_pairs * D * H * (W + 3) * sizeof(float2);
}

extern "C" int trb_affine_build_pairs(const float *moving_dev, float *pairs_dev, int n_pairs, int D, int H, int W, void *stream)
{
    int rc = validate_common(3, n_pairs, D, H, W);
    if (rc) return rc;
    if (!moving_dev || !pairs_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    const long long rows = (long long)n_pairs * D * H;
    long long nb = (rows * (W + 3) + 255) / 256;
    if (nb > 148 * 32) nb = 148 * 32;
    affine_build_pairs_kernel<<<(unsigned)nb, 256, 0, (cudaStream_t)stream>>>(moving_dev, reinterpret_cast<float2 *>(pairs_dev), rows, W);
    return check_cuda(cudaGetLastError(), "affine_build_pairs");
}

extern "C" int trb_affine_attach_pairs(void *workspace_dev, size_t workspace_bytes, int n_pairs, const float *pairs_dev, void *stream)
{
    if (!workspace_dev || n_pairs < 1 || workspace_bytes < affine_ws_bytes(n_pairs)) { set_error("workspace too small / null"); return TRB_ERR_WORKSPACE; }
    unsigned *tickets = (unsigned *)((char *)workspace_dev + (size_t)n_pairs * kMaxBlocksPerPair * TRB_MOMENTS * sizeof(double));
    affine_attach_pairs_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(tickets, (unsigned long long)(uintptr_t)pairs_dev);
    return check_cuda(cudaGetLastError(), "affine_attach_pairs");
}

extern "C" int trb_affine_set_params(float *state_dev, int n_pairs, int n_params, const float *params_host, int n_rows, void *stream)
{
    if (!state_dev || !params_host || n_pairs < 1) { set_error("null state / params"); return TRB_ERR_ARG; }
    if (n_params < 1 || n_params > 12 || (n_rows != 1 && n_rows != n_pairs)) { set_error("bad n_params / n_rows"); return TRB_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    for (int p0 = 0; p0 < n_pairs; p0 += ParamBlock::kPairs) {
        const int n = n_pairs - p0 < ParamBlock::kPairs ? n_pairs - p0 : ParamBlock::kPairs;
        ParamBlock b{};
        for (int i = 0; i < n; ++i)
            for (int j = 0; j < n_params; ++j) b.v[i * 12 + j] = params_host[(size_t)(n_rows == 1 ? 0 : p0 + i) * n_params + j];
        affine_set_params_kernel<<<1, ParamBlock::kPairs * 12, 0, s>>>(state_dev + (size_t)p0 * TRB_STATE_FLOATS, n, n_params, b);
    }
    return check_cuda(cudaGetLastError(), "affine_set_params");
}

extern "C" int trb_affine_init_state(int ndim, int mode, float *state_dev, int n_pairs, void *stream)
{
    if (ndim != 2 && ndim != 3) { set_error("ndim must be 2 or 3"); return TRB_ERR_ARG; }
    if (!state_dev || n_pairs < 1) { set_error("null state / n_pairs"); return TRB_ERR_ARG; }
    cudaStream_t s = (cudaStream_t)stream;
    const int tb = 64, nb = (n_pairs + tb - 1) / tb;
    if (ndim == 3) affine_init_state_kernel<3><<<nb, tb, 0, s>>>(state_dev, n_pairs, mode);
    else affine_init_state_kernel<2><<<nb, tb, 0, s>>>(state_dev, n_pairs, mode);
    return check_cuda(cudaGetLastError(), "affine_init_state");
}

static int fill_params(AffineParams &p, int ndim, const float *moving, const float *target, long long pair_stride,
                       int n_pairs, int D, int H, int W, const float *xb, const float *yb, const float *zb,
                       void *ws, size_t ws_bytes)
{
    int rc = validate_common(ndim, n_pairs, D, H, W);
    if (rc) return rc;
    if (!moving || !target || !xb || !yb || (ndim == 3 && !zb)) { set_error("null input pointer"); return TRB_ERR_ARG; }
    if (!ws || ws_bytes < affine_ws_bytes(n_pairs)) { set_error("workspace too small: need %zu bytes", affine_ws_bytes(n_pairs)); return TRB_ERR_WORKSPACE; }
    p.moving = moving; p.target = target; p.pair_stride = pair_stride;
    p.D = ndim == 3 ? D : 1; p.H = H; p.W = W;
    p.xb = xb; p.yb = yb; p.zb = zb;
    p.partials = (double *)ws;
    p.tickets = (unsigned *)((char *)ws + (size_t)n_pairs * kMaxBlocksPerPair * TRB_MOMENTS * sizeof(double));
    return TRB_OK;
}

extern "C" int trb_affine_tile_fits(int D, int H, int W, const float *theta_host)
{
    // the footprint test of the producer (csrc/affine_persist.cu) for the tile at the centre of the volume, on the host
    if (!theta_host || D < 1 || H < 1 || W < 1) return 0;
    const double h[3] = {0.5 * W, 0.5 * H, 0.5 * D};
    const double T[3] = {(double)(TX < W ? TX : W), (double)(TY < H ? TY : H), (double)(TZ < D ? TZ : D)};
    const double step[3] = {2.0 / W, 2.0 / H, 2.0 / D};          // base coordinate per voxel
    const int B[3] = {kBX, kBY, kBZ};
    for (int r = 0; r < 3; ++r) {
        double ext = 0.0;
        for (int c = 0; c < 3; ++c) ext += fabs((double)theta_host[r * 4 + c]) * h[r] * step[c] * (T[c] - 1.0);
        const double need = ext + 2.06 + (r == 0 ? 3.0 : 0.0);   // + the cell's far corner, + 16-byte alignment of the box start in x
        if (need > (double)B[r] - 1.0) return 0;
    }
    return 1;
}

extern "C" int trb_affine_optim(int ndim, int mode, const float *moving_dev, const float *target_dev,
                                long long pair_stride, int n_pairs, int D, int H, int W,
                                const float *xb_dev, const float *yb_dev, const float *zb_dev,
                                float *state_dev, float *loss_log_dev, int log_stride, int epoch0, int n_epochs,
                                float w_mse, float w_ncc, float lr, int optimiser, float beta1, float beta2,
                                float adam_eps, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    return trb_affine_optim_ex(ndim, mode, moving_dev, target_dev, pair_stride, n_pairs, D, H, W, xb_dev, yb_dev, zb_dev, state_dev,
                               loss_log_dev, log_stride, epoch0, n_epochs, w_mse, w_ncc, lr, optimiser, beta1, beta2, adam_eps,
                               0, workspace_dev, workspace_bytes, stream);
}

extern "C" int trb_affine_optim_ex(int ndim, int mode, const float *moving_dev, const float *target_dev,
                                   long long pair_stride, int n_pairs, int D, int H, int W,
                                   const float *xb_dev, const float *yb_dev, const float *zb_dev,
                                   float *state_dev, float *loss_log_dev, int log_stride, int epoch0, int n_epochs,
                                   float w_mse, float w_ncc, float lr, int optimiser, float beta1, float beta2,
                                   float adam_eps, int flags, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    AffineParams p{};
    int rc = fill_params(p, ndim, moving_dev, target_dev, pair_stride, n_pairs, D, H, W, xb_dev, yb_dev, zb_dev,
                         workspace_dev, workspace_bytes);
    if (rc) return rc;
    if (!state_dev) { set_error("null state"); return TRB_ERR_ARG; }
    if (mode != TRB_MODE_RIGID && mode != TRB_MODE_AFFINE) { set_error("bad mode %d", mode); return TRB_ERR_ARG; }
    if (optimiser != TRB_OPT_SGD && optimiser != TRB_OPT_ADAM) { set_error("bad optimiser %d", optimiser); return TRB_ERR_ARG; }
    if (loss_log_dev && epoch0 + n_epochs > log_stride) { set_error("loss log too short"); return TRB_ERR_ARG; }
    p.s_begin = 0; p.s_end = ndim == 3 ? D : H;
    p.state = state_dev; p.loss_log = loss_log_dev; p.log_stride = log_stride;
    p.w_mse = w_mse; p.w_ncc = w_ncc; p.lr = lr; p.mode = mode; p.optimiser = optimiser;
    p.beta1 = beta1; p.beta2 = beta2; p.adam_eps = adam_eps;
    p.gather = (flags & TRB_FLAG_LARGE_ROTATION) ? ((flags & TRB_FLAG_QUAD_VOLUME) ? 3 : (flags & TRB_FLAG_PAIR_VOLUME) ? 2 : 1) : 0;
    cudaStream_t s = (cudaStream_t)stream;
    if (!g_force_direct && tma_path_eligible(ndim, p, n_pairs)) {
        if (n_epochs <= 0) return TRB_OK;
        rc = launch_affine3d_persist(p, n_pairs, epoch0, n_epochs, s);      // all epochs in one cooperative launch
        if (rc != TRB_ERR_UNSUPPORTED) return rc;
        return launch_affine3d_tma(p, n_pairs, true, epoch0, n_epochs, s);  // one launch per epoch
    }
    int sms;
    if ((rc = sm_count(sms))) return rc;
    const int rows = ndim == 3 ? D * H : H;
    const dim3 grid(blocks_per_pair(rows, n_pairs, sms), n_pairs);
    for (int e = 0; e < n_epochs; ++e) {
        p.epoch = epoch0 + e;
        if (ndim == 3) affine_moments_kernel<3, true><<<grid, kThreads, 0, s>>>(p);
        else affine_moments_kernel<2, true><<<grid, kThreads, 0, s>>>(p);
    }
    return check_cuda(cudaGetLastError(), "affine_optim");
}

extern "C" int trb_affine_optim_peer(const float *moving_dev, const float *target_dev, int D, int H, int W, int s_begin, int s_end,
                                     const float *xb_dev, const float *yb_dev, const float *zb_dev, int mode,
                                     float *state_dev, float *loss_log_dev, int log_stride, int epoch0, int n_epochs,
                                     float w_mse, float w_ncc, float lr, int optimiser, float beta1, float beta2, float adam_eps,
                                     void *const *mailbox_ptrs, int rank, int world, unsigned long long seq0,
                                     void *workspace_dev, size_t workspace_bytes, void *stream)
{
    AffineParams p{};
    int rc = fill_params(p, 3, moving_dev, target_dev, 0, 1, D, H, W, xb_dev, yb_dev, zb_dev, workspace_dev, workspace_bytes);
    if (rc) return rc;
    if (!state_dev) { set_error("null state"); return TRB_ERR_ARG; }
    if (mode != TRB_MODE_RIGID && mode != TRB_MODE_AFFINE) { set_error("bad mode %d", mode); return TRB_ERR_ARG; }
    if (optimiser != TRB_OPT_SGD && optimiser != TRB_OPT_ADAM) { set_error("bad optimiser %d", optimiser); return TRB_ERR_ARG; }
    if (loss_log_dev && epoch0 + n_epochs > log_stride) { set_error("loss log too short"); return TRB_ERR_ARG; }
    if (s_begin < 0 || s_end > D || s_begin >= s_end) { set_error("bad slab [%d,%d) of %d", s_begin, s_end, D); return TRB_ERR_ARG; }
    if (world < 1 || world > 8 || rank < 0 || rank >= world || !mailbox_ptrs || seq0 < 1) { set_error("bad peer set (world 1..8, seq0 >= 1)"); return TRB_ERR_ARG; }
    for (int r = 0; r < world; ++r) {
        if (!mailbox_ptrs[r]) { set_error("null mailbox pointer for rank %d", r); return TRB_ERR_ARG; }
        p.peer.mailbox[r] = (double *)mailbox_ptrs[r];
    }
    p.peer.rank = rank; p.peer.world = world; p.peer.seq = seq0;
    p.s_begin = s_begin; p.s_end = s_end;
    p.state = state_dev; p.loss_log = loss_log_dev; p.log_stride = log_stride;
    p.w_mse = w_mse; p.w_ncc = w_ncc; p.lr = lr; p.mode = mode; p.optimiser = optimiser;
    p.beta1 = beta1; p.beta2 = beta2; p.adam_eps = adam_eps;
    if (!tma_path_eligible(3, p, 1)) { set_error("the fused sharded epoch needs the TMA kernel (3-D, W %% 4 == 0, W >= 32, H >= 16)"); return TRB_ERR_UNSUPPORTED; }
    if (n_epochs <= 0) return TRB_OK;             // validation only
    rc = launch_affine3d_persist(p, 1, epoch0, n_epochs, (cudaStream_t)stream);   // all epochs in one launch, exchange inside
    if (rc != TRB_ERR_UNSUPPORTED) return rc;
    return launch_affine3d_tma(p, 1, true, epoch0, n_epochs, (cudaStream_t)stream);
}

int trb::affine_moments_impl(int ndim, const float *moving_dev, const float *target_dev, long long pair_stride,
                             int n_pairs, int D, int H, int W, int s_begin, int s_end,
                             const float *xb_dev, const float *yb_dev, const float *zb_dev,
                             const float *state_dev, double *moments_dev, int flags, int target_sums,
                             float *warped_out, bool *wrote_warped, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    // target_sums: 0 = the caller does not need sum t / sum t^2 (vjp pass), 1 = compute them (stand-alone call), 3 = compute
    // them and keep them for later calls, 2 = an earlier call with 3 on this workspace and these targets left them valid
    // (only the persistent kernel keeps them apart from the pass)
    if (wrote_warped) *wrote_warped = false;
    AffineParams p{};
    int rc = fill_params(p, ndim, moving_dev, target_dev, pair_stride, n_pairs, D, H, W, xb_dev, yb_dev, zb_dev,
                         workspace_dev, workspace_bytes);
    if (rc) return rc;
    const int smax = ndim == 3 ? D : H;
    if (s_begin < 0 || s_end > smax || s_begin >= s_end) { set_error("bad slab [%d,%d) of %d", s_begin, s_end, smax); return TRB_ERR_ARG; }
    if (!state_dev || !moments_dev) { set_error("null state/moments"); return TRB_ERR_ARG; }
    p.s_begin = s_begin; p.s_end = s_end;
    p.state = const_cast<float *>(state_dev);
    p.moments_out = moments_dev;
    p.gather = (flags & TRB_FLAG_LARGE_ROTATION) ? ((flags & TRB_FLAG_QUAD_VOLUME) ? 3 : (flags & TRB_FLAG_PAIR_VOLUME) ? 2 : 1) : 0;
    int sms;
    if ((rc = sm_count(sms))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (!g_force_direct && tma_path_eligible(ndim, p, n_pairs)) {
        // both TMA-tile kernels store the warped samples on request (whole volumes of single-channel pairs only)
        const bool store = warped_out && s_begin == 0 && s_end == D && pair_stride == (long long)D * H * W;
        // One pass of the persistent kernel (steady-state rate of the fused loop, ~15 us of cooperative launch + publish)
        // against the per-epoch kernel (lower fixed cost, 25 % slower per tile): large rotations always (its gather
        // variant is 2-3x faster than the per-epoch kernel's uncached fallback), else from ~10 tiles per SM on — unless the
        // pass would have to recompute the target sums (a separate pass over the targets in the persistent design: the
        // default-loss loop caches them after its first epoch, a stand-alone trb_affine_moments call cannot)
        const long long tiles = (long long)n_pairs * ((W + TX - 1) / TX) * ((H + TY - 1) / TY) * ((s_end - s_begin + TZ - 1) / TZ);
        if (p.gather || (target_sums != 1 && tiles >= 10LL * sms)) {
            if (store) p.warped_out = warped_out;
            rc = launch_affine3d_persist(p, n_pairs, 0, 1, s, target_sums == 0 ? 2 : (target_sums == 2 ? 3 : 1));   // 1 and 3: compute
            if (rc != TRB_ERR_UNSUPPORTED) {
                if (rc == TRB_OK && store && wrote_warped) *wrote_warped = true;
                return rc;
            }
            p.warped_out = nullptr;
        }
        if (store) {
            p.warped_out = warped_out;
            if (wrote_warped) *wrote_warped = true;
        }
        return launch_affine3d_tma(p, n_pairs, false, 0, 1, s);
    }
    const int rows = (s_end - s_begin) * (ndim == 3 ? H : 1);
    const dim3 grid(blocks_per_pair(rows, n_pairs, sms), n_pairs);
    if (ndim == 3) affine_moments_kernel<3, false><<<grid, kThreads, 0, s>>>(p);
    else affine_moments_kernel<2, false><<<grid, kThreads, 0, s>>>(p);
    return check_cuda(cudaGetLastError(), "affine_moments");
}

extern "C" int trb_affine_moments(int ndim, const float *moving_dev, const float *target_dev, long long pair_stride,
                                  int n_pairs, int D, int H, int W, int s_begin, int s_end,
                                  const float *xb_dev, const float *yb_dev, const float *zb_dev,
                                  const float *state_dev, double *moments_dev,
                                  void *workspace_dev, size_t workspace_bytes, void *stream)
{
    return affine_moments_impl(ndim, moving_dev, target_dev, pair_stride, n_pairs, D, H, W, s_begin, s_end, xb_dev, yb_dev, zb_dev,
                               state_dev, moments_dev, 0, 1, nullptr, nullptr, workspace_dev, workspace_bytes, stream);
}

extern "C" int trb_affine_moments_ex(int ndim, const float *moving_dev, const float *target_dev, long long pair_stride,
                                     int n_pairs, int D, int H, int W, int s_begin, int s_end,
                                     const float *xb_dev, const float *yb_dev, const float *zb_dev,
                                     const float *state_dev, double *moments_dev, int flags,
                                     void *workspace_dev, size_t workspace_bytes, void *stream)
{
    return affine_moments_impl(ndim, moving_dev, target_dev, pair_stride, n_pairs, D, H, W, s_begin, s_end, xb_dev, yb_dev, zb_dev,
                               state_dev, moments_dev, flags, 1, nullptr, nullptr, workspace_dev, workspace_bytes, stream);
}

extern "C" int trb_affine_apply(int ndim, int mode, const double *moments_dev, int n_pairs, int D, int H, int W,
                                float *state_dev, float *loss_log_dev, int log_stride, int epoch,
                                float w_mse, float w_ncc, float lr, int optimiser, float beta1, float beta2,
                                float adam_eps, const double *extra_dev, void *stream)
{
    int rc = validate_common(ndim, n_pairs, D, H, W);
    if (rc) return rc;
    if (!moments_dev || !state_dev) { set_error("null moments/state"); return TRB_ERR_ARG; }
    if (loss_log_dev && epoch >= log_stride) { set_error("loss log too short"); return TRB_ERR_ARG; }
    AffineParams p{};
    p.pair_stride = n_pairs;     // apply kernel: number of pairs rides in pair_stride
    p.D = ndim == 3 ? D : 1; p.H = H; p.W = W;
    p.state = state_dev; p.loss_log = loss_log_dev; p.log_stride = log_stride; p.epoch = epoch;
    p.w_mse = w_mse; p.w_ncc = w_ncc; p.lr = lr; p.mode = mode; p.optimiser = optimiser;
    p.beta1 = beta1; p.beta2 = beta2; p.adam_eps = adam_eps;
    p.extra = extra_dev;
    cudaStream_t s = (cudaStream_t)stream;
    const int tb = 32, nb = (n_pairs + tb - 1) / tb;
    if (ndim == 3) affine_apply_kernel<3><<<nb, tb, 0, s>>>(p, moments_dev);
    else affine_apply_kernel<2><<<nb, tb, 0, s>>>(p, moments_dev);
    return check_cuda(cudaGetLastError(), "affine_apply");
}

extern "C" int trb_warp_affine(int ndim, const float *moving_dev, float *out_dev, int n_channels, int D, int H, int W,
                               const float *theta_dev, const float *xb_dev, const float *yb_dev, const float *zb_dev,
                               void *stream)
{
    return trb_warp_affine_batch(ndim, moving_dev, out_dev, 1, n_channels, D, H, W, theta_dev, xb_dev, yb_dev, zb_dev, 0, stream);
}

extern "C" int trb_warp_affine_batch(int ndim, const float *moving_dev, float *out_dev, int n_pairs, int n_channels, int D, int H, int W,
                                     const float *theta_dev, const float *xb_dev, const float *yb_dev, const float *zb_dev,
                                     int flags, void *stream)
{
    int rc = validate_common(ndim, n_pairs, D, H, W);
    if (rc) return rc;
    // the nearest kernels round through round_idx; the bilinear gather kernels floor with floorf and take any axis (the
    // TMA-staged ones are only eligible for axes far below the limit)
    if ((flags & TRB_FLAG_NEAREST) && (rc = check_fast_floor_axes(ndim, D, H, W))) return rc;
    if (!moving_dev || !out_dev || !theta_dev || !xb_dev || !yb_dev || (ndim == 3 && !zb_dev) || n_channels < 1) {
        set_error("null pointer / n_channels"); return TRB_ERR_ARG;
    }
    if (n_pairs > 65535) { set_error("at most 65535 pairs per call"); return TRB_ERR_ARG; }
    const size_t vol = (size_t)(ndim == 3 ? D : 1) * H * W;
    cudaStream_t s = (cudaStream_t)stream;
    // 3-D: TMA-staged tiles unless the caller knows theta is a large rotation (then the gathers of the one-thread-per-
    // voxel kernel, which keeps the whole L1, are the better path)
    const bool nearest = flags & TRB_FLAG_NEAREST;
    if (ndim == 3 && !g_force_direct && !(flags & TRB_FLAG_LARGE_ROTATION) &&
        warp_tma_eligible(moving_dev, out_dev, n_pairs * n_channels, (long long)vol, D, H, W))
        return launch_warp_affine_tma(moving_dev, out_dev, n_pairs, n_channels, D, H, W, theta_dev, xb_dev, yb_dev, nearest, s);
    int sms;
    if ((rc = sm_count(sms))) return rc;
    size_t nb = (vol + 255) / 256;
    if (nb > (size_t)sms * 16) nb = (size_t)sms * 16;
    const dim3 grid((unsigned)nb, (unsigned)n_pairs);
    if (nearest) {
        if (ndim == 3) warp_affine_nearest_kernel<3><<<grid, 256, 0, s>>>(moving_dev, out_dev, n_channels, D, H, W, theta_dev, xb_dev, yb_dev, zb_dev);
        else warp_affine_nearest_kernel<2><<<grid, 256, 0, s>>>(moving_dev, out_dev, n_channels, 1, H, W, theta_dev, xb_dev, yb_dev, zb_dev);
    } else if (ndim == 3) {
        warp_affine_kernel<3><<<grid, 256, 0, s>>>(moving_dev, out_dev, n_channels, D, H, W, theta_dev, xb_dev, yb_dev, zb_dev);
    } else {
        warp_affine_kernel<2><<<grid, 256, 0, s>>>(moving_dev, out_dev, n_channels, 1, H, W, theta_dev, xb_dev, yb_dev, zb_dev);
    }
    return check_cuda(cudaGetLastError(), "warp_affine");
}

extern "C" int trb_warp_affine_vjp(int ndim, const float *moving_dev, const float *gout_dev, int D, int H, int W,
                                   const float *theta_dev, const float *xb_dev, const float *yb_dev, const float *zb_dev,
                                   double *dtheta_dev, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    return trb_warp_affine_vjp_ex(ndim, moving_dev, gout_dev, D, H, W, theta_dev, xb_dev, yb_dev, zb_dev, dtheta_dev, 0,
                                  workspace_dev, workspace_bytes, stream);
}

extern "C" int trb_warp_affine_vjp_ex(int ndim, const float *moving_dev, const float *gout_dev, int D, int H, int W,
                                      const float *theta_dev, const float *xb_dev, const float *yb_dev, const float *zb_dev,
                                      double *dtheta_dev, int flags, void *workspace_dev, size_t workspace_bytes, void *stream)
{
    // Reuses the moments pass with gout in the target slot: sum_v gout_v * J_v is moment block [17..28].
    // The unfused pass only ever reads state[TRB_STATE_THETA .. +12), so a bare theta pointer is rebased.
    if (!dtheta_dev) { set_error("null dtheta"); return TRB_ERR_ARG; }
    if (workspace_bytes < affine_ws_bytes(1) + TRB_MOMENTS * sizeof(double)) {
        set_error("workspace too small: need %zu bytes", affine_ws_bytes(1) + TRB_MOMENTS * sizeof(double));
        return TRB_ERR_WORKSPACE;
    }
    double *mom = (double *)((char *)workspace_dev + affine_ws_bytes(1));
    int rc = affine_moments_impl(ndim, moving_dev, gout_dev, 0, 1, D, H, W, 0, ndim == 3 ? D : H, xb_dev, yb_dev, zb_dev,
                                 theta_dev - TRB_STATE_THETA, mom, flags, 0, nullptr, nullptr, workspace_dev, affine_ws_bytes(1), stream);
    if (rc) return rc;
    vjp_extract_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(mom, dtheta_dev, ndim, ndim == 3 ? D : 1, H, W);
    return check_cuda(cudaGetLastError(), "warp_affine_vjp");
}
