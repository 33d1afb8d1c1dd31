// flow_direct.cu — EXTENSION (north_star items 2b/3; BASELINE configs[2] "direct" variant and configs[4]):
// direct per-voxel flow optimisation.  The reference optimises the weights of a U-Net whose output is the
// flow (warpings.py:178-233); there is no per-voxel flow optimiser and no smoothness term in it, so this
// path has no reference counterpart — its oracle is oracle/torch_port.py:direct_flow_loop, assembled from
// the reference's own SpatialTransformer (utils.py:350-365) + MSE/NCC (utils.py:197-205) + torch SGD/Adam +
// a VoxelMorph-style smoothness penalty (mean over axes of the mean squared forward difference).
//
// One epoch = two streaming passes over a z-slab of the volume:
//   stats : warp(moving, flow) -> 5 similarity moments + the smoothness sum            (20 B/voxel + halo)
//   update: same sample + derivative, dL/dflow = (cw*w + ct*t + c0)*G + lambda*stencil, SGD or Adam,
//           written out of place (32 B/voxel SGD, 80 B/voxel Adam)
// Between the passes the caller all-reduces the 6 moments when the volume is sharded over GPUs
// (parallel.ShardedDirectFlow); on one GPU trb_flow_direct_epoch chains both.
// Layout of a slab: flow/adam [ndim][Ds][H][W], target [Ds][H][W] hold slices [z_off, z_off+Ds) of the
// volume; `moving` is the full [D][H][W] volume; halo_lo / halo_hi are the neighbour ranks' flow slices
// z_off-1 and z_off+Ds ([ndim][H][W]) or NULL at the volume boundary.
#include "common.cuh"
#include "peer.cuh"
#include "tma_utils.cuh"
#include <math.h>

namespace trb {

// row-wise voxel loop over a slab (see flow.cu): f(idx, x, y, zl)
template <typename F>
__device__ __forceinline__ void for_each_slab_voxel(int Ds, int H, int W, F f)
{
    const int rows = Ds * H;
    const int rx = threadIdx.x & 127, ry = threadIdx.x >> 7;
    for (int row = 2 * blockIdx.x + ry; row < rows; row += 2 * gridDim.x) {
        const int zl = row / H, y = row - zl * H;
        const size_t base = (size_t)row * W;
#pragma unroll 1
        for (int x = rx; x < W; x += 128) f(base + x, x, y, zl);
    }
}

struct DirectParams {
    const float *moving, *target, *flow_in, *halo_lo, *halo_hi;
    float *flow_out, *adam_m, *adam_v, *loss_log;
    int D, H, W, z_off, Ds;
    double *moments;        // [6]
    double *partials;       // [blocks][6]
    unsigned *ticket;
    float w_mse, w_ncc, lambda, lr;
    int optimiser, step, epoch;
    float beta1, beta2, eps;
    int complete_prev;      // fused step: moments[5] / the stash belong to the previous call, finish its loss entry
    // fused step: launch-invariant values computed on the host so they are constant-bank operands, not registers
    AxisMap ax, ay, az;
    float wsm[3], ssm[3];   // smoothness weights per axis (x, y, z) and 2*lambda*weight
    float step_size, inv_bc2s, ob1, ob2;
    // sharded, fused: halo slices read in place from the neighbour ranks' flow buffers (channel stride = their Ds*H*W),
    // the 6 sums all-reduced by the last CTA through peer mailboxes (peer.cuh)
    int halo_lo_cs, halo_hi_cs;
    PeerExchange peer;
};

// flow value of channel c at slab-local (zl, y, x) with zl in [-1, Ds] resolved through the halos
template <int NDIM>
__device__ __forceinline__ float flow_at(const DirectParams &p, int c, int zl, int y, int x)
{
    const size_t HW = (size_t)p.H * p.W;
    if (NDIM == 3) {
        if (zl < 0) return __ldg(p.halo_lo + (size_t)c * HW + (size_t)y * p.W + x);
        if (zl >= p.Ds) return __ldg(p.halo_hi + (size_t)c * HW + (size_t)y * p.W + x);
        return __ldg(p.flow_in + ((size_t)c * p.Ds + zl) * HW + (size_t)y * p.W + x);
    }
    return __ldg(p.flow_in + (size_t)c * HW + (size_t)y * p.W + x);
}

// weight of one squared forward difference along axis a in  mean_axes( mean(diff^2) )
template <int NDIM>
__device__ __forceinline__ float smooth_weight(const DirectParams &p, int a)
{
    const double dims[3] = {(double)p.W, (double)p.H, (double)(NDIM == 3 ? p.D : 1)};
    double n = (double)NDIM;                   // channels
    for (int k = 0; k < NDIM; ++k) n *= (k == a) ? dims[k] - 1.0 : dims[k];
    return (float)(1.0 / (n * NDIM));
}

template <int NDIM>
__global__ void __launch_bounds__(256) flow_direct_stats_kernel(const DirectParams p)
{
    const int W = p.W, H = p.H, D = NDIM == 3 ? p.D : 1, Ds = NDIM == 3 ? p.Ds : 1;
    const size_t HW = (size_t)H * W, slab = HW * Ds;
    const AxisMap ax = axis_map(W), ay = axis_map(H), az = axis_map(D > 1 ? D : 2);
    const float wx = smooth_weight<NDIM>(p, 0), wy = smooth_weight<NDIM>(p, 1), wz = NDIM == 3 ? smooth_weight<NDIM>(p, 2) : 0.f;
    float s[6] = {0, 0, 0, 0, 0, 0};          // fp32 per thread (~50 voxels), fp64 above (see flow.cu)
    for_each_slab_voxel(Ds, H, W, [&](size_t idx, int x, int y, int zl) {
        const int z = p.z_off + zl;
        float f[3] = {0.f, 0.f, 0.f};          // f[c]: channel c displaces spatial axis c (0 = D|H first axis)
#pragma unroll
        for (int c = 0; c < NDIM; ++c) f[c] = ld_stream_f(p.flow_in + (size_t)c * slab + idx);
        float px, py, pz = 0.f;
        if (NDIM == 3) { pz = flow_pos(az, z, f[0]); py = flow_pos(ay, y, f[1]); px = flow_pos(ax, x, f[2]); }
        else { py = flow_pos(ay, y, f[0]); px = flow_pos(ax, x, f[1]); }
        const Sample<NDIM> sp = sample_zero_pad<NDIM, true>(p.moving, D, H, W, px, py, pz);
        const float val = sp.val;
        const float g[3] = {sp.g[0], sp.g[1], NDIM == 3 ? sp.g[NDIM - 1] : 0.f};
        const float t = ld_stream_f(p.target + idx);
        s[0] += t; s[1] += val;
        s[2] = fmaf(t, t, s[2]); s[3] = fmaf(val, val, s[3]); s[4] = fmaf(t, val, s[4]);
        if (p.lambda != 0.f) {
            float sm = 0.f;
#pragma unroll
            for (int c = 0; c < NDIM; ++c) {
                if (x + 1 < W) { const float d = flow_at<NDIM>(p, c, zl, y, x + 1) - f[c]; sm = fmaf(wx * d, d, sm); }
                if (y + 1 < H) { const float d = flow_at<NDIM>(p, c, zl, y + 1, x) - f[c]; sm = fmaf(wy * d, d, sm); }
                if (NDIM == 3 && z + 1 < D) { const float d = flow_at<NDIM>(p, c, zl + 1, y, x) - f[c]; sm = fmaf(wz * d, d, sm); }
            }
            s[5] += sm;
        }
    });
    __shared__ double red[kWarps][6];
    if (grid_sum(s, red, p.partials, p.ticket) && threadIdx.x < 6) p.moments[threadIdx.x] = red[0][threadIdx.x];
}

template <int NDIM>
__global__ void __launch_bounds__(256) flow_direct_update_kernel(const DirectParams p)
{
    const int W = p.W, H = p.H, D = NDIM == 3 ? p.D : 1, Ds = NDIM == 3 ? p.Ds : 1;
    const size_t HW = (size_t)H * W, slab = HW * Ds;
    const AxisMap ax = axis_map(W), ay = axis_map(H), az = axis_map(D > 1 ? D : 2);
    __shared__ float coef[3];
    if (threadIdx.x == 0) {
        const double n = (double)D * H * W;
        const LossCoef lc = loss_coefficients(n, p.moments[0], p.moments[1], p.moments[2], p.moments[3], p.moments[4],
                                              (double)p.w_mse, (double)p.w_ncc);
        coef[0] = (float)lc.cw; coef[1] = (float)lc.ct; coef[2] = (float)lc.c0;
        if (blockIdx.x == 0 && p.loss_log) p.loss_log[p.epoch] = (float)(lc.loss + (double)p.lambda * p.moments[5]);
    }
    __syncthreads();
    const float cw = coef[0], ct = coef[1], c0 = coef[2];
    const float sw[3] = {2.f * p.lambda * smooth_weight<NDIM>(p, 0), 2.f * p.lambda * smooth_weight<NDIM>(p, 1),
                         NDIM == 3 ? 2.f * p.lambda * smooth_weight<NDIM>(p, 2) : 0.f};
    float bc1 = 1.f, bc2s = 1.f;
    if (p.optimiser == TRB_OPT_ADAM) {
        bc1 = 1.f - powf(p.beta1, (float)p.step);
        bc2s = sqrtf(1.f - powf(p.beta2, (float)p.step));
    }
    for_each_slab_voxel(Ds, H, W, [&](size_t idx, int x, int y, int zl) {
        const int z = p.z_off + zl;
        float f[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for (int c = 0; c < NDIM; ++c) f[c] = ld_stream_f(p.flow_in + (size_t)c * slab + idx);
        float px, py, pz = 0.f;
        if (NDIM == 3) { pz = flow_pos(az, z, f[0]); py = flow_pos(ay, y, f[1]); px = flow_pos(ax, x, f[2]); }
        else { py = flow_pos(ay, y, f[0]); px = flow_pos(ax, x, f[1]); }
        const Sample<NDIM> sp = sample_zero_pad<NDIM, true>(p.moving, D, H, W, px, py, pz);
        const float val = sp.val;
        const float g[3] = {sp.g[0], sp.g[1], NDIM == 3 ? sp.g[NDIM - 1] : 0.f};
        const float t = ld_stream_f(p.target + idx);
        const float r = fmaf(cw, val, fmaf(ct, t, c0));
#pragma unroll
        for (int c = 0; c < NDIM; ++c) {
            float gr = r * g[NDIM - 1 - c];          // channel c <-> sampling coordinate NDIM-1-c
            if (p.lambda != 0.f) {
                float st = 0.f;
                if (x + 1 < W) st -= sw[0] * (flow_at<NDIM>(p, c, zl, y, x + 1) - f[c]);
                if (x > 0) st += sw[0] * (f[c] - flow_at<NDIM>(p, c, zl, y, x - 1));
                if (y + 1 < H) st -= sw[1] * (flow_at<NDIM>(p, c, zl, y + 1, x) - f[c]);
                if (y > 0) st += sw[1] * (f[c] - flow_at<NDIM>(p, c, zl, y - 1, x));
                if (NDIM == 3) {
                    if (z + 1 < D) st -= sw[2] * (flow_at<NDIM>(p, c, zl + 1, y, x) - f[c]);
                    if (z > 0) st += sw[2] * (f[c] - flow_at<NDIM>(p, c, zl - 1, y, x));
                }
                gr += st;
            }
            const size_t o = (size_t)c * slab + idx;
            float nv;
            if (p.optimiser == TRB_OPT_SGD) {
                nv = f[c] - p.lr * gr;
            } else {
                float m = p.adam_m[o], v = p.adam_v[o];
                m = p.beta1 * m + (1.f - p.beta1) * gr;
                v = p.beta2 * v + (1.f - p.beta2) * gr * gr;
                p.adam_m[o] = m; p.adam_v[o] = v;
                nv = f[c] - (p.lr / bc1) * (m / (sqrtf(v) / bc2s + p.eps));
            }
            p.flow_out[o] = nv;
        }
    });
}

// The update pass of the LNCC epoch (lncc.cu): dL/dJ comes from an array (trb_lncc_backward, which already added the
// pointwise MSE / NCC terms) instead of cw*w + ct*t + c0; the sample gradient G, the smoothness stencil and SGD / Adam
// are those of flow_direct_update_kernel.  Whole volume only (z_off 0, Ds = D): LNCC is single-GPU.
// loss_log[epoch] = similarity(moments) + w_lncc * lncc_stats[1] + lambda * moments[5], the loss of flow_in.
template <int NDIM>
__global__ void __launch_bounds__(256) flow_direct_update_lncc_kernel(const DirectParams p, const float *__restrict__ resid,
                                                                      const double *__restrict__ lncc_stats, const float w_lncc)
{
    const int W = p.W, H = p.H, D = NDIM == 3 ? p.D : 1, Ds = NDIM == 3 ? p.Ds : 1;
    const size_t HW = (size_t)H * W, slab = HW * Ds;
    const AxisMap ax = axis_map(W), ay = axis_map(H), az = axis_map(D > 1 ? D : 2);
    if (threadIdx.x == 0 && blockIdx.x == 0 && p.loss_log) {
        const double n = (double)D * H * W;
        const LossCoef lc = loss_coefficients(n, p.moments[0], p.moments[1], p.moments[2], p.moments[3], p.moments[4],
                                              (double)p.w_mse, (double)p.w_ncc);
        p.loss_log[p.epoch] = (float)(lc.loss + (double)w_lncc * lncc_stats[1] + (double)p.lambda * p.moments[5]);
    }
    const float sw[3] = {2.f * p.lambda * smooth_weight<NDIM>(p, 0), 2.f * p.lambda * smooth_weight<NDIM>(p, 1),
                         NDIM == 3 ? 2.f * p.lambda * smooth_weight<NDIM>(p, 2) : 0.f};
    float bc1 = 1.f, bc2s = 1.f;
    if (p.optimiser == TRB_OPT_ADAM) {
        bc1 = 1.f - powf(p.beta1, (float)p.step);
        bc2s = sqrtf(1.f - powf(p.beta2, (float)p.step));
    }
    for_each_slab_voxel(Ds, H, W, [&](size_t idx, int x, int y, int zl) {
        const int z = p.z_off + zl;
        float f[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for (int c = 0; c < NDIM; ++c) f[c] = ld_stream_f(p.flow_in + (size_t)c * slab + idx);
        float px, py, pz = 0.f;
        if (NDIM == 3) { pz = flow_pos(az, z, f[0]); py = flow_pos(ay, y, f[1]); px = flow_pos(ax, x, f[2]); }
        else { py = flow_pos(ay, y, f[0]); px = flow_pos(ax, x, f[1]); }
        const Sample<NDIM> sp = sample_zero_pad<NDIM, true>(p.moving, D, H, W, px, py, pz);
        const float g[3] = {sp.g[0], sp.g[1], NDIM == 3 ? sp.g[NDIM - 1] : 0.f};
        const float r = ld_stream_f(resid + idx);
#pragma unroll
        for (int c = 0; c < NDIM; ++c) {
            float gr = r * g[NDIM - 1 - c];          // channel c <-> sampling coordinate NDIM-1-c
            if (p.lambda != 0.f) {
                float st = 0.f;
                if (x + 1 < W) st -= sw[0] * (flow_at<NDIM>(p, c, zl, y, x + 1) - f[c]);
                if (x > 0) st += sw[0] * (f[c] - flow_at<NDIM>(p, c, zl, y, x - 1));
                if (y + 1 < H) st -= sw[1] * (flow_at<NDIM>(p, c, zl, y + 1, x) - f[c]);
                if (y > 0) st += sw[1] * (f[c] - flow_at<NDIM>(p, c, zl, y - 1, x));
                if (NDIM == 3) {
                    if (z + 1 < D) st -= sw[2] * (flow_at<NDIM>(p, c, zl + 1, y, x) - f[c]);
                    if (z > 0) st += sw[2] * (f[c] - flow_at<NDIM>(p, c, zl - 1, y, x));
                }
                gr += st;
            }
            const size_t o = (size_t)c * slab + idx;
            float nv;
            if (p.optimiser == TRB_OPT_SGD) {
                nv = f[c] - p.lr * gr;
            } else {
                float m = p.adam_m[o], v = p.adam_v[o];
                m = p.beta1 * m + (1.f - p.beta1) * gr;
                v = p.beta2 * v + (1.f - p.beta2) * gr * gr;
                p.adam_m[o] = m; p.adam_v[o] = v;
                nv = f[c] - (p.lr / bc1) * (m / (sqrtf(v) / bc2s + p.eps));
            }
            p.flow_out[o] = nv;
        }
    });
}

// ---- fused single-pass epoch (3-D) -------------------------------------------------------------------------
// One kernel per epoch instead of two.  A CTA owns a 32x8 (x,y) tile and marches along z over a chunk of
// slices: the z-1 / z / z+1 flow values of a voxel are the thread's own registers (sliding window), the x+-1 /
// y+-1 neighbours come from a double-buffered shared tile with a one-cell halo, so every flow value is read from
// global once (+ halo).  The similarity moments the NEXT epoch's coefficients need are those of the flow this
// kernel writes, so (NEXT) the new position is sampled right away while its cells are still in L1; the MSE-only
// case (coefficients independent of the moments) accumulates the moments of the incoming flow instead.
//   moments[0..4]: in  = similarity sums of flow_in over the whole volume (all-reduced when sharded; NEXT only)
//                  out = this slab's sums of flow_out (NEXT) / of flow_in (!NEXT)
//   moments[5]   : out = this slab's smoothness sum of flow_in
// loss_log[e] = similarity(flow_e) + lambda * smooth(flow_e) is therefore complete one call later: the prologue
// of epoch e+1 (or trb_flow_direct_finish after the last epoch) writes it; NEXT keeps similarity(flow_e) in a
// workspace scalar meanwhile.  Algorithmic traffic: 32 B/voxel (SGD), 80 B/voxel (Adam).
constexpr int kTX = 32, kTY = 8;

// halo values may live in a neighbour GPU's memory and are rewritten every epoch: plain (coherent) load, not __ldg
__device__ __forceinline__ float ld_halo(const float *p) { return *reinterpret_cast<const volatile float *>(p); }

// MUFU.SQRT (2 ulp): the Adam denominator does not need the ~10-instruction IEEE sequence with its slow-path branch
__device__ __forceinline__ float sqrt_approx(float v)
{
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(v));
    return r;
}

__device__ __forceinline__ void direct_log_losses(const DirectParams &p, const double *m, bool next, bool new_epoch,
                                                  double *stash)
{
    const double n = (double)p.D * p.H * p.W;
    const double sim = loss_coefficients(n, m[0], m[1], m[2], m[3], m[4], (double)p.w_mse, (double)p.w_ncc).loss;
    if (!p.loss_log) return;
    const bool prev = p.complete_prev && p.epoch > 0;
    if (next) {
        if (prev) p.loss_log[p.epoch - 1] = (float)(*stash + (double)p.lambda * m[5]);
        if (new_epoch) { *stash = sim; p.loss_log[p.epoch] = (float)sim; }
    } else if (prev) {
        p.loss_log[p.epoch - 1] = (float)(sim + (double)p.lambda * m[5]);
    }
}

#ifndef TRB_STEP_MINB
#define TRB_STEP_MINB 4
#endif
#ifndef TRB_STEP_UNROLL
#define TRB_STEP_UNROLL 1
#endif
constexpr int kStepUnroll = TRB_STEP_UNROLL;
template <bool NEXT, bool ADAM, bool SMOOTH>
__global__ void __launch_bounds__(256, TRB_STEP_MINB) flow_direct_step_kernel(const DirectParams p, const int tiles_x, const int tiles_y,
                                                               const int zc)
{
    const int W = p.W, H = p.H, D = p.D, Ds = p.Ds;
    const int HW = H * W, slab = HW * Ds;              // host guarantees 3*slab < 2^31
    __shared__ float tile[2][3][kTY + 2][kTX + 2];
    __shared__ float coef[3];
    __shared__ double red[kWarps][6];
    if (threadIdx.x == 0) {
        const double n = (double)D * H * W;
        const LossCoef lc = loss_coefficients(n, p.moments[0], p.moments[1], p.moments[2], p.moments[3], p.moments[4],
                                              (double)p.w_mse, (double)p.w_ncc);
        coef[0] = (float)lc.cw; coef[1] = (float)lc.ct; coef[2] = (float)lc.c0;
        if (blockIdx.x == 0) direct_log_losses(p, p.moments, NEXT, true, (double *)p.ticket + 1);
    }
    __syncthreads();
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    // halo cell of the shared tile this thread refreshes every slice (240 cells: 3 channels x (2 rows + 2 columns))
    int hc = 0, hx = 0, hy = 0;
    const bool halo_thread = SMOOTH && threadIdx.x < 240;
    if (halo_thread) {
        hc = threadIdx.x / 80;
        const int r = threadIdx.x - hc * 80;
        if (r < 32) { hy = -1; hx = r; }
        else if (r < 64) { hy = kTY; hx = r - 32; }
        else if (r < 72) { hx = -1; hy = r - 64; }
        else { hx = kTX; hy = r - 72; }
    }
    const int tiles_xy = tiles_x * tiles_y;
    const int chunks = (Ds + zc - 1) / zc;
    const int items = tiles_xy * chunks;
    float s[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const int chunk = item / tiles_xy, t2 = item - chunk * tiles_xy;
        const int by = t2 / tiles_x, bx = t2 - by * tiles_x;
        const int x = bx * kTX + tx, y = by * kTY + ty;
        const bool active = x < W && y < H;
        const int xy = y * W + x;
        const int zl0 = chunk * zc, zl1 = min(zl0 + zc, Ds);
        int hoff = -1;
        if (halo_thread) {
            const int gx = bx * kTX + hx, gy = by * kTY + hy;
            if (gx >= 0 && gx < W && gy >= 0 && gy < H) hoff = hc * slab + gy * W + gx;
        }
        float fm[3] = {0.f, 0.f, 0.f}, fc[3] = {0.f, 0.f, 0.f}, fp[3] = {0.f, 0.f, 0.f}, hcur = 0.f;
        if (active) {
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                fc[c] = ld_stream_f(p.flow_in + c * slab + zl0 * HW + xy);
                if (SMOOTH) {
                    if (zl0 > 0) fm[c] = __ldg(p.flow_in + c * slab + (zl0 - 1) * HW + xy);
                    else if (p.z_off > 0) fm[c] = ld_halo(p.halo_lo + c * p.halo_lo_cs + xy);
                    else fm[c] = fc[c];
                }
            }
        }
        if (hoff >= 0) hcur = __ldg(p.flow_in + hoff + zl0 * HW);
        __syncthreads();                                   // the previous item's readers are done with the tile
#pragma unroll kStepUnroll
        for (int zl = zl0; zl < zl1; ++zl) {
            const int z = p.z_off + zl, b = zl & 1;
            const int o = zl * HW + xy;
            float t = 0.f, am[3] = {0.f, 0.f, 0.f}, av[3] = {0.f, 0.f, 0.f};
            if (active) {
                t = ld_stream_f(p.target + o);
                if (ADAM) {
#pragma unroll
                    for (int c = 0; c < 3; ++c) { am[c] = __ldcs(p.adam_m + c * slab + o); av[c] = __ldcs(p.adam_v + c * slab + o); }
                }
                // next slice into registers while this one is processed
                if (zl + 1 < Ds) {
                    if (SMOOTH || zl + 1 < zl1) {
#pragma unroll
                        for (int c = 0; c < 3; ++c) fp[c] = ld_stream_f(p.flow_in + c * slab + o + HW);
                    }
                } else if (SMOOTH) {
#pragma unroll
                    for (int c = 0; c < 3; ++c) fp[c] = (z + 1 < D) ? ld_halo(p.halo_hi + c * p.halo_hi_cs + xy) : fc[c];
                }
            }
            Cell3 cell;
            if (active)          // the gather goes out before the barrier: its latency overlaps the stencil exchange
                cell = gather_cell3(p.moving, D, H, W, flow_pos(p.ax, x, fc[2]), flow_pos(p.ay, y, fc[1]), flow_pos(p.az, z, fc[0]));
            if (SMOOTH) {
                if (active) {
#pragma unroll
                    for (int c = 0; c < 3; ++c) tile[b][c][ty + 1][tx + 1] = fc[c];
                }
                if (hoff >= 0) {
                    tile[b][hc][hy + 1][hx + 1] = hcur;
                    if (zl + 1 < zl1) hcur = __ldg(p.flow_in + hoff + (zl + 1) * HW);
                }
                __syncthreads();
            }
            if (active) {
                const Sample<3> sp = blend_cell3<true>(cell);
                const float val = sp.val;
                const float *g = sp.g;
                const float r = fmaf(coef[0], val, fmaf(coef[1], t, coef[2]));
                float nv[3];
                float sm = 0.f;
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    float gr = r * g[2 - c];               // channel c <-> sampling coordinate 2-c
                    if (SMOOTH) {
                        const float f = fc[c];
                        const float xm = x > 0 ? tile[b][c][ty + 1][tx] : f, xp = x + 1 < W ? tile[b][c][ty + 1][tx + 2] : f;
                        const float ym = y > 0 ? tile[b][c][ty][tx + 1] : f, yp = y + 1 < H ? tile[b][c][ty + 2][tx + 1] : f;
                        const float zm = fm[c], zp = fp[c];
                        const float dxp = xp - f, dyp = yp - f, dzp = zp - f;
                        float st = p.ssm[0] * ((f - xm) - dxp);
                        st = fmaf(p.ssm[1], (f - ym) - dyp, st);
                        st = fmaf(p.ssm[2], (f - zm) - dzp, st);
                        gr += st;
                        sm = fmaf(p.wsm[0] * dxp, dxp, sm);
                        sm = fmaf(p.wsm[1] * dyp, dyp, sm);
                        sm = fmaf(p.wsm[2] * dzp, dzp, sm);
                    }
                    if (!ADAM) {
                        nv[c] = fc[c] - p.lr * gr;
                    } else {
                        // torch.optim.Adam: p -= lr/bc1 * m / (sqrt(v)/sqrt(bc2) + eps)
                        am[c] = fmaf(p.beta1, am[c], p.ob1 * gr);
                        av[c] = fmaf(p.beta2, av[c], p.ob2 * gr * gr);
                        nv[c] = fmaf(-p.step_size, __fdividef(am[c], fmaf(sqrt_approx(av[c]), p.inv_bc2s, p.eps)), fc[c]);
                    }
                }
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    __stcs(p.flow_out + c * slab + o, nv[c]);
                    if (ADAM) { __stcs(p.adam_m + c * slab + o, am[c]); __stcs(p.adam_v + c * slab + o, av[c]); }
                }
                float wv = val;
                if (NEXT) {
                    const float qz = flow_pos(p.az, z, nv[0]), qy = flow_pos(p.ay, y, nv[1]), qx = flow_pos(p.ax, x, nv[2]);
                    // SGD: the step stays inside the gathered cell almost always; Adam has no registers to keep the cell (measured)
                    wv = ADAM ? sample_zero_pad<3, false>(p.moving, D, H, W, qx, qy, qz).val : sample_near(cell, p.moving, D, H, W, qx, qy, qz);
                }
                s[0] += t; s[1] += wv;
                s[2] = fmaf(t, t, s[2]); s[3] = fmaf(wv, wv, s[3]); s[4] = fmaf(t, wv, s[4]);
                s[5] += sm;
#pragma unroll
                for (int c = 0; c < 3; ++c) { fm[c] = fc[c]; fc[c] = fp[c]; }
            }
        }
    }
    // fp32 per thread (tens of voxels), fp64 above
    if (!grid_sum(s, red, p.partials, p.ticket) || threadIdx.x >= 32) return;
    if (p.peer.world > 1) {                     // sharded: every rank leaves the kernel with the global sums
        __threadfence_system();                 // this rank's flow_out is complete before its sums reach the peers
        peer_allreduce(&red[0][0], 6, p.peer, threadIdx.x);
    }
    if (threadIdx.x < 6) p.moments[threadIdx.x] = red[0][threadIdx.x];
}

// ---- the same epoch with the flow and target tiles staged by TMA (smoothness variants) ---------------------------
// The stencil halo made the register/LDG version pay 168 L1 sectors per 256 voxels (48 of them single-float column
// loads).  Here one elected thread issues, per slice, ONE tensor load of the 3-channel flow tile with its halo
// (box 40 x 10 x 1 x 3 at (x0-4, y0-1, z, 0): 16-byte aligned start, out-of-range rows/columns zero-filled) and one of
// the 32 x 8 target tile into a ring of kStepStages stages; all threads wait on the stage's mbarrier and read centre,
// x/y neighbours, the next slice's centre (z+1) and the target from shared memory.  The ring runs ahead across work
// items, so only the gathers of the moving volume (and Adam's m, v) are register-staged global loads.
constexpr int kStepStages = 4;
constexpr int kSX = kTX + 8, kSY = kTY + 2;              // staged flow tile: 4 extra floats left/right (alignment), 1 row up/down
struct __align__(128) StepStage {
    float flow[3][kSY][kSX];                             // 4800 B
    float pad[16];                                       // next member on a 128-byte boundary
    float tgt[kTY][kTX];                                 // 1024 B
};
constexpr unsigned kStageTx = 3 * kSY * kSX * 4 + kTY * kTX * 4;

struct StepCursor {                                      // position in this CTA's flat sequence of (item, slice)
    int item, i, nsl, x0, y0, zl0;
};
__device__ __forceinline__ void cursor_load(StepCursor &c, int items, int tiles_x, int tiles_xy, int zc, int Ds)
{
    if (c.item >= items) { c.nsl = 0; return; }
    const int chunk = c.item / tiles_xy, t2 = c.item - chunk * tiles_xy;
    const int by = t2 / tiles_x, bx = t2 - by * tiles_x;
    c.x0 = bx * kTX; c.y0 = by * kTY; c.zl0 = chunk * zc;
    c.nsl = min(zc, Ds - c.zl0);
    c.i = 0;
}
__device__ __forceinline__ void cursor_next(StepCursor &c, int items, int tiles_x, int tiles_xy, int zc, int Ds, int stride)
{
    if (++c.i < c.nsl) return;
    c.item += stride;
    cursor_load(c, items, tiles_x, tiles_xy, zc, Ds);
}

template <bool NEXT, bool ADAM>
__global__ void __launch_bounds__(256, 4) flow_direct_step_tma_kernel(const DirectParams p, const int tiles_x, const int tiles_y,
                                                                      const int zc, const __grid_constant__ CUtensorMap map_flow,
                                                                      const __grid_constant__ CUtensorMap map_tgt)
{
    const int W = p.W, H = p.H, D = p.D, Ds = p.Ds;
    const int HW = H * W, slab = HW * Ds;
    __shared__ StepStage stages[kStepStages];
    __shared__ __align__(8) uint64_t full[kStepStages];
    __shared__ float coef[3];
    __shared__ double red[kWarps][6];
    __shared__ bool is_last;
    if (threadIdx.x == 0) {
        for (int i = 0; i < kStepStages; ++i) tma::mbar_init(full + i, 1);
        tma::fence_barrier_init();
        const double n = (double)D * H * W;
        const LossCoef lc = loss_coefficients(n, p.moments[0], p.moments[1], p.moments[2], p.moments[3], p.moments[4],
                                              (double)p.w_mse, (double)p.w_ncc);
        coef[0] = (float)lc.cw; coef[1] = (float)lc.ct; coef[2] = (float)lc.c0;
        if (blockIdx.x == 0) direct_log_losses(p, p.moments, NEXT, true, (double *)p.ticket + 1);
    }
    __syncthreads();
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int tiles_xy = tiles_x * tiles_y;
    const int items = tiles_xy * ((Ds + zc - 1) / zc);
    const int stride = gridDim.x;
    StepCursor cons, prod;
    cons.item = prod.item = blockIdx.x;
    cursor_load(cons, items, tiles_x, tiles_xy, zc, Ds);
    prod = cons;
    unsigned issued = 0, consumed = 0;                   // slices issued / consumed by this CTA: stage = n % kStepStages
    auto issue_one = [&]() {                             // thread 0 only
        StepStage &st = stages[issued % kStepStages];
        uint64_t *bar = full + issued % kStepStages;
        tma::mbar_arrive_expect_tx(bar, kStageTx);
        tma::load_4d(&st.flow[0][0][0], &map_flow, bar, prod.x0 - 4, prod.y0 - 1, prod.zl0 + prod.i, 0);
        tma::load_4d(&st.tgt[0][0], &map_tgt, bar, prod.x0, prod.y0, prod.zl0 + prod.i, 0);
        ++issued;
        cursor_next(prod, items, tiles_x, tiles_xy, zc, Ds, stride);
    };
    if (threadIdx.x == 0)
        for (int k = 0; k < kStepStages && prod.nsl > 0; ++k) issue_one();
    float s[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    while (cons.nsl > 0) {
        // per item: everything that does not change along z
        const int x = cons.x0 + tx, y = cons.y0 + ty;
        const bool active = x < W && y < H;
        const int xy = y * W + x;
        const int nsl = cons.nsl, zl0 = cons.zl0;
        // volume-boundary neighbours: the staged halo holds zeros there; a 0/1 factor on the difference is the
        // replicate boundary (difference 0) without per-slice predicates
        const float mxm = x > 0 ? 1.f : 0.f, mxp = x + 1 < W ? 1.f : 0.f, mym = y > 0 ? 1.f : 0.f, myp = y + 1 < H ? 1.f : 0.f;
        float fprev[3] = {0.f, 0.f, 0.f};
        int o = zl0 * HW + xy;
        for (int i = 0; i < nsl; ++i, o += HW) {
            const int zl = zl0 + i, z = p.z_off + zl;
            const bool last_of_item = i + 1 == nsl;
            const StepStage &st = stages[consumed % kStepStages];
            tma::mbar_wait(full + consumed % kStepStages, (consumed / kStepStages) & 1u);
            const StepStage &nx = stages[(consumed + 1) % kStepStages];
            if (!last_of_item) tma::mbar_wait(full + (consumed + 1) % kStepStages, ((consumed + 1) / kStepStages) & 1u);
            if (active) {
                float fc[3], fm[3], fp[3], am[3] = {0.f, 0.f, 0.f}, av[3] = {0.f, 0.f, 0.f};
#pragma unroll
                for (int c = 0; c < 3; ++c) fc[c] = st.flow[c][ty + 1][tx + 4];
                const Cell3 cell = gather_cell3(p.moving, D, H, W, flow_pos(p.ax, x, fc[2]), flow_pos(p.ay, y, fc[1]), flow_pos(p.az, z, fc[0]));
                // z neighbours: inside an item the previous slice's centre is still in registers and the next one is the
                // next stage's centre; at the item's ends they come from global memory / the neighbour rank's halo slice
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    if (i > 0) fm[c] = fprev[c];
                    else if (zl > 0) fm[c] = __ldg(p.flow_in + c * slab + o - HW);
                    else if (p.z_off > 0) fm[c] = ld_halo(p.halo_lo + c * p.halo_lo_cs + xy);
                    else fm[c] = fc[c];
                    if (!last_of_item) fp[c] = nx.flow[c][ty + 1][tx + 4];
                    else if (zl + 1 < Ds) fp[c] = __ldg(p.flow_in + c * slab + o + HW);
                    else if (z + 1 < D) fp[c] = ld_halo(p.halo_hi + c * p.halo_hi_cs + xy);
                    else fp[c] = fc[c];
                }
                const float t = st.tgt[ty][tx];
                const Sample<3> sp = blend_cell3<true>(cell);
                const float val = sp.val;
                const float r = fmaf(coef[0], val, fmaf(coef[1], t, coef[2]));
                if (ADAM) {                                 // after the gathered cell is consumed: 11 registers fewer live
#pragma unroll
                    for (int c = 0; c < 3; ++c) { am[c] = __ldcs(p.adam_m + c * slab + o); av[c] = __ldcs(p.adam_v + c * slab + o); }
                }
                float nv[3], sm = 0.f;
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const float f = fc[c];
                    const float dxm = (f - st.flow[c][ty + 1][tx + 3]) * mxm, dxp = (st.flow[c][ty + 1][tx + 5] - f) * mxp;
                    const float dym = (f - st.flow[c][ty][tx + 4]) * mym, dyp = (st.flow[c][ty + 2][tx + 4] - f) * myp;
                    const float dzp = fp[c] - f;
                    float stn = p.ssm[0] * (dxm - dxp);
                    stn = fmaf(p.ssm[1], dym - dyp, stn);
                    stn = fmaf(p.ssm[2], (f - fm[c]) - dzp, stn);
                    const float gr = fmaf(r, sp.g[2 - c], stn);             // channel c <-> sampling coordinate 2-c
                    sm = fmaf(p.wsm[0] * dxp, dxp, sm);
                    sm = fmaf(p.wsm[1] * dyp, dyp, sm);
                    sm = fmaf(p.wsm[2] * dzp, dzp, sm);
                    if (!ADAM) {
                        nv[c] = f - p.lr * gr;
                    } else {
                        am[c] = fmaf(p.beta1, am[c], p.ob1 * gr);
                        av[c] = fmaf(p.beta2, av[c], p.ob2 * gr * gr);
                        nv[c] = fmaf(-p.step_size, __fdividef(am[c], fmaf(sqrt_approx(av[c]), p.inv_bc2s, p.eps)), f);
                    }
                }
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    __stcs(p.flow_out + c * slab + o, nv[c]);
                    if (ADAM) { __stcs(p.adam_m + c * slab + o, am[c]); __stcs(p.adam_v + c * slab + o, av[c]); }
                }
                float wv = val;
                if (NEXT) {
                    const float qz = flow_pos(p.az, z, nv[0]), qy = flow_pos(p.ay, y, nv[1]), qx = flow_pos(p.ax, x, nv[2]);
                    // SGD: the step stays inside the gathered cell almost always; Adam has no registers to keep the cell (measured)
                    wv = ADAM ? sample_zero_pad<3, false>(p.moving, D, H, W, qx, qy, qz).val : sample_near(cell, p.moving, D, H, W, qx, qy, qz);
                }
                s[0] += t; s[1] += wv;
                s[2] = fmaf(t, t, s[2]); s[3] = fmaf(wv, wv, s[3]); s[4] = fmaf(t, wv, s[4]);
                s[5] += sm;
#pragma unroll
                for (int c = 0; c < 3; ++c) fprev[c] = fc[c];
            }
            ++consumed;
            __syncthreads();                              // everybody is done with the stage just consumed
            if (threadIdx.x == 0 && prod.nsl > 0) issue_one();
        }
        cons.item += stride;
        cursor_load(cons, items, tiles_x, tiles_xy, zc, Ds);
    }
    // The same sums and order as grid_sum (common.cuh), written out: with the helpers ptxas schedules the main loop of
    // this kernel differently, and the SGD + MSE + smoothness epoch at 256^3 took 211.6 us instead of 203.5 us on a B200
    // (1000 W).
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < 6; ++i) {
        const double v = warp_sum((double)s[i]);
        if (lane == 0) red[warp][i] = v;
    }
    __syncthreads();
    if (threadIdx.x < 6) {
        double v = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
        __stcg(p.partials + (size_t)blockIdx.x * 6 + threadIdx.x, v);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = (atomicAdd(p.ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    if (warp < 6) {
        double v = 0.0;
        for (int b = lane; b < (int)gridDim.x; b += 32) v += __ldcg(p.partials + (size_t)b * 6 + warp);
        v = warp_sum(v);
        if (lane == 0) { p.moments[warp] = v; red[0][warp] = v; }
    }
    if (threadIdx.x == 0) *p.ticket = 0u;
    if (p.peer.world > 1) {                     // sharded: every rank leaves the kernel with the global sums
        __syncthreads();
        if (warp == 0) {
            __threadfence_system();             // this rank's flow_out is complete before its sums reach the peers
            peer_allreduce(&red[0][0], 6, p.peer, lane);
            if (lane < 6) p.moments[lane] = red[0][lane];
        }
    }
}

__global__ void flow_direct_finish_kernel(const DirectParams p, const int next)
{
    if (threadIdx.x == 0 && blockIdx.x == 0) direct_log_losses(p, p.moments, next != 0, false, (double *)p.ticket + 1);
}

constexpr int kDirectMaxBlocks = 4096;

static int direct_grid(size_t n, unsigned &grid)
{
    int sms;
    if (int rc = sm_count(sms)) return rc;
    size_t nb = (n + 255) / 256;
    const size_t cap = (size_t)sms * 8;
    if (nb > cap) nb = cap;
    if (nb > kDirectMaxBlocks) nb = kDirectMaxBlocks;
    grid = (unsigned)(nb < 1 ? 1 : nb);
    return TRB_OK;
}

static int fill_direct(DirectParams &p, int ndim, const float *moving, const float *target, const float *flow_in,
                       const float *halo_lo, const float *halo_hi, int D, int H, int W, int z_off, int Ds,
                       double *moments, void *ws, size_t ws_bytes, float lambda)
{
    if (ndim != 2 && ndim != 3) { set_error("ndim must be 2 or 3"); return TRB_ERR_ARG; }
    if (H < 2 || W < 2 || (ndim == 3 && D < 2)) { set_error("flow needs every axis >= 2"); return TRB_ERR_ARG; }
    if (int rc = check_fast_floor_axes(ndim, D, H, W)) return rc;
    if (!moving || !target || !flow_in || !moments) { set_error("null pointer"); return TRB_ERR_ARG; }
    if ((unsigned long long)(ndim == 3 ? D : 1) * H * W >= (1ull << 31)) { set_error("flow kernels index volumes with 32 bits: D*H*W must stay below 2^31"); return TRB_ERR_ARG; }
    if (ndim == 3 && (z_off < 0 || Ds < 1 || z_off + Ds > D)) { set_error("bad slab [%d,%d) of %d", z_off, z_off + Ds, D); return TRB_ERR_ARG; }
    if (ndim == 3 && lambda != 0.f && ((z_off > 0 && !halo_lo) || (z_off + Ds < D && !halo_hi))) { set_error("interior slab needs both halos"); return TRB_ERR_ARG; }
    if (!ws || ws_bytes < (size_t)(kDirectMaxBlocks * 6 + 2) * sizeof(double)) { set_error("workspace too small"); return TRB_ERR_WORKSPACE; }
    p.moving = moving; p.target = target; p.flow_in = flow_in; p.halo_lo = halo_lo; p.halo_hi = halo_hi;
    p.D = ndim == 3 ? D : 1; p.H = H; p.W = W; p.z_off = ndim == 3 ? z_off : 0; p.Ds = ndim == 3 ? Ds : 1;
    p.moments = moments;
    p.partials = (double *)ws + 2;
    p.ticket = (unsigned *)ws;
    return TRB_OK;
}

}  // namespace trb

using namespace trb;

extern "C" size_t trb_flow_direct_workspace_bytes(void) { return (size_t)(kDirectMaxBlocks * 6 + 2) * sizeof(double); }

extern "C" int trb_flow_direct_stats(int ndim, const float *moving_dev, const float *target_slab_dev, const float *flow_slab_dev,
                                     const float *halo_lo_dev, const float *halo_hi_dev, int D, int H, int W, int z_off, int Ds,
                                     float smooth_lambda, double *moments6_dev, void *workspace_dev, size_t workspace_bytes,
                                     void *stream)
{
    DirectParams p{};
    int rc = fill_direct(p, ndim, moving_dev, target_slab_dev, flow_slab_dev, halo_lo_dev, halo_hi_dev, D, H, W, z_off, Ds,
                         moments6_dev, workspace_dev, workspace_bytes, smooth_lambda);
    if (rc) return rc;
    p.lambda = smooth_lambda;
    unsigned g;
    if ((rc = direct_grid((size_t)p.Ds * H * W, g))) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (ndim == 3) flow_direct_stats_kernel<3><<<g, 256, 0, s>>>(p);
    else flow_direct_stats_kernel<2><<<g, 256, 0, s>>>(p);
    return check_cuda(cudaGetLastError(), "flow_direct_stats");
}

extern "C" int trb_flow_direct_update(int ndim, const float *moving_dev, const float *target_slab_dev,
                                      const float *flow_in_slab_dev, float *flow_out_slab_dev,
                                      const float *halo_lo_dev, const float *halo_hi_dev, int D, int H, int W, int z_off, int Ds,
                                      const double *moments6_dev, float w_mse, float w_ncc, float smooth_lambda, float lr,
                                      int optimiser, float beta1, float beta2, float adam_eps, int step_index,
                                      float *adam_m_dev, float *adam_v_dev, float *loss_log_dev, int epoch, void *stream)
{
    DirectParams p{};
    if (ndim != 2 && ndim != 3) { set_error("ndim must be 2 or 3"); return TRB_ERR_ARG; }
    if (int rc = check_fast_floor_axes(ndim, D, H, W)) return rc;
    if (!moving_dev || !target_slab_dev || !flow_in_slab_dev || !flow_out_slab_dev || !moments6_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    if (flow_in_slab_dev == flow_out_slab_dev) { set_error("update is out of place: flow_out must differ from flow_in"); return TRB_ERR_ARG; }
    if ((unsigned long long)(ndim == 3 ? D : 1) * H * W >= (1ull << 31)) { set_error("flow kernels index volumes with 32 bits: D*H*W must stay below 2^31"); return TRB_ERR_ARG; }
    if (optimiser != TRB_OPT_SGD && optimiser != TRB_OPT_ADAM) { set_error("bad optimiser"); return TRB_ERR_ARG; }
    if (optimiser == TRB_OPT_ADAM && (!adam_m_dev || !adam_v_dev || step_index < 1)) { set_error("Adam needs m, v and step_index >= 1"); return TRB_ERR_ARG; }
    if (ndim == 3 && (z_off < 0 || Ds < 1 || z_off + Ds > D)) { set_error("bad slab"); return TRB_ERR_ARG; }
    if (ndim == 3 && smooth_lambda != 0.f && ((z_off > 0 && !halo_lo_dev) || (z_off + Ds < D && !halo_hi_dev))) { set_error("interior slab needs both halos"); return TRB_ERR_ARG; }
    p.moving = moving_dev; p.target = target_slab_dev; p.flow_in = flow_in_slab_dev; p.flow_out = flow_out_slab_dev;
    p.halo_lo = halo_lo_dev; p.halo_hi = halo_hi_dev;
    p.D = ndim == 3 ? D : 1; p.H = H; p.W = W; p.z_off = ndim == 3 ? z_off : 0; p.Ds = ndim == 3 ? Ds : 1;
    p.moments = const_cast<double *>(moments6_dev);
    p.w_mse = w_mse; p.w_ncc = w_ncc; p.lambda = smooth_lambda; p.lr = lr;
    p.optimiser = optimiser; p.beta1 = beta1; p.beta2 = beta2; p.eps = adam_eps; p.step = step_index;
    p.adam_m = adam_m_dev; p.adam_v = adam_v_dev; p.loss_log = loss_log_dev; p.epoch = epoch;
    unsigned g;
    if (int rc = direct_grid((size_t)p.Ds * H * W, g)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (ndim == 3) flow_direct_update_kernel<3><<<g, 256, 0, s>>>(p);
    else flow_direct_update_kernel<2><<<g, 256, 0, s>>>(p);
    return check_cuda(cudaGetLastError(), "flow_direct_update");
}

extern "C" int trb_flow_direct_update_lncc(int ndim, const float *moving_dev, const float *flow_in_dev, float *flow_out_dev,
                                           const float *resid_dev, int D, int H, int W, const double *moments6_dev,
                                           const double *lncc_stats_dev, float w_mse, float w_ncc, float w_lncc,
                                           float smooth_lambda, float lr, int optimiser, float beta1, float beta2,
                                           float adam_eps, int step_index, float *adam_m_dev, float *adam_v_dev,
                                           float *loss_log_dev, int epoch, void *stream)
{
    DirectParams p{};
    if (ndim != 2 && ndim != 3) { set_error("ndim must be 2 or 3"); return TRB_ERR_ARG; }
    if (ndim == 2) D = 1;
    if (H < 2 || W < 2 || (ndim == 3 && D < 2)) { set_error("flow needs every axis >= 2"); return TRB_ERR_ARG; }
    if (int rc = check_fast_floor_axes(ndim, D, H, W)) return rc;
    if ((unsigned long long)D * H * W >= (1ull << 31)) { set_error("flow kernels index volumes with 32 bits: D*H*W must stay below 2^31"); return TRB_ERR_ARG; }
    if (!moving_dev || !flow_in_dev || !flow_out_dev || !resid_dev || !moments6_dev || !lncc_stats_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    const size_t vol = (size_t)D * H * W, fb = (size_t)ndim * vol * sizeof(float);
    const char *fi = (const char *)flow_in_dev, *fo = (const char *)flow_out_dev, *rr = (const char *)resid_dev;
    if ((fo < fi + fb && fi < fo + fb) || (fo < rr + vol * sizeof(float) && rr < fo + fb)) {
        set_error("update is out of place: flow_out must not overlap flow_in or the residual");
        return TRB_ERR_ARG;
    }
    if (optimiser != TRB_OPT_SGD && optimiser != TRB_OPT_ADAM) { set_error("bad optimiser"); return TRB_ERR_ARG; }
    if (optimiser == TRB_OPT_ADAM && (!adam_m_dev || !adam_v_dev || step_index < 1)) { set_error("Adam needs m, v and step_index >= 1"); return TRB_ERR_ARG; }
    p.moving = moving_dev; p.flow_in = flow_in_dev; p.flow_out = flow_out_dev;
    p.D = D; p.H = H; p.W = W; p.z_off = 0; p.Ds = D;
    p.moments = const_cast<double *>(moments6_dev);
    p.w_mse = w_mse; p.w_ncc = w_ncc; p.lambda = smooth_lambda; p.lr = lr;
    p.optimiser = optimiser; p.beta1 = beta1; p.beta2 = beta2; p.eps = adam_eps; p.step = step_index;
    p.adam_m = adam_m_dev; p.adam_v = adam_v_dev; p.loss_log = loss_log_dev; p.epoch = epoch;
    unsigned g;
    if (int rc = direct_grid(vol, g)) return rc;
    cudaStream_t s = (cudaStream_t)stream;
    if (ndim == 3) flow_direct_update_lncc_kernel<3><<<g, 256, 0, s>>>(p, resid_dev, lncc_stats_dev, w_lncc);
    else flow_direct_update_lncc_kernel<2><<<g, 256, 0, s>>>(p, resid_dev, lncc_stats_dev, w_lncc);
    return check_cuda(cudaGetLastError(), "flow_direct_update_lncc");
}

namespace trb {
static int g_step_no_tma = 0;       // trb_flow_direct_set_path: 1 = register-staged kernel for the smoothness variants too (A/B)
template <bool NEXT, bool ADAM>
static void launch_step(const DirectParams &p, bool smooth, unsigned grid, int tiles_x, int tiles_y, int zc, cudaStream_t s)
{
    if (smooth) flow_direct_step_kernel<NEXT, ADAM, true><<<grid, 256, 0, s>>>(p, tiles_x, tiles_y, zc);
    else flow_direct_step_kernel<NEXT, ADAM, false><<<grid, 256, 0, s>>>(p, tiles_x, tiles_y, zc);
}
template <bool NEXT, bool ADAM>
static int step_occupancy()
{
    int a = 0, b = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&a, flow_direct_step_kernel<NEXT, ADAM, true>, 256, 0);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, flow_direct_step_kernel<NEXT, ADAM, false>, 256, 0);
    const int o = a < b ? a : b;
    return o < 1 ? 1 : o;
}
}  // namespace trb

extern "C" void trb_flow_direct_set_path(int no_tma) { trb::g_step_no_tma = no_tma ? 1 : 0; }

static int flow_direct_step_impl(const float *moving_dev, const float *target_slab_dev,
                                    const float *flow_in_slab_dev, float *flow_out_slab_dev,
                                    const float *halo_lo_dev, const float *halo_hi_dev, int D, int H, int W, int z_off, int Ds,
                                    double *moments6_dev, float w_mse, float w_ncc, float smooth_lambda, float lr,
                                    int optimiser, float beta1, float beta2, float adam_eps, int step_index,
                                    float *adam_m_dev, float *adam_v_dev, float *loss_log_dev, int epoch, int complete_prev,
                                    void *workspace_dev, size_t workspace_bytes, void *stream,
                                    long long halo_lo_cs, long long halo_hi_cs, const PeerExchange *peer)
{
    DirectParams p{};
    int rc = fill_direct(p, 3, moving_dev, target_slab_dev, flow_in_slab_dev, halo_lo_dev, halo_hi_dev, D, H, W, z_off, Ds,
                         moments6_dev, workspace_dev, workspace_bytes, smooth_lambda);
    if (rc) return rc;
    if (!flow_out_slab_dev || flow_in_slab_dev == flow_out_slab_dev) { set_error("step is out of place: flow_out must differ from flow_in"); return TRB_ERR_ARG; }
    if (optimiser != TRB_OPT_SGD && optimiser != TRB_OPT_ADAM) { set_error("bad optimiser"); return TRB_ERR_ARG; }
    if (optimiser == TRB_OPT_ADAM && (!adam_m_dev || !adam_v_dev || step_index < 1)) { set_error("Adam needs m, v and step_index >= 1"); return TRB_ERR_ARG; }
    if (3ull * (unsigned long long)Ds * H * W >= (1ull << 31) || (unsigned long long)D * H * W >= (1ull << 31)) {
        set_error("fused step needs 3*Ds*H*W < 2^31 (use stats + update)");
        return TRB_ERR_ARG;
    }
    if (epoch < 0) { set_error("bad epoch"); return TRB_ERR_ARG; }
    p.flow_out = flow_out_slab_dev;
    p.w_mse = w_mse; p.w_ncc = w_ncc; p.lambda = smooth_lambda; p.lr = lr;
    p.optimiser = optimiser; p.beta1 = beta1; p.beta2 = beta2; p.eps = adam_eps; p.step = step_index;
    p.adam_m = adam_m_dev; p.adam_v = adam_v_dev; p.loss_log = loss_log_dev; p.epoch = epoch;
    p.complete_prev = complete_prev;
    p.halo_lo_cs = (int)(halo_lo_cs > 0 ? halo_lo_cs : (long long)H * W);
    p.halo_hi_cs = (int)(halo_hi_cs > 0 ? halo_hi_cs : (long long)H * W);
    if (peer) p.peer = *peer;
    p.ax.d = (float)(W - 1); p.ay.d = (float)(H - 1); p.az.d = (float)(D - 1);
    p.ax.r = 1.f / p.ax.d; p.ay.r = 1.f / p.ay.d; p.az.r = 1.f / p.az.d;       // IEEE: what __frcp_rn gives on the device
    const double dims[3] = {(double)W, (double)H, (double)D};
    for (int a = 0; a < 3; ++a) {                                             // smooth_weight<3>, on the host
        double n = 3.0;
        for (int k = 0; k < 3; ++k) n *= (k == a) ? dims[k] - 1.0 : dims[k];
        p.wsm[a] = (float)(1.0 / (n * 3.0));
        p.ssm[a] = 2.f * smooth_lambda * p.wsm[a];
    }
    p.step_size = lr; p.inv_bc2s = 1.f; p.ob1 = 1.f - beta1; p.ob2 = 1.f - beta2;
    if (optimiser == TRB_OPT_ADAM) {
        p.step_size = lr / (1.f - powf(beta1, (float)step_index));
        p.inv_bc2s = 1.f / sqrtf(1.f - powf(beta2, (float)step_index));
    }
    const bool next = w_ncc != 0.f, adam = optimiser == TRB_OPT_ADAM, smooth = smooth_lambda != 0.f;
    int sms;
    if ((rc = sm_count(sms))) return rc;
    static int occ[2][2] = {{0, 0}, {0, 0}};
    int &oc = occ[next][adam];
    if (!oc) oc = next ? (adam ? step_occupancy<true, true>() : step_occupancy<true, false>())
                       : (adam ? step_occupancy<false, true>() : step_occupancy<false, false>());
    const int tiles_x = (W + kTX - 1) / kTX, tiles_y = (H + kTY - 1) / kTY;
    int cap = sms * oc;
    if (cap > kDirectMaxBlocks) cap = kDirectMaxBlocks;
    // z-chunk length: long chunks amortise the chunk prologue, short ones balance the grid (>= ~6 items per CTA)
    int zc = 32;
    while (zc > 4 && (long long)tiles_x * tiles_y * ((p.Ds + zc - 1) / zc) < 6ll * cap) zc >>= 1;
    const long long items = (long long)tiles_x * tiles_y * ((p.Ds + zc - 1) / zc);
    const unsigned grid = (unsigned)(items < cap ? items : cap);
    cudaStream_t s = (cudaStream_t)stream;
    // smoothness variants: flow + halo and target tiles staged by TMA (needs 16-byte row pitch and base alignment)
    // (Adam + NCC is the one variant where the register-staged kernel measures 2 % faster: 64 registers are too few)
    if (smooth && !(next && adam) && !g_step_no_tma && W % 4 == 0 && W >= kSX && H >= kSY && ((uintptr_t)flow_in_slab_dev & 15) == 0 && ((uintptr_t)target_slab_dev & 15) == 0) {
        CUtensorMap map_flow, map_tgt;
        const cuuint64_t fdims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)p.Ds, 3};
        const cuuint64_t fstr[3] = {(cuuint64_t)W * 4, (cuuint64_t)W * H * 4, (cuuint64_t)W * H * p.Ds * 4};
        const cuuint32_t fbox[4] = {(cuuint32_t)kSX, (cuuint32_t)kSY, 1, 3};
        const cuuint64_t tdims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)p.Ds, 1};
        const cuuint32_t tbox[4] = {(cuuint32_t)kTX, (cuuint32_t)kTY, 1, 1};
        if (tma::make_map_f32(&map_flow, flow_in_slab_dev, fdims, fstr, fbox) && tma::make_map_f32(&map_tgt, target_slab_dev, tdims, fstr, tbox)) {
            int occ_t = 4;
            const unsigned tgrid = (unsigned)(items < (long long)sms * occ_t ? items : (long long)sms * occ_t);
            if (next) { if (adam) flow_direct_step_tma_kernel<true, true><<<tgrid, 256, 0, s>>>(p, tiles_x, tiles_y, zc, map_flow, map_tgt);
                        else flow_direct_step_tma_kernel<true, false><<<tgrid, 256, 0, s>>>(p, tiles_x, tiles_y, zc, map_flow, map_tgt); }
            else { if (adam) flow_direct_step_tma_kernel<false, true><<<tgrid, 256, 0, s>>>(p, tiles_x, tiles_y, zc, map_flow, map_tgt);
                   else flow_direct_step_tma_kernel<false, false><<<tgrid, 256, 0, s>>>(p, tiles_x, tiles_y, zc, map_flow, map_tgt); }
            return check_cuda(cudaGetLastError(), "flow_direct_step(tma)");
        }
    }
    if (next) { if (adam) launch_step<true, true>(p, smooth, grid, tiles_x, tiles_y, zc, s); else launch_step<true, false>(p, smooth, grid, tiles_x, tiles_y, zc, s); }
    else { if (adam) launch_step<false, true>(p, smooth, grid, tiles_x, tiles_y, zc, s); else launch_step<false, false>(p, smooth, grid, tiles_x, tiles_y, zc, s); }
    return check_cuda(cudaGetLastError(), "flow_direct_step");
}

extern "C" int trb_flow_direct_step(const float *moving_dev, const float *target_slab_dev,
                                    const float *flow_in_slab_dev, float *flow_out_slab_dev,
                                    const float *halo_lo_dev, const float *halo_hi_dev, int D, int H, int W, int z_off, int Ds,
                                    double *moments6_dev, float w_mse, float w_ncc, float smooth_lambda, float lr,
                                    int optimiser, float beta1, float beta2, float adam_eps, int step_index,
                                    float *adam_m_dev, float *adam_v_dev, float *loss_log_dev, int epoch, int complete_prev,
                                    void *workspace_dev, size_t workspace_bytes, void *stream)
{
    return flow_direct_step_impl(moving_dev, target_slab_dev, flow_in_slab_dev, flow_out_slab_dev, halo_lo_dev, halo_hi_dev,
                                 D, H, W, z_off, Ds, moments6_dev, w_mse, w_ncc, smooth_lambda, lr, optimiser, beta1, beta2,
                                 adam_eps, step_index, adam_m_dev, adam_v_dev, loss_log_dev, epoch, complete_prev,
                                 workspace_dev, workspace_bytes, stream, 0, 0, nullptr);
}

extern "C" int trb_flow_direct_step_peer(const float *moving_dev, const float *target_slab_dev,
                                         const float *flow_in_slab_dev, float *flow_out_slab_dev,
                                         const float *halo_lo_dev, long long halo_lo_channel_stride,
                                         const float *halo_hi_dev, long long halo_hi_channel_stride,
                                         int D, int H, int W, int z_off, int Ds,
                                         double *moments6_dev, float w_mse, float w_ncc, float smooth_lambda, float lr,
                                         int optimiser, float beta1, float beta2, float adam_eps, int step_index,
                                         float *adam_m_dev, float *adam_v_dev, float *loss_log_dev, int epoch, int complete_prev,
                                         void *const *mailbox_ptrs, int rank, int world, unsigned long long seq,
                                         void *workspace_dev, size_t workspace_bytes, void *stream)
{
    if (world < 1 || world > 8 || rank < 0 || rank >= world || !mailbox_ptrs || seq < 1) { set_error("bad peer set (world 1..8, seq >= 1)"); return TRB_ERR_ARG; }
    if (halo_lo_channel_stride >= (1ll << 31) || halo_hi_channel_stride >= (1ll << 31)) { set_error("halo channel stride too large"); return TRB_ERR_ARG; }
    PeerExchange px{};
    for (int r = 0; r < world; ++r) {
        if (!mailbox_ptrs[r]) { set_error("null mailbox pointer for rank %d", r); return TRB_ERR_ARG; }
        px.mailbox[r] = (double *)mailbox_ptrs[r];
    }
    px.rank = rank; px.world = world; px.seq = seq;
    return flow_direct_step_impl(moving_dev, target_slab_dev, flow_in_slab_dev, flow_out_slab_dev, halo_lo_dev, halo_hi_dev,
                                 D, H, W, z_off, Ds, moments6_dev, w_mse, w_ncc, smooth_lambda, lr, optimiser, beta1, beta2,
                                 adam_eps, step_index, adam_m_dev, adam_v_dev, loss_log_dev, epoch, complete_prev,
                                 workspace_dev, workspace_bytes, stream, halo_lo_channel_stride, halo_hi_channel_stride, &px);
}

extern "C" int trb_flow_direct_finish(const double *moments6_dev, int D, int H, int W, float w_mse, float w_ncc,
                                      float smooth_lambda, float *loss_log_dev, int epochs_done,
                                      void *workspace_dev, size_t workspace_bytes, void *stream)
{
    if (!moments6_dev || !workspace_dev || workspace_bytes < 2 * sizeof(double)) { set_error("null pointer / workspace"); return TRB_ERR_ARG; }
    if (epochs_done < 1 || !loss_log_dev) return TRB_OK;
    DirectParams p{};
    p.D = D; p.H = H; p.W = W;
    p.moments = const_cast<double *>(moments6_dev);
    p.ticket = (unsigned *)workspace_dev;
    p.w_mse = w_mse; p.w_ncc = w_ncc; p.lambda = smooth_lambda; p.loss_log = loss_log_dev; p.epoch = epochs_done;
    p.complete_prev = 1;
    flow_direct_finish_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(p, w_ncc != 0.f ? 1 : 0);
    return check_cuda(cudaGetLastError(), "flow_direct_finish");
}
