// lncc.cu — local (windowed) normalised cross-correlation and its gradient (sm_100a).
//
// VoxelMorph's NCC with the sign turned so the loss is >= 0.  For target I, warped J (one channel, N pairs never mixed
// in a window), an odd window win, nd spatial axes, n = win^nd and zero-padded box sums S_X = conv(X, ones, pad win/2):
//   A = S_IJ - S_I S_J / n,   B = S_II - S_I^2 / n,   C = S_JJ - S_J^2 / n,   cc = A^2 / (B C + eps)
//   loss = 1 - mean over every voxel of every pair of cc.
// Out-of-volume positions count as zeros and n stays fixed, as in VoxelMorph.  The gradient w.r.t. J is again a box
// filter, of three per-voxel coefficient fields (den = B C + eps):
//   gamma = 2 A / den,  beta = -A^2 B / den^2,  alpha = -gamma S_I / n - 2 beta S_J / n
//   dL/dJ = -(1/N_vox) (box(alpha) + 2 J box(beta) + I box(gamma))
// lncc_forward forms the five box sums and writes alpha, beta, gamma and the loss; lncc_backward forms the three box sums
// and writes dL/dJ times a caller scale, optionally plus the pointwise MSE / global NCC gradient cw J + ct I + c0.
//
// One engine serves both: a CTA owns a 32 x 8 (x, y) output tile and marches along z over a chunk of slices.  Per input
// slice it stages the tile plus a win/2 halo in shared memory, sums along x (rows of the halo included), then along y,
// and keeps that slice's 2-D window sums in a shared ring of win planes (each thread reads and writes only its own
// column of the ring).  An output sum adds its win planes in index order.  Every window sum is therefore formed in one
// fixed order, whatever the chunking, and there is no running add-and-subtract along z to drift over long volumes.
// 2-D is the same engine with a one-plane ring.  Algorithmic traffic: forward 20 B/voxel (I, J read; alpha, beta, gamma
// written), backward 24 B/voxel (alpha, beta, gamma, I, J read; dL/dJ written).
#include "common.cuh"

namespace trb {

constexpr int kLTX = 32, kLTY = 8;
constexpr int kLnccMaxBlocks = 2048;      // partial rows of the workspace (trb_lncc_workspace_bytes)
constexpr int kLnccMaxWin = 15;

struct LnccArgs {
    const float *tgt, *wrp;     // I, J: [N][D][H][W]
    const float *coef;          // alpha, beta, gamma: [3][N][D][H][W] (backward input)
    float *out;                 // forward: alpha, beta, gamma (coef layout); backward: dL/dJ [N][D][H][W]
    int N, D, H, W, r, rz;      // window half-widths in (x, y) and z (0 in 2-D)
    int tiles_x, tiles_y, zc, chunks;
    float n, eps, gscale;       // gscale: -scale / N_vox (backward)
    double nvox;
    const double *moments;      // backward: the five global moments of (I, J) for the pointwise MSE / NCC term, or NULL
    float w_mse, w_ncc;
    double *stats, *partials;
    unsigned *ticket;
};

__host__ __device__ constexpr int lncc_in(bool fwd) { return fwd ? 2 : 3; }     // staged inputs per voxel
__host__ __device__ constexpr int lncc_q(bool fwd) { return fwd ? 5 : 3; }      // box sums per voxel

static size_t lncc_smem_bytes(bool fwd, int r, int rz)
{
    const int tyh = kLTY + 2 * r, txh = kLTX + 2 * r;
    return sizeof(float) * ((size_t)lncc_in(fwd) * tyh * txh + (size_t)lncc_q(fwd) * tyh * kLTX +
                            (size_t)(2 * rz + 1) * lncc_q(fwd) * kLTX * kLTY);
}

template <bool FWD>
__global__ void __launch_bounds__(kThreads) lncc_kernel(const LnccArgs a)
{
    constexpr int QI = lncc_in(FWD), Q = lncc_q(FWD), TP = kLTX * kLTY;
    extern __shared__ float smem[];
    const int r = a.r, rz = a.rz, win = 2 * r + 1, wz = 2 * rz + 1;
    const int tyh = kLTY + 2 * r, txh = kLTX + 2 * r;
    float *tin = smem;                                  // [QI][tyh][txh]
    float *xs = tin + QI * tyh * txh;                   // [Q][tyh][32]
    float *ring = xs + Q * tyh * kLTX;                  // [wz][Q][256]
    __shared__ float coef[3];
    if (!FWD) {
        if (threadIdx.x == 0) {
            float c[3] = {0.f, 0.f, 0.f};
            if (a.moments) {
                const double *m = a.moments;
                const LossCoef lc = loss_coefficients((double)a.D * a.H * a.W, m[0], m[1], m[2], m[3], m[4],
                                                      (double)a.w_mse, (double)a.w_ncc);
                c[0] = (float)lc.cw; c[1] = (float)lc.ct; c[2] = (float)lc.c0;
            }
            coef[0] = c[0]; coef[1] = c[1]; coef[2] = c[2];
        }
        __syncthreads();
    }
    const int W = a.W, H = a.H, D = a.D;
    const size_t HW = (size_t)H * W, vol = HW * D, all = vol * a.N;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const long long items = (long long)a.N * a.chunks * a.tiles_y * a.tiles_x;
    double acc = 0.0;
    for (long long item = blockIdx.x; item < items; item += gridDim.x) {
        long long t = item;
        const int bx = (int)(t % a.tiles_x); t /= a.tiles_x;
        const int by = (int)(t % a.tiles_y); t /= a.tiles_y;
        const int chunk = (int)(t % a.chunks);
        const int pair = (int)(t / a.chunks);
        const int x0 = bx * kLTX, y0 = by * kLTY, z0 = chunk * a.zc, z1 = min(z0 + a.zc, D);
        const int x = x0 + tx, y = y0 + ty;
        const bool active = x < W && y < H;
        const size_t pbase = (size_t)pair * vol;
        for (int zi = z0 - rz; zi < z1 + rz; ++zi) {
            float *rs = ring + ((zi - z0 + rz) % wz) * Q * TP;
            if (zi < 0 || zi >= D) {                     // a plane of the zero padding (uniform over the CTA)
#pragma unroll
                for (int q = 0; q < Q; ++q) rs[q * TP + threadIdx.x] = 0.f;
            } else {
                const size_t sbase = pbase + (size_t)zi * HW;
                for (int e = threadIdx.x; e < tyh * txh; e += kThreads) {
                    const int cy = e / txh, cx = e - cy * txh;
                    const int gx = x0 - r + cx, gy = y0 - r + cy;
                    const bool in = (unsigned)gx < (unsigned)W && (unsigned)gy < (unsigned)H;
                    const size_t o = sbase + (size_t)gy * W + gx;
                    if (FWD) {
                        tin[e] = in ? __ldg(a.tgt + o) : 0.f;
                        tin[tyh * txh + e] = in ? __ldg(a.wrp + o) : 0.f;
                    } else {
#pragma unroll
                        for (int q = 0; q < 3; ++q) tin[q * tyh * txh + e] = in ? __ldg(a.coef + q * all + o) : 0.f;
                    }
                }
                __syncthreads();                         // tile staged; the previous slice's y sums are read
                for (int ry = ty; ry < tyh; ry += kLTY) {
                    float s[Q];
#pragma unroll
                    for (int q = 0; q < Q; ++q) s[q] = 0.f;
                    const float *row = tin + ry * txh + tx;
                    for (int k = 0; k < win; ++k) {
                        if (FWD) {
                            const float i = row[k], j = row[tyh * txh + k];
                            s[0] += i; s[1] += j;
                            s[2] = fmaf(i, i, s[2]); s[3] = fmaf(j, j, s[3]); s[4] = fmaf(i, j, s[4]);
                        } else {
#pragma unroll
                            for (int q = 0; q < Q; ++q) s[q] += row[q * tyh * txh + k];
                        }
                    }
#pragma unroll
                    for (int q = 0; q < Q; ++q) xs[(q * tyh + ry) * kLTX + tx] = s[q];
                }
                __syncthreads();                         // x sums complete; the staged tile is free again
#pragma unroll
                for (int q = 0; q < Q; ++q) {
                    float s = 0.f;
                    for (int k = 0; k < win; ++k) s += xs[(q * tyh + ty + k) * kLTX + tx];
                    rs[q * TP + threadIdx.x] = s;
                }
            }
            const int z = zi - rz;
            if (z < z0) continue;
            float S[Q];
#pragma unroll
            for (int q = 0; q < Q; ++q) S[q] = 0.f;
            int sl = (z - z0) % wz;                      // slot of plane z - rz
            for (int k = 0; k < wz; ++k) {               // planes z - rz .. z + rz, in that order
                const float *p = ring + sl * Q * TP + threadIdx.x;
#pragma unroll
                for (int q = 0; q < Q; ++q) S[q] += p[q * TP];
                sl = sl + 1 == wz ? 0 : sl + 1;
            }
            if (!active) continue;
            const size_t o = pbase + (size_t)z * HW + (size_t)y * W + x;
            if (FWD) {
                const float n = a.n;
                const float SI = S[0], SJ = S[1], SII = S[2], SJJ = S[3], SIJ = S[4];
                const float A = SIJ - SI * SJ / n, B = SII - SI * SI / n, C = SJJ - SJ * SJ / n;
                const float den = B * C + a.eps;
                const float cc = A * A / den;
                const float gam = 2.f * A / den;
                const float bet = -cc * (B / den);
                const float alp = -gam * SI / n - 2.f * bet * SJ / n;
                a.out[o] = alp;
                a.out[all + o] = bet;
                a.out[2 * all + o] = gam;
                acc += (double)cc;
            } else {
                const float iv = __ldg(a.tgt + o), jv = __ldg(a.wrp + o);
                const float g = a.gscale * (S[0] + 2.f * jv * S[1] + iv * S[2]);
                a.out[o] = g + fmaf(coef[0], jv, fmaf(coef[1], iv, coef[2]));
            }
        }
    }
    if (FWD) {
        __shared__ double red[kWarps][1];
        const double v[1] = {acc};
        if (grid_sum(v, red, a.partials, a.ticket) && threadIdx.x == 0) {
            a.stats[0] = red[0][0];
            a.stats[1] = 1.0 - red[0][0] / a.nvox;
        }
    }
}

static bool overlap(const void *p, size_t pn, const void *q, size_t qn)
{
    const char *a = (const char *)p, *b = (const char *)q;
    return a && b && a < b + qn && b < a + pn;
}

// shape and window rules shared by both calls; fills the launch-invariant fields
static int lncc_setup(LnccArgs &a, int ndim, int N, int D, int H, int W, int win)
{
    if (ndim != 2 && ndim != 3) { set_error("ndim must be 2 or 3 (got %d)", ndim); return TRB_ERR_ARG; }
    if (ndim == 2) D = 1;
    if (win < 3 || win > kLnccMaxWin || win % 2 == 0) {
        set_error("LNCC window must be odd and in [3, %d] (got %d)", kLnccMaxWin, win);
        return TRB_ERR_UNSUPPORTED;
    }
    if (N < 1 || D < 1 || H < 1 || W < 1) { set_error("bad shape N=%d %dx%dx%d", N, D, H, W); return TRB_ERR_ARG; }
    if ((unsigned long long)D * H * W >= (1ull << 31)) { set_error("LNCC kernels need D*H*W < 2^31"); return TRB_ERR_ARG; }
    if (int rc = check_fast_floor_axes(ndim, D, H, W)) return rc;
    a.N = N; a.D = D; a.H = H; a.W = W;
    a.r = win / 2; a.rz = ndim == 3 ? win / 2 : 0;
    a.n = (float)(ndim == 3 ? win * win * win : win * win);
    a.nvox = (double)N * D * H * W;
    a.tiles_x = (W + kLTX - 1) / kLTX; a.tiles_y = (H + kLTY - 1) / kLTY;
    return TRB_OK;
}

template <bool FWD>
static int lncc_launch(LnccArgs &a, cudaStream_t s)
{
    const size_t smem = lncc_smem_bytes(FWD, a.r, a.rz);
    int dev = 0, sms = 0;
    if (int rc = check_cuda(cudaGetDevice(&dev), "cudaGetDevice")) return rc;
    if (int rc = sm_count(sms)) return rc;
    // per device: the shared-memory opt-in for the widest window (one value for every launch of the kernel); per
    // device and window: the resident CTAs per SM
    static bool opted[64] = {};
    if (!opted[dev & 63]) {
        const int most = (int)lncc_smem_bytes(FWD, kLnccMaxWin / 2, kLnccMaxWin / 2);
        if (int rc = check_cuda(cudaFuncSetAttribute(lncc_kernel<FWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, most),
                                "lncc shared memory")) return rc;
        opted[dev & 63] = true;
    }
    static int occ[64][kLnccMaxWin + 1] = {};
    int &oc = occ[dev & 63][2 * a.r + (a.rz ? 1 : 0)];
    if (!oc) {
        if (int rc = check_cuda(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&oc, lncc_kernel<FWD>, kThreads, smem), "lncc occupancy"))
            return rc;
        if (oc < 1) oc = 1;
    }
    long long cap = (long long)sms * oc;
    if (cap > kLnccMaxBlocks) cap = kLnccMaxBlocks;
    // z-chunk length: long chunks amortise the 2 rz halo planes, short ones give every CTA several items
    const long long tiles = (long long)a.N * a.tiles_x * a.tiles_y;
    int zc = 64;
    while (zc > 8 && tiles * ((a.D + zc - 1) / zc) < 4 * cap) zc >>= 1;
    a.zc = zc;
    a.chunks = (a.D + zc - 1) / zc;
    const long long items = tiles * a.chunks;
    const unsigned grid = (unsigned)(items < cap ? items : cap);
    lncc_kernel<FWD><<<grid, kThreads, smem, s>>>(a);
    return check_cuda(cudaGetLastError(), FWD ? "lncc_forward" : "lncc_backward");
}

}  // namespace trb

using namespace trb;

extern "C" size_t trb_lncc_workspace_bytes(void) { return (size_t)(8 + kLnccMaxBlocks) * sizeof(double); }

extern "C" int trb_lncc_forward(int ndim, const float *target_dev, const float *warped_dev, int N, int D, int H, int W, int win,
                                float eps, float *coef_dev, double *stats_dev, void *workspace_dev, size_t workspace_bytes,
                                void *stream)
{
    LnccArgs a{};
    if (int rc = lncc_setup(a, ndim, N, D, H, W, win)) return rc;
    if (!target_dev || !warped_dev || !coef_dev || !stats_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    if (!(eps > 0.f) || !isfinite(eps)) { set_error("eps must be finite and > 0"); return TRB_ERR_ARG; }
    if (!workspace_dev || workspace_bytes < trb_lncc_workspace_bytes()) {
        set_error("workspace too small: need %zu bytes (trb_lncc_workspace_bytes)", trb_lncc_workspace_bytes());
        return TRB_ERR_WORKSPACE;
    }
    const size_t nb = (size_t)a.nvox * sizeof(float);
    if (overlap(coef_dev, 3 * nb, target_dev, nb) || overlap(coef_dev, 3 * nb, warped_dev, nb) ||
        overlap(stats_dev, 2 * sizeof(double), coef_dev, 3 * nb)) {
        set_error("lncc_forward: an output overlaps an input");
        return TRB_ERR_ARG;
    }
    a.tgt = target_dev; a.wrp = warped_dev; a.out = coef_dev; a.eps = eps; a.stats = stats_dev;
    a.ticket = (unsigned *)workspace_dev;
    a.partials = (double *)workspace_dev + 8;
    return lncc_launch<true>(a, (cudaStream_t)stream);
}

extern "C" int trb_lncc_backward(int ndim, const float *target_dev, const float *warped_dev, const float *coef_dev, int N, int D,
                                 int H, int W, int win, float scale, const double *moments6_dev, float w_mse, float w_ncc,
                                 float *grad_dev, void *stream)
{
    LnccArgs a{};
    if (int rc = lncc_setup(a, ndim, N, D, H, W, win)) return rc;
    if (!target_dev || !warped_dev || !coef_dev || !grad_dev) { set_error("null pointer"); return TRB_ERR_ARG; }
    if (moments6_dev && N != 1) { set_error("the pointwise MSE / NCC term is for one pair (N == 1)"); return TRB_ERR_ARG; }
    const size_t nb = (size_t)a.nvox * sizeof(float);
    if (overlap(grad_dev, nb, coef_dev, 3 * nb) || overlap(grad_dev, nb, target_dev, nb) || overlap(grad_dev, nb, warped_dev, nb)) {
        set_error("lncc_backward: the gradient overlaps an input");
        return TRB_ERR_ARG;
    }
    a.tgt = target_dev; a.wrp = warped_dev; a.coef = coef_dev; a.out = grad_dev;
    a.gscale = (float)(-(double)scale / a.nvox);
    a.moments = moments6_dev; a.w_mse = w_mse; a.w_ncc = w_ncc;
    return lncc_launch<false>(a, (cudaStream_t)stream);
}
