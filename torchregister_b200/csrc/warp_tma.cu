// warp_tma.cu — TMA-staged forward warp for Register.__call__ / get_affine_warp on 3-D volumes (sm_100a):
// out[p][c] = grid_sample(moving[p][c], affine_grid(theta[p]), bilinear, zeros, align_corners=False)
// (reference warpings.py:18-26 as used by torchregister.py:123-128), all pairs and channels of a batch in ONE launch.
//
// The one-thread-per-voxel kernel of round 1 (warp_affine_kernel, affine.cu) ran at 0.16 of the HBM roofline: 8 scattered
// loads per voxel through a cache hierarchy.  This kernel uses the staging of the epoch kernel (affine_persist.cu): a
// producer warp bounds the source footprint of every 32x16x8 output tile under theta, fetches that box of the moving
// volume with one cp.async.bulk.tensor into a 4-stage mbarrier ring (TMA's zero fill is the zeros padding), 16 consumer
// warps interpolate from shared memory with packed f32x2 arithmetic and write coalesced 128-byte rows.  Tiles whose
// footprint does not fit the box (large rotations) gather from global memory.  Same coordinate arithmetic as the
// epoch kernel, so a warp with the optimised theta reproduces the samples the optimisation saw.
#include "affine_tile.cuh"

namespace trb {

constexpr int kWarpThreads = kTmaThreads + 32;          // 16 consumer warps + the producer warp
constexpr int kWColSlots = 8;
enum { kWFits = 1, kWNewCol = 2, kWEnd = 8 };
struct __align__(16) WTile { float Mrel, zf0; int nz, flags; int colslot, z0, pad0, pad1; };
struct __align__(16) WCol { int x0, y0, item, pad; float coef[12]; };

constexpr size_t kWStageBytes = (size_t)kBX * kBY * kBZ * 4;
constexpr size_t kWOffBars = 0;
constexpr size_t kWOffTiles = 16 * sizeof(uint64_t);
constexpr size_t kWOffCols = kWOffTiles + kStages * sizeof(WTile);
constexpr size_t kWOffStages = (kWOffCols + kWColSlots * sizeof(WCol) + 1023) / 1024 * 1024;
constexpr size_t kWSmem = kWOffStages + kStages * kWStageBytes;

struct WarpParams {
    TmaParams t;                 // t.a: moving, D/H/W, xb/yb, pair_stride (= one channel volume); t.n_pairs = pairs * channels
    const float *theta;          // [pairs][12]
    float *out;
    int n_channels;
};

// NEAREST: grid_sample(mode='nearest'): same producer, box bound, ring and tile walk; each consumer reads the one staged
// voxel at the rounded coordinate (box_nearest), tiles off the box one predicated global load (nearest_offset)
template <bool NEAREST>
__device__ __forceinline__ void warp_affine_tma_body(const WarpParams &wp, const CUtensorMap &map_mov)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + kWOffBars);
    uint64_t *full_bar = bars, *empty_bar = bars + kStages;
    WTile *tiles = reinterpret_cast<WTile *>(smem_raw + kWOffTiles);
    WCol *cols = reinterpret_cast<WCol *>(smem_raw + kWOffCols);
    const TmaParams &p = wp.t;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int W = p.a.W, H = p.a.H, D = p.a.D;
    const int G = gridDim.x, b = blockIdx.x;
    const float inv_d2 = 2.f / (float)D, zoff = 1.f / (float)D - 1.f;

    if (threadIdx.x == 0) {
        for (int i = 0; i < kStages; ++i) { mbar_init(full_bar + i, 1); mbar_init(empty_bar + i, kConsumerWarps); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    if (warp == kConsumerWarps) {
        // ---------------------------------- producer ------------------------------------------------------
        TileIter t;
        iter_begin(t, p, b, G);
        int it = 0, k = 0;
        bool newcol = true;
        ColConst c;
        Coef kf;
        while (t.phase != 2) {
            if (newcol) {
                const int item = t.cg / p.cols_per_pair;
                const float *th = wp.theta + (size_t)(item / wp.n_channels) * 12;
                float thv[12];
#pragma unroll
                for (int i = 0; i < 12; ++i) thv[i] = __ldg(th + i);
                kf = make_coef(thv, D, H, W);
                const int col = t.cg - item * p.cols_per_pair;
                const int ty_i = col / p.tiles_x;
                const int x0 = (col - ty_i * p.tiles_x) * TX, y0 = ty_i * TY;
                const float xa = __ldg(p.a.xb + x0), xe = __ldg(p.a.xb + min(x0 + TX - 1, W - 1));
                const float ya = __ldg(p.a.yb + y0), ye = __ldg(p.a.yb + min(y0 + TY - 1, H - 1));
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    const float base = kf.A[r][0] * xa + kf.A[r][1] * ya + kf.A[r][2] * zoff + kf.C[r];
                    const float dx = kf.A[r][0] * (xe - xa), dy = kf.A[r][1] * (ye - ya), dz = kf.A[r][2] * inv_d2 * (float)(TZ - 1);
                    c.lo[r] = base + fminf(dx, 0.f) + fminf(dy, 0.f) + fminf(dz, 0.f) - 0.03f;
                    c.hi[r] = base + fmaxf(dx, 0.f) + fmaxf(dy, 0.f) + fmaxf(dz, 0.f) + 0.03f;
                    c.step[r] = kf.A[r][2] * inv_d2 * (float)TZ;
                }
                c.pair = item; c.x0 = x0; c.y0 = y0;
                if (lane == 0) {
                    WCol &pc = cols[k % kWColSlots];
                    pc.x0 = x0; pc.y0 = y0; pc.item = item; pc.pad = 0;
#pragma unroll
                    for (int r = 0; r < 3; ++r) {
#pragma unroll
                        for (int j = 0; j < 3; ++j) pc.coef[r * 4 + j] = kf.A[r][j];
                        pc.coef[r * 4 + 3] = kf.C[r];
                    }
                }
            }
            const int stage = it % kStages;
            if (it >= kStages) mbar_wait(empty_bar + stage, (unsigned)((it / kStages) - 1) & 1u);
            TileIter nx = t;
            const bool moved = iter_next(nx, p, b, G);
            if (lane == 0) {
                int o[3];
                bool fits = true;
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
                const int z0 = t.tz_i * TZ;
                WTile m;
                m.Mrel = 2.f - kIdxScale * (float)(o[0] + kBX * o[1] + kBX * kBY * o[2]);
                m.zf0 = (float)z0;
                m.nz = min(TZ, D - z0);
                m.flags = (fits ? kWFits : 0) | (newcol ? kWNewCol : 0);
                m.colslot = k % kWColSlots; m.z0 = z0; m.pad0 = m.pad1 = 0;
                tiles[stage] = m;
                if (fits) {
                    mbar_arrive_expect_tx(full_bar + stage, (unsigned)kWStageBytes);
                    tma_load_4d(smem_raw + kWOffStages + (size_t)stage * kWStageBytes, &map_mov, full_bar + stage, o[0], o[1], o[2], c.pair);
                } else {
                    mbar_arrive(full_bar + stage);
                }
            }
            __syncwarp();
            if (moved) ++k;
            newcol = moved;
            t = nx;
            ++it;
        }
        const int stage = it % kStages;
        if (it >= kStages) mbar_wait(empty_bar + stage, (unsigned)((it / kStages) - 1) & 1u);
        if (lane == 0) {
            WTile m = {};
            m.flags = kWEnd;
            tiles[stage] = m;
            mbar_arrive(full_bar + stage);
        }
        return;
    }

    // -------------------------------------- consumers -----------------------------------------------------
    int x = 0, y = 0;
    bool valid = false;
    float pxy[3] = {0.f, 0.f, 0.f}, sz[3] = {0.f, 0.f, 0.f};
    const float *__restrict__ mov = p.a.moving;
    float *__restrict__ dst = wp.out;
    for (int it = 0;; ++it) {
        const int stage = it % kStages;
        mbar_wait(full_bar + stage, (unsigned)(it / kStages) & 1u);
        const WTile m = tiles[stage];
        if (m.flags & kWEnd) break;
        if (m.flags & kWNewCol) {
            const WCol &pc = cols[m.colslot];
            x = pc.x0 + lane; y = pc.y0 + warp;
            valid = (x < W) && (y < H);
            const float xv = __ldg(p.a.xb + min(x, W - 1)), yv = __ldg(p.a.yb + min(y, H - 1));
#pragma unroll
            for (int r = 0; r < 3; ++r) {
                pxy[r] = fmaf(pc.coef[r * 4 + 0], xv, fmaf(pc.coef[r * 4 + 1], yv, fmaf(pc.coef[r * 4 + 2], zoff, pc.coef[r * 4 + 3])));
                sz[r] = pc.coef[r * 4 + 2] * inv_d2;
            }
            mov = p.a.moving + (size_t)pc.item * p.a.pair_stride;
            dst = wp.out + (size_t)pc.item * p.a.pair_stride + (size_t)y * W + x;
        }
        const uint32_t box_addr = smem_u32(smem_raw + kWOffStages + (size_t)stage * kWStageBytes);
        const size_t HW = (size_t)H * W;
        if (valid) {
            float *o = dst + (size_t)m.z0 * HW;
            if constexpr (NEAREST) {
                if (m.flags & kWFits) {
                    // voxel pairs (z, z + 1) as in the bilinear path; an odd tail's second voxel lies inside the
                    // bounded footprint (the bound covers all TZ slices of a tile) and is not stored
                    float2 zf = make_float2(m.zf0, m.zf0 + 1.f);
                    for (int zz = 0; zz < m.nz; zz += 2) {
                        const float2 tb = box_nearest<kBX, kBY>(m.Mrel, __ffma2_rn(f2(sz[0]), zf, f2(pxy[0])),
                                                                __ffma2_rn(f2(sz[1]), zf, f2(pxy[1])), __ffma2_rn(f2(sz[2]), zf, f2(pxy[2])));
                        __stcs(o + (size_t)zz * HW, lds_f<0>(cell_addr(box_addr, tb.x)));
                        if (zz + 1 < m.nz) __stcs(o + (size_t)(zz + 1) * HW, lds_f<0>(cell_addr(box_addr, tb.y)));
                        zf = __fadd2_rn(zf, f2(2.f));
                    }
                } else {
                    for (int zz = 0; zz < m.nz; ++zz) {
                        const float zf = m.zf0 + (float)zz;
                        long long off;
                        const bool v = nearest_offset(D, H, W, fmaf(sz[0], zf, pxy[0]), fmaf(sz[1], zf, pxy[1]), fmaf(sz[2], zf, pxy[2]), off);
                        __stcs(o + (size_t)zz * HW, v ? __ldg(mov + off) : 0.f);
                    }
                }
            } else if ((m.flags & kWFits) && m.nz == TZ) {
                float2 zf = make_float2(m.zf0, m.zf0 + 1.f);
#pragma unroll
                for (int j = 0; j < TZ / 2; ++j) {
                    const float2 ix = __ffma2_rn(f2(sz[0]), zf, f2(pxy[0]));
                    const float2 iy = __ffma2_rn(f2(sz[1]), zf, f2(pxy[1]));
                    const float2 iz = __ffma2_rn(f2(sz[2]), zf, f2(pxy[2]));
                    const float2 v = pair_sample<kBX, kBY, false>(box_addr, box_cells<kBX, kBY>(m.Mrel, ix, iy, iz)).val;
                    __stcs(o + (size_t)(2 * j) * HW, v.x);
                    __stcs(o + (size_t)(2 * j + 1) * HW, v.y);
                    zf = __fadd2_rn(zf, f2(2.f));
                }
            } else if (m.flags & kWFits) {
                for (int zz = 0; zz < m.nz; ++zz) {
                    const float za = m.zf0 + (float)zz;
                    const float2 zf = make_float2(za, za);
                    const BoxCells c = box_cells<kBX, kBY>(m.Mrel, __ffma2_rn(f2(sz[0]), zf, f2(pxy[0])),
                                                           __ffma2_rn(f2(sz[1]), zf, f2(pxy[1])), __ffma2_rn(f2(sz[2]), zf, f2(pxy[2])));
                    const float2 v = pair_sample<kBX, kBY, false>(box_addr, c).val;
                    __stcs(o + (size_t)zz * HW, v.x);
                }
            } else {
                for (int zz = 0; zz < m.nz; ++zz) {
                    const float zf = m.zf0 + (float)zz;
                    const Cell3 k = gather_clamped3(mov, D, H, W, fmaf(sz[0], zf, pxy[0]), fmaf(sz[1], zf, pxy[1]), fmaf(sz[2], zf, pxy[2]));
                    __stcs(o + (size_t)zz * HW, blend_cell3<false>(k).val);
                }
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(empty_bar + stage);
    }
}

__global__ void __launch_bounds__(kWarpThreads, 1)
warp_affine_tma_kernel(const WarpParams wp, const __grid_constant__ CUtensorMap map_mov)
{
    warp_affine_tma_body<false>(wp, map_mov);
}

__global__ void __launch_bounds__(kWarpThreads, 1)
warp_affine_nearest_tma_kernel(const WarpParams wp, const __grid_constant__ CUtensorMap map_mov)
{
    warp_affine_tma_body<true>(wp, map_mov);
}

bool warp_tma_eligible(const float *moving, const float *out, int n_items, long long vol, int D, int H, int W)
{
    if (W % 4 != 0 || W < TX || H < TY || D < 1) return false;
    if (((uintptr_t)moving & 15) || ((uintptr_t)out & 3)) return false;
    if (n_items > 1 && (vol % 4 != 0)) return false;
    // the staged-box index range; it also keeps every axis far below kMaxFastFloorAxis (the kMagic floor / rint)
    if ((double)W + (double)kBX * H + (double)kBX * kBY * D > 1.8e6) return false;
    return encode_fn() != nullptr;
}

// all (pair, channel) volumes of a batch in one launch; theta_dev: [n_pairs][12]
int launch_warp_affine_tma(const float *moving, float *out, int n_pairs, int n_channels, int D, int H, int W,
                           const float *theta_dev, const float *xb, const float *yb, bool nearest, cudaStream_t stream)
{
    const int n_items = n_pairs * n_channels;
    const long long vol = (long long)D * H * W;
    CUtensorMap map_mov;
    int rc = make_map(&map_mov, moving, n_items, vol, D, H, W, kBX, kBY, kBZ);
    if (rc) return rc;
    WarpParams wp{};
    wp.t.a.moving = moving; wp.t.a.pair_stride = vol;
    wp.t.a.D = D; wp.t.a.H = H; wp.t.a.W = W; wp.t.a.xb = xb; wp.t.a.yb = yb;
    wp.t.a.s_begin = 0; wp.t.a.s_end = D;
    wp.t.n_pairs = n_items;
    wp.t.tiles_x = (W + TX - 1) / TX; wp.t.tiles_y = (H + TY - 1) / TY; wp.t.tiles_z = (D + TZ - 1) / TZ;
    wp.t.cols_per_pair = wp.t.tiles_x * wp.t.tiles_y;
    wp.theta = theta_dev; wp.out = out; wp.n_channels = n_channels;
    int sms;
    if ((rc = sm_count(sms))) return rc;
    const long long total_cols = (long long)n_items * wp.t.cols_per_pair;
    long long grid_ll = sms;
    if (grid_ll > total_cols * wp.t.tiles_z) grid_ll = total_cols * wp.t.tiles_z;
    const int grid = (int)grid_ll;
    wp.t.full_rounds = (int)(total_cols / grid);
    wp.t.tail_tiles = (total_cols - (long long)wp.t.full_rounds * grid) * wp.t.tiles_z;
    const auto kernel = nearest ? warp_affine_nearest_tma_kernel : warp_affine_tma_kernel;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWSmem);
    if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(warp_affine_tma)");
    kernel<<<grid, kWarpThreads, kWSmem, stream>>>(wp, map_mov);
    return check_cuda(cudaGetLastError(), "warp_affine_tma");
}

}  // namespace trb
