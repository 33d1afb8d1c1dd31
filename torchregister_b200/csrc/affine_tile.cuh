// affine_tile.cuh — device pieces shared by the TMA-staged 3-D rigid/affine kernels (sm_100a):
// affine_tma.cu (one launch per epoch; also the unfused moments pass) and affine_persist.cu (persistent,
// warp-specialised multi-epoch kernel), and by the forward warp (warp_tma.cu).  PTX wrappers, the staged-box sampling
// (box_cells, pair_sample, voxel_staged) and the moment accumulation over it (pair_step, pair_step2), the clamped global
// gather of the fallback paths (gather_clamped3), the work decomposition (TileIter), the footprint bound and the
// tensor-map encoder.  The scalar blend itself is common.cuh's blend_cell3.
#pragma once
#include "common.cuh"
#include "affine_shared.cuh"
#include <cuda.h>
#include <type_traits>

namespace trb {

// Tile depth / ring depth (build-time A/B: TRB_DEFINES="TRB_TZ=8 TRB_STAGES=4" is the round-1 geometry).  16 slices per tile
// halve the per-tile fixed work of every consumer warp (barrier wait, descriptor, addresses: ~110 issue slots) against
// the same 16 voxel-pair steps; two 97 KB stages buffer as many bytes as four 54 KB ones did.  Measured on the 8-pair batch:
// 120.1 -> 114.8 us/epoch; 512^3 348 -> 334; the rotation a staged box tolerates is unchanged (the z slack is 4 in both).
#ifndef TRB_TZ
#define TRB_TZ 16
#endif
#ifndef TRB_STAGES
#define TRB_STAGES 2
#endif
constexpr int TX = 32, TY = 16, TZ = TRB_TZ;     // output tile (voxels)
constexpr int kBX = 40, kBY = 20, kBZ = TZ + 4, kStages = TRB_STAGES;   // staged box of the moving volume (incl. halo), ring depth
constexpr int kConsumerWarps = TY;               // warp <-> y row of the tile
constexpr int kTmaThreads = kConsumerWarps * 32;
constexpr float kMagic = 12582912.f;             // 1.5 * 2^23
constexpr float kIdxScale = 1.f / 4194304.f;     // 2^-22

// ---- PTX helpers ---------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}"
        ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void *dst, const CUtensorMap *map, uint64_t *bar, int c0, int c1, int c2, int c3)
{
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cta.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}

__device__ __forceinline__ float2 f2(float a) { return make_float2(a, a); }

// compile-time loop: f(std::integral_constant<int, I>) for I in [I0, N) — the index can then pick immediates
template <int I, int N, typename F>
__device__ __forceinline__ void static_for(F &&f)
{
    if constexpr (I < N) {
        f(std::integral_constant<int, I>{});
        static_for<I + 1, N>(f);
    }
}
__device__ __forceinline__ float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }

#ifdef TRB_TIMING
#ifdef TRB_TIMING_OWNER
__device__ unsigned long long g_dbg[1024 * 16];
#endif
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define TRB_T(slot) do { if (lane == 0) atomicMax(&g_dbg[blockIdx.x * 16 + (slot)], gtime()); } while (0)
#define TRB_TD(slot, t0) do { if (lane == 0) atomicMax(&g_dbg[blockIdx.x * 16 + (slot)], gtime() - (t0)); } while (0)
#else
#define TRB_T(slot) do { } while (0)
#define TRB_TD(slot, t0) do { } while (0)
#endif

struct TmaParams {
    AffineParams a;
    int n_pairs;
    int tiles_x, tiles_y, tiles_z;     // output tiles per axis
    int cols_per_pair;                 // tiles_x * tiles_y
    int full_rounds;                   // rounds in which every CTA owns one whole column
    long long tail_tiles;              // tiles of the remaining columns, cut into one span per CTA
    int use_groups;                    // grid reduction: 1 = 16-CTA groups folded during the launch (many pairs),
                                       // 0 = the last CTA folds all slots directly with all its warps (few pairs)
};

struct TileMeta { int ox, oy, oz, fits; };

// per-axis affine map voxel index -> un-normalised source coordinate (grid_sample align_corners=False
// folded into affine_grid): i_r = A[r][0]*xv + A[r][1]*yv + A[r][2]*zv + C[r], xv/yv/zv the base coordinates
struct Coef { float A[3][3], C[3]; };

__device__ __forceinline__ Coef make_coef(const float *th, int D, int H, int W)
{
    Coef k;
    const float h[3] = {0.5f * W, 0.5f * H, 0.5f * D};
#pragma unroll
    for (int r = 0; r < 3; ++r) {
#pragma unroll
        for (int c = 0; c < 3; ++c) k.A[r][c] = th[r * 4 + c] * h[r];
        k.C[r] = fmaf(th[r * 4 + 3] + 1.f, h[r], -0.5f);
    }
    return k;
}

template <int BX, int BY, int BZ>
struct SmemLayout {
    static constexpr int kBoxFloats = BX * BY * BZ;
    static constexpr int kTgtFloats = TX * TY * TZ;
    static constexpr int kStageBytes = ((kBoxFloats + kTgtFloats) * 4 + 127) / 128 * 128;
};


template <int OFF>
__device__ __forceinline__ float lds_f(uint32_t addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(addr), "n"(OFF));
    return v;
}
__device__ __forceinline__ float lds_f_dyn(uint32_t addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}

struct Acc {
    float2 s[5];        // sum t, w, t^2, w^2, t*w            (two partial streams: voxel a / voxel b)
    float2 P[3][3];     // sum k*G_r,        k in {1, t, w}
    float2 Q[3][3];     // sum k*G_r*z
};

// Staged-box cells of two voxels (same x,y; z and z+1): fractions and box indices.
// floor() = round-down add of 1.5*2^23 (FADD.RM) and subtracting it again; FRND on the XU pipe was
// tried instead (it frees 6 packed fp32 ops per pair) but its latency lengthened the dependent
// chain and the step got 11% slower (profiles/r01_notes.md)
struct BoxCells {
    float2 tx, ty, tz;      // fractions (voxel a, voxel b)
    float2 tb;              // box indices of the two cells' (x0,y0,z0) corners, see cell_addr
};
template <int BX, int BY>
__device__ __forceinline__ BoxCells box_cells(float Mrel, float2 ix, float2 iy, float2 iz)
{
    BoxCells b;
    const float2 M = f2(kMagic), nM = f2(-kMagic);
    const float2 flx = __fadd2_rd(ix, M), fly = __fadd2_rd(iy, M), flz = __fadd2_rd(iz, M);
    const float2 fx = __fadd2_rn(flx, nM), fy = __fadd2_rn(fly, nM), fz = __fadd2_rn(flz, nM);
    b.tx = sub2(ix, fx); b.ty = sub2(iy, fy); b.tz = sub2(iz, fz);
    b.tb = __ffma2_rn(f2(kIdxScale * (float)(BX * BY)), fz,
                      __ffma2_rn(f2(kIdxScale * (float)BX), fy, __ffma2_rn(f2(kIdxScale), fx, f2(Mrel))));
    return b;
}
// The nearest-neighbour twin (grid_sample mode='nearest'): box indices of the voxels at ix, iy, iz rounded half to even,
// the same add in round-to-nearest mode.  The rounded index lies in {floor, floor + 1}, so a box that holds the cells
// holds these voxels too.
template <int BX, int BY>
__device__ __forceinline__ float2 box_nearest(float Mrel, float2 ix, float2 iy, float2 iz)
{
    const float2 M = f2(kMagic), nM = f2(-kMagic);
    const float2 rx = __fadd2_rn(__fadd2_rn(ix, M), nM), ry = __fadd2_rn(__fadd2_rn(iy, M), nM), rz = __fadd2_rn(__fadd2_rn(iz, M), nM);
    return __ffma2_rn(f2(kIdxScale * (float)(BX * BY)), rz,
                      __ffma2_rn(f2(kIdxScale * (float)BX), ry, __ffma2_rn(f2(kIdxScale), rx, f2(Mrel))));
}
// smem byte address of a cell's corner; box_m: smem byte address of the staged box.  The box-relative linear index
// is formed in fp32 and scaled by 2^-22 onto [2, 4): exact, and the bit pattern is 0x40000000 + index, so (bits << 2)
// IS the byte offset (the 0x4 wraps away)
__device__ __forceinline__ uint32_t cell_addr(uint32_t box_m, float tb) { return box_m + ((uint32_t)__float_as_int(tb) << 2); }

// trilinear sample of both voxels from the staged box, packed (voxel a, voxel b) in every value;
// g: d val / d (x, y, z) in voxel units (WANT_GRAD only)
struct PairSample {
    float2 val, g[3];
};
template <int BX, int BY, bool WANT_GRAD>
__device__ __forceinline__ PairSample pair_sample(uint32_t box_m, const BoxCells &b)
{
    PairSample s;
    const uint32_t qa = cell_addr(box_m, b.tb.x), qb = cell_addr(box_m, b.tb.y);
    const float2 tx = b.tx, ty = b.ty, tz = b.tz;
    constexpr int SY = BX * 4, SZ = BX * BY * 4;
    const float2 c000 = make_float2(lds_f<0>(qa), lds_f<0>(qb)), c001 = make_float2(lds_f<4>(qa), lds_f<4>(qb));
    const float2 c010 = make_float2(lds_f<SY>(qa), lds_f<SY>(qb)), c011 = make_float2(lds_f<SY + 4>(qa), lds_f<SY + 4>(qb));
    const float2 c100 = make_float2(lds_f<SZ>(qa), lds_f<SZ>(qb)), c101 = make_float2(lds_f<SZ + 4>(qa), lds_f<SZ + 4>(qb));
    const float2 c110 = make_float2(lds_f<SZ + SY>(qa), lds_f<SZ + SY>(qb));
    const float2 c111 = make_float2(lds_f<SZ + SY + 4>(qa), lds_f<SZ + SY + 4>(qb));
    const float2 d00 = sub2(c001, c000), d01 = sub2(c011, c010), d10 = sub2(c101, c100), d11 = sub2(c111, c110);
    const float2 v00 = __ffma2_rn(tx, d00, c000), v01 = __ffma2_rn(tx, d01, c010);
    const float2 v10 = __ffma2_rn(tx, d10, c100), v11 = __ffma2_rn(tx, d11, c110);
    const float2 e0 = sub2(v01, v00), e1 = sub2(v11, v10);
    const float2 w0 = __ffma2_rn(ty, e0, v00), w1 = __ffma2_rn(ty, e1, v10);
    const float2 gz = sub2(w1, w0);
    s.val = __ffma2_rn(tz, gz, w0);
    if (WANT_GRAD) {
        s.g[2] = gz;
        s.g[1] = __ffma2_rn(tz, sub2(e1, e0), e0);
        const float2 dx0 = __ffma2_rn(ty, sub2(d01, d00), d00), dx1 = __ffma2_rn(ty, sub2(d11, d10), d10);
        s.g[0] = __ffma2_rn(tz, sub2(dx1, dx0), dx0);
    }
    return s;
}

// one pair of voxels (same x,y; z and z+1) into the round-1 accumulators.  SECOND=false masks voxel b.
template <int BX, int BY, bool SECOND, bool MSE_ONLY>
__device__ __forceinline__ float2 pair_step(uint32_t box_m, float Mrel, float2 ix, float2 iy, float2 iz,
                                            float2 t, float2 zf, Acc &A)
{
    const PairSample s = pair_sample<BX, BY, true>(box_m, box_cells<BX, BY>(Mrel, ix, iy, iz));
    float2 G[3] = {s.g[0], s.g[1], s.g[2]};
    float2 val = s.val;
    if (!SECOND) {                       // odd tail: the duplicate voxel contributes nothing
        const float2 m = make_float2(1.f, 0.f);
        val = __fmul2_rn(val, m); t = __fmul2_rn(t, m);
#pragma unroll
        for (int r = 0; r < 3; ++r) G[r] = __fmul2_rn(G[r], m);
    }
    if (MSE_ONLY) {
        // w_ncc == 0: dL/dw_v = gm * (w_v - t_v) is known up front, so ONE weighted family (d = w - t) replaces
        // the three (1, t, w): 9 packed moment updates instead of 25.  Stored in the "w" slots with the "t"
        // slots left at zero, which the shared epilogue turns into gm * sum d*J.
        const float2 d = sub2(val, t);
        A.s[2] = __ffma2_rn(d, d, A.s[2]);                 // sum d^2 rides in the sum t^2 slot
        const float2 dzf = __fmul2_rn(d, zf);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            A.P[2][r] = __ffma2_rn(d, G[r], A.P[2][r]);
            A.Q[2][r] = __ffma2_rn(dzf, G[r], A.Q[2][r]);
        }
    } else {
        A.s[0] = __fadd2_rn(A.s[0], t);
        A.s[1] = __fadd2_rn(A.s[1], val);
        A.s[2] = __ffma2_rn(t, t, A.s[2]);
        A.s[3] = __ffma2_rn(val, val, A.s[3]);
        A.s[4] = __ffma2_rn(t, val, A.s[4]);
        const float2 tzf = __fmul2_rn(t, zf), wzf = __fmul2_rn(val, zf);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            A.P[0][r] = __fadd2_rn(A.P[0][r], G[r]);
            A.P[1][r] = __ffma2_rn(t, G[r], A.P[1][r]);
            A.P[2][r] = __ffma2_rn(val, G[r], A.P[2][r]);
            A.Q[0][r] = __ffma2_rn(zf, G[r], A.Q[0][r]);
            A.Q[1][r] = __ffma2_rn(tzf, G[r], A.Q[1][r]);
            A.Q[2][r] = __ffma2_rn(wzf, G[r], A.Q[2][r]);
        }
    }
    return val;                          // the two warped samples (z, z + 1)
}

// ---- second formulation of the per-voxel arithmetic (round 2; used by affine_persist.cu) ------------------------------
// tools/microbench2.cu: on sm_100a a packed fp32 instruction is bounded by REGISTER-FILE READS, not by the fp32 pipe: an
// FFMA2 with three distinct register pairs costs 4.2 cycles per sub-partition, one whose third source is a 32-bit
// broadcast or sits in the operand reuse cache 2.6, two broadcasts 2.15 (profiles/r02_microbench_ffma2_operands.txt).
// pair_step packs voxel a / voxel b into the two halves of every value, so its moment updates read three pairs
// (k, G_r, accumulator).  Here the two halves of a pair belong to the SAME voxel instead:
//   * interpolation: the x- and y-stage run on pairs over the two z planes of the cell ((c000,c100), ...) with the
//     fractions as 32-bit broadcast operands; the z-stage is scalar and leaves val, G0, G1, G2 in freely allocatable
//     registers, i.e. as the pairs GA = (G0,G1), GB = (G2,val) at no cost;
//   * moments: acc_k += k * GA, acc_k' += k * GB with k in {1, t, val, z, t z, val z} a broadcast scalar — two source
//     pairs per instruction, one of them (GA / GB) shared by six consecutive instructions.  The second lane of GB yields
//     sum w, sum t w, sum w^2 for free.  Both voxels of a step add into the same accumulators: 12 pairs = 24 registers
//     instead of 23 x 2 lanes = 46;
//   * sum t and sum t^2 do not depend on theta: they are not accumulated here at all (target_sums_kernel computes them
//     once per launch).
// Every interpolation operation is the same IEEE operation as in pair_step (same values bit for bit); only the order
// in which the moments are summed differs.
struct Acc2 {
    float2 a[12];    // [2*f + h]: family f in {1, t, w, z, tz, wz}, h = 0: (sum k G0, sum k G1), h = 1: (sum k G2, sum k w)
};                   // MSE_ONLY uses [0..3]: family d = w - t and d z, with h = 1: (sum d G2, sum d^2) / (sum d z G2, -)

template <bool MSE_ONLY>
__device__ __forceinline__ void moments_accumulate(float t, float z, float val, float G0, float G1, float G2, Acc2 &A)
{
    const float2 GA = make_float2(G0, G1);
    if (MSE_ONLY) {
        const float d = val - t, dz = d * z;
        const float2 GB = make_float2(G2, d);
        A.a[0] = __ffma2_rn(f2(d), GA, A.a[0]);
        A.a[2] = __ffma2_rn(f2(dz), GA, A.a[2]);
        A.a[1] = __ffma2_rn(f2(d), GB, A.a[1]);
        A.a[3] = __ffma2_rn(f2(dz), GB, A.a[3]);
    } else {
        const float2 GB = make_float2(G2, val);
        const float tz = t * z, wz = val * z;
        A.a[0] = __fadd2_rn(A.a[0], GA);
        A.a[2] = __ffma2_rn(f2(t), GA, A.a[2]);
        A.a[4] = __ffma2_rn(f2(val), GA, A.a[4]);
        A.a[6] = __ffma2_rn(f2(z), GA, A.a[6]);
        A.a[8] = __ffma2_rn(f2(tz), GA, A.a[8]);
        A.a[10] = __ffma2_rn(f2(wz), GA, A.a[10]);
        A.a[1] = __fadd2_rn(A.a[1], GB);
        A.a[3] = __ffma2_rn(f2(t), GB, A.a[3]);
        A.a[5] = __ffma2_rn(f2(val), GB, A.a[5]);
        A.a[7] = __ffma2_rn(f2(z), GB, A.a[7]);
        A.a[9] = __ffma2_rn(f2(tz), GB, A.a[9]);
        A.a[11] = __ffma2_rn(f2(wz), GB, A.a[11]);
    }
}

// one voxel whose cell is staged in shared memory at byte address q (its corner (x0,y0,z0)); returns the warped sample
template <int BX, int BY, bool MSE_ONLY>
__device__ __forceinline__ float voxel_staged(uint32_t q, float tx, float ty, float tz, float t, float z, Acc2 &A)
{
    constexpr int SY = BX * 4, SZ = BX * BY * 4;
    const float2 P0 = make_float2(lds_f<0>(q), lds_f<SZ>(q)), P1 = make_float2(lds_f<4>(q), lds_f<SZ + 4>(q));
    const float2 R0 = make_float2(lds_f<SY>(q), lds_f<SZ + SY>(q)), R1 = make_float2(lds_f<SY + 4>(q), lds_f<SZ + SY + 4>(q));
    const float2 dP = sub2(P1, P0), dR = sub2(R1, R0);                   // (d00, d10), (d01, d11)
    const float2 vA = __ffma2_rn(f2(tx), dP, P0), vB = __ffma2_rn(f2(tx), dR, R0);   // (v00, v10), (v01, v11)
    const float2 e = sub2(vB, vA);                                        // (e0, e1)
    const float2 w = __ffma2_rn(f2(ty), e, vA);                           // (w0, w1)
    const float2 dx = __ffma2_rn(f2(ty), sub2(dR, dP), dP);               // (dx0, dx1)
    const float G2 = w.y - w.x;
    const float val = fmaf(tz, G2, w.x);
    const float G1 = fmaf(tz, e.y - e.x, e.x);
    const float G0 = fmaf(tz, dx.y - dx.x, dx.x);
    moments_accumulate<MSE_ONLY>(t, z, val, G0, G1, G2, A);
    return val;
}

// two voxels (same x,y; z and z+1): coordinates, floor, fraction and index stay packed over the two voxels (their
// operands are per-thread constants, i.e. broadcasts); SECOND = false skips voxel b.  Returns the two warped samples.
template <int BX, int BY, bool SECOND, bool MSE_ONLY>
__device__ __forceinline__ float2 pair_step2(uint32_t box_m, float Mrel, float2 ix, float2 iy, float2 iz, float2 t, float2 zf, Acc2 &A)
{
    const BoxCells c = box_cells<BX, BY>(Mrel, ix, iy, iz);
    float2 w;
    w.x = voxel_staged<BX, BY, MSE_ONLY>(cell_addr(box_m, c.tb.x), c.tx.x, c.ty.x, c.tz.x, t.x, zf.x, A);
    w.y = 0.f;
    if (SECOND) w.y = voxel_staged<BX, BY, MSE_ONLY>(cell_addr(box_m, c.tb.y), c.tx.y, c.ty.y, c.tz.y, t.y, zf.y, A);
    return w;
}

// Global gather for the voxels whose cell is not staged: the position is clamped to [-4, S + 4] (keeps the
// magic-number floor in range; a clamped cell lies wholly in the zero padding), then 8 predicated loads.
__device__ __forceinline__ Cell3 gather_clamped3(const float *__restrict__ mov, int D, int H, int W, float ix, float iy, float iz)
{
    Cell3 k;
    ix = fminf(fmaxf(ix, -4.f), (float)W + 4.f);
    iy = fminf(fmaxf(iy, -4.f), (float)H + 4.f);
    iz = fminf(fmaxf(iz, -4.f), (float)D + 4.f);
    k.fx = __fadd_rd(ix, kMagic) - kMagic; k.fy = __fadd_rd(iy, kMagic) - kMagic; k.fz = __fadd_rd(iz, kMagic) - kMagic;
    k.tx = ix - k.fx; k.ty = iy - k.fy; k.tz = iz - k.fz;
    load_cell3(mov, D, H, W, (int)k.fx, (int)k.fy, (int)k.fz, k.c);
    return k;
}

// fallback for tiles whose source footprint does not fit the TMA box: one voxel, global gathers (Acc2 form)
template <bool MSE_ONLY>
__device__ __forceinline__ float voxel_direct2(const float *__restrict__ mov, int D, int H, int W, float ix, float iy, float iz,
                                               float t, float zf, Acc2 &A)
{
    const Sample<3> s = blend_cell3<true>(gather_clamped3(mov, D, H, W, ix, iy, iz));
    moments_accumulate<MSE_ONLY>(t, zf, s.val, s.g[0], s.g[1], s.g[2], A);
    return s.val;
}

// the same voxel from the PAIR volume (large-rotation variant): P[z][y][xr] = (v[xr-2], v[xr-1]) with W + 3 records per row and
// zeros outside, so ONE 8-byte load per (y, z) corner brings both x neighbours and the zero padding in x: 4 gathers instead of 8
// — the gathers of a rotated warp are bound by the number of cache lines they touch, not by bytes
constexpr int kPairPad = 3;
template <bool MSE_ONLY>
__device__ __forceinline__ float voxel_direct2p(const float2 *__restrict__ P, int D, int H, int W, float ix, float iy, float iz,
                                                float t, float zf, Acc2 &A)
{
    ix = fminf(fmaxf(ix, -2.f), (float)W + 0.5f);       // x0 in [-2, W]: records 0 and W + 2 are (0, 0)
    iy = fminf(fmaxf(iy, -4.f), (float)H + 4.f);
    iz = fminf(fmaxf(iz, -4.f), (float)D + 4.f);
    const float fx = __fadd_rd(ix, kMagic) - kMagic, fy = __fadd_rd(iy, kMagic) - kMagic, fz = __fadd_rd(iz, kMagic) - kMagic;
    const float tx = ix - fx, ty = iy - fy, tz = iz - fz;
    const int x0 = (int)fx, y0 = (int)fy, z0 = (int)fz;
    const bool vy0 = (unsigned)y0 < (unsigned)H, vy1 = (unsigned)(y0 + 1) < (unsigned)H;
    const bool vz0 = (unsigned)z0 < (unsigned)D, vz1 = (unsigned)(z0 + 1) < (unsigned)D;
    const long long Wp = W + kPairPad, HWp = (long long)H * Wp, o = ((long long)z0 * H + y0) * Wp + (x0 + 2);
    const float2 zero = make_float2(0.f, 0.f);
    const float2 r00 = (vz0 & vy0) ? __ldg(P + o) : zero, r01 = (vz0 & vy1) ? __ldg(P + o + Wp) : zero;
    const float2 r10 = (vz1 & vy0) ? __ldg(P + o + HWp) : zero, r11 = (vz1 & vy1) ? __ldg(P + o + HWp + Wp) : zero;
    Cell3 k;
    k.c[0] = r00.x; k.c[1] = r00.y; k.c[2] = r01.x; k.c[3] = r01.y; k.c[4] = r10.x; k.c[5] = r10.y; k.c[6] = r11.x; k.c[7] = r11.y;
    k.tx = tx; k.ty = ty; k.tz = tz;
    const Sample<3> s = blend_cell3<true>(k);
    moments_accumulate<MSE_ONLY>(t, zf, s.val, s.g[0], s.g[1], s.g[2], A);
    return s.val;
}

// and from the QUAD volume: Q[z][yr][xr] = (v[y][x], v[y][x+1], v[y+1][x], v[y+1][x+1]) at (x, y) = (xr - 2, yr - 2), H + 3 rows
// of W + 3 records, zeros outside: ONE 16-byte load per z plane of the cell brings its four corners and the zero padding in x
// and y — 2 gathers per voxel
template <bool MSE_ONLY>
__device__ __forceinline__ float voxel_direct2q(const float4 *__restrict__ Q, int D, int H, int W, float ix, float iy, float iz,
                                                float t, float zf, Acc2 &A)
{
    ix = fminf(fmaxf(ix, -2.f), (float)W + 0.5f);       // x0 in [-2, W], y0 in [-2, H]: the border records are zero
    iy = fminf(fmaxf(iy, -2.f), (float)H + 0.5f);
    iz = fminf(fmaxf(iz, -4.f), (float)D + 4.f);
    const float fx = __fadd_rd(ix, kMagic) - kMagic, fy = __fadd_rd(iy, kMagic) - kMagic, fz = __fadd_rd(iz, kMagic) - kMagic;
    const float tx = ix - fx, ty = iy - fy, tz = iz - fz;
    const int x0 = (int)fx, y0 = (int)fy, z0 = (int)fz;
    const bool vz0 = (unsigned)z0 < (unsigned)D, vz1 = (unsigned)(z0 + 1) < (unsigned)D;
    const long long Wp = W + kPairPad, HWp = (long long)(H + kPairPad) * Wp, o = (long long)z0 * HWp + (long long)(y0 + 2) * Wp + (x0 + 2);
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4 q0 = vz0 ? __ldg(Q + o) : zero, q1 = vz1 ? __ldg(Q + o + HWp) : zero;      // (c00, c01, c10, c11) of plane z0 / z0 + 1
    Cell3 k;
    k.c[0] = q0.x; k.c[1] = q0.y; k.c[2] = q0.z; k.c[3] = q0.w; k.c[4] = q1.x; k.c[5] = q1.y; k.c[6] = q1.z; k.c[7] = q1.w;
    k.tx = tx; k.ty = ty; k.tz = tz;
    const Sample<3> s = blend_cell3<true>(k);
    moments_accumulate<MSE_ONLY>(t, zf, s.val, s.g[0], s.g[1], s.g[2], A);
    return s.val;
}

// fallback for tiles whose source footprint does not fit the TMA box: one voxel, global gathers
template <bool MSE_ONLY>
__device__ __forceinline__ float voxel_direct(const float *__restrict__ mov, int D, int H, int W, float ix, float iy, float iz,
                                              float t, float zf, Acc &A)
{
    const Sample<3> s = blend_cell3<true>(gather_clamped3(mov, D, H, W, ix, iy, iz));
    const float val = s.val;
    const float *G = s.g;
    if (MSE_ONLY) {
        const float d = val - t;
        A.s[2].x = fmaf(d, d, A.s[2].x);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            A.P[2][r].x = fmaf(d, G[r], A.P[2][r].x);
            A.Q[2][r].x = fmaf(zf * d, G[r], A.Q[2][r].x);
        }
    } else {
        A.s[0].x += t; A.s[1].x += val;
        A.s[2].x = fmaf(t, t, A.s[2].x); A.s[3].x = fmaf(val, val, A.s[3].x); A.s[4].x = fmaf(t, val, A.s[4].x);
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const float g = G[r], tg = t * g, wg = val * g;
            A.P[0][r].x += g; A.P[1][r].x += tg; A.P[2][r].x += wg;
            A.Q[0][r].x = fmaf(zf, g, A.Q[0][r].x); A.Q[1][r].x = fmaf(zf, tg, A.Q[1][r].x); A.Q[2][r].x = fmaf(zf, wg, A.Q[2][r].x);
        }
    }
    return val;
}

// Work decomposition.  A COLUMN is the full z-run of tiles at one (pair, y-tile, x-tile).  Columns are
// numbered (pair, y, x) with x fastest and dealt out cyclically: in round r CTA b owns column r*G + b, so
// at any moment the G CTAs sit on G x/y-adjacent columns at about the same z and the halo one CTA needs
// was just fetched by its neighbour (L2 hit); a thread keeps its (x, y) for a whole column (one fold of
// its sums per ~200 voxels).  The columns left after the last full round are cut into contiguous tile
// spans (z fastest), one per CTA, so every SM stays busy to within one tile.
struct TileIter {
    int phase;                   // 0: full-column rounds, 1: tail span, 2: done
    int r;                       // round
    long long tt, tt_end;        // tail tile index / end of this CTA's tail span
    int cg, tz_i;                // global column index, z-tile
};
__device__ __forceinline__ void iter_enter_tail(TileIter &it, const TmaParams &p, int b, int G)
{
    it.tt = p.tail_tiles * (long long)b / G;
    it.tt_end = p.tail_tiles * (long long)(b + 1) / G;
    if (it.tt >= it.tt_end) { it.phase = 2; return; }
    it.phase = 1;
    const int c = (int)(it.tt / p.tiles_z);
    it.cg = p.full_rounds * G + c;
    it.tz_i = (int)(it.tt - (long long)c * p.tiles_z);
}
__device__ __forceinline__ void iter_begin(TileIter &it, const TmaParams &p, int b, int G)
{
    it.r = 0; it.tt = it.tt_end = 0; it.tz_i = 0;
    if (p.full_rounds > 0) { it.phase = 0; it.cg = b; }
    else iter_enter_tail(it, p, b, G);
}
__device__ __forceinline__ bool iter_next(TileIter &it, const TmaParams &p, int b, int G)     // true: column changed / done
{
    if (it.phase == 0) {
        if (++it.tz_i < p.tiles_z) return false;
        it.tz_i = 0;
        if (++it.r < p.full_rounds) it.cg = it.r * G + b;
        else iter_enter_tail(it, p, b, G);
        return true;
    }
    if (++it.tt >= it.tt_end) { it.phase = 2; return true; }
    if (++it.tz_i < p.tiles_z) return false;
    it.tz_i = 0;
    ++it.cg;
    return true;
}

constexpr int kMaxTmaPairs = 1024;       // pairs per launch of the TMA kernel (touched-pair bitmask)
constexpr int kMaxCachedPairs = 64;     // coordinate maps kept in smem (12 floats per pair)

__device__ __forceinline__ Coef load_coef(const float *coef_s, const TmaParams &p, int pair)
{
    Coef k;
    if (p.n_pairs <= kMaxCachedPairs) {
        const float *c = coef_s + pair * 12;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
#pragma unroll
            for (int j = 0; j < 3; ++j) k.A[r][j] = c[r * 4 + j];
            k.C[r] = c[r * 4 + 3];
        }
    } else {
        const float *st = p.a.state + (size_t)pair * TRB_STATE_FLOATS + TRB_STATE_THETA;
        float th[12];
#pragma unroll
        for (int i = 0; i < 12; ++i) th[i] = __ldcg(st + i);
        k = make_coef(th, p.a.D, p.a.H, p.a.W);
    }
    return k;
}

// Per-column constants of the footprint bound: the box needed by z-tile k of a column is
// [lo_r + k*step_r, hi_r + k*step_r] per source axis r.  Computed once per column (table look-ups and the
// theta coefficients are off the per-tile path), kept per warp in smem, 12 words.
struct ColConst {
    float lo[3], hi[3], step[3];
    int pair, x0, y0;
};

__device__ __forceinline__ void compute_col(ColConst &c, const TileIter &t, const TmaParams &p, const float *coef_s,
                                            float inv_d2, float zoff)
{
    const int W = p.a.W, H = p.a.H;
    const int pair = t.cg / p.cols_per_pair;
    const int col = t.cg - pair * p.cols_per_pair;
    const Coef k = load_coef(coef_s, p, pair);
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

// Decide whether the tile's source footprint fits the TMA box, publish the box origin and start the loads
// for `stage`.  Executed by ONE lane; ~40 instructions (the per-column part lives in ColConst).
template <int BX, int BY, int BZ>
__device__ __forceinline__ void issue_tile(int tz_i, const ColConst &c, const TmaParams &p, unsigned char *stg,
                                           uint64_t *full, TileMeta *meta, const CUtensorMap *map_mov,
                                           const CUtensorMap *map_tgt)
{
    using L = SmemLayout<BX, BY, BZ>;
    int o[3];
    bool fits = true;
    const int B[3] = {BX, BY, BZ};
    const float kf = (float)tz_i;
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const float lo = fmaf(kf, c.step[r], c.lo[r]), hi = fmaf(kf, c.step[r], c.hi[r]);
        // keep the float->int conversions defined for wild thetas
        const float loc = fminf(fmaxf(lo, -1.0e6f), 1.0e6f), hic = fminf(fmaxf(hi, -1.0e6f), 1.0e6f);
        // TMA needs the box start 16-byte aligned along x (tools/tma_probe.cu: an unaligned innermost
        // coordinate raises an illegal-instruction fault); y and z are free
        o[r] = r == 0 ? 4 * (int)floorf(loc * 0.25f) : (int)floorf(loc);
        fits = fits && ((int)floorf(hic) + 1 <= o[r] + B[r] - 1);
    }
    // the fp32 index trick needs |x + BX*y + BX*BY*z| < 2^21
    fits = fits && (fabsf((float)o[0]) + BX * fabsf((float)o[1]) + (float)(BX * BY) * fabsf((float)o[2]) < 1.9e6f);
    TileMeta m;
    m.ox = o[0]; m.oy = o[1]; m.oz = o[2]; m.fits = fits ? 1 : 0;
    *meta = m;
    const unsigned tgt_bytes = L::kTgtFloats * 4, box_bytes = L::kBoxFloats * 4;
    mbar_arrive_expect_tx(full, fits ? (tgt_bytes + box_bytes) : tgt_bytes);
    if (fits) tma_load_4d(stg, map_mov, full, o[0], o[1], o[2], c.pair);
    tma_load_4d(stg + L::kBoxFloats * 4, map_tgt, full, c.x0, c.y0, p.a.s_begin + tz_i * TZ, c.pair);
}

// sum 41 per-lane values over the warp.  The first 32 are reduced "transposed" (recursive halving:
// 31 shuffles instead of 160); lane l ends up holding the warp total of value l.
__device__ __forceinline__ void warp_reduce_moments(const float (&acc)[TRB_MOMENTS], float *dst /*[41] smem*/, int lane)
{
    float v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = acc[i];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < off; ++i) {
            const float send = up ? v[i] : v[i + off];
            const float keep = up ? v[i + off] : v[i];
            v[i] = keep + __shfl_xor_sync(kFull, send, off);
        }
    }
    dst[lane] = v[0];
#pragma unroll
    for (int i = 32; i < TRB_MOMENTS; ++i) {
        const float r = warp_sum(acc[i]);
        if (lane == 0) dst[i] = r;
    }
}

// the same with the nine values beyond 32 reduced "transposed" as well (padded to 16: 16 shuffles instead of 45)
__device__ __forceinline__ void warp_reduce_moments2(const float (&acc)[TRB_MOMENTS], float *dst /*[41] smem*/, int lane)
{
    float v[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = acc[i];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const bool up = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < off; ++i) {
            const float send = up ? v[i] : v[i + off];
            const float keep = up ? v[i + off] : v[i];
            v[i] = keep + __shfl_xor_sync(kFull, send, off);
        }
    }
    dst[lane] = v[0];
    float w[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) w[i] = (32 + i < TRB_MOMENTS) ? acc[32 + i] : 0.f;
#pragma unroll
    for (int off = 16, cnt = 16; off >= 1; off >>= 1) {
        const bool up = (lane & off) != 0;
        if (cnt > 1) {
            const int half = cnt / 2;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                if (i < half) {
                    const float send = up ? w[i] : w[i + half];
                    const float keep = up ? w[i + half] : w[i];
                    w[i] = keep + __shfl_xor_sync(kFull, send, off);
                }
            }
            cnt = half;
        } else {
            w[0] += __shfl_xor_sync(kFull, w[0], off);
        }
    }
    // lane l holds value 32 + ((l >> 1) & 15) (lanes l and l ^ 1 the same total)
    const int idx = 32 + ((lane >> 1) & 15);
    if ((lane & 1) == 0 && idx < TRB_MOMENTS) dst[idx] = w[0];
}

// ---- host side ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static inline EncodeTiledFn encode_fn()
{
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            return nullptr;
        fn = (EncodeTiledFn)ptr;
    }
    return fn;
}

// 4-D map over [pair][D][H][W] fp32 with a (bx,by,bz,1) box; out-of-range elements read as zero
static inline int make_map(CUtensorMap *map, const float *base, int n_pairs, long long pair_stride, int D, int H, int W,
                    int bx, int by, int bz)
{
    EncodeTiledFn enc = encode_fn();
    if (!enc) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return TRB_ERR_UNSUPPORTED; }
    const cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)n_pairs};
    const cuuint64_t strides[3] = {(cuuint64_t)W * 4, (cuuint64_t)W * H * 4,
                                   (cuuint64_t)(n_pairs > 1 ? pair_stride : (long long)W * H * D) * 4};
    const cuuint32_t box[4] = {(cuuint32_t)bx, (cuuint32_t)by, (cuuint32_t)bz, 1};
    const cuuint32_t estr[4] = {1, 1, 1, 1};
    CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, (void *)base, dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return TRB_ERR_UNSUPPORTED; }
    return TRB_OK;
}

}  // namespace trb
