// Brick geometry, brick keys and payload conventions shared by the partition and tile kernels of the sorted deposit
// (deposit_sorted.cu).
#pragma once
#include "apk_common.cuh"
#include "deposit_common.cuh"
#include <algorithm>
#include <cstdint>
#include <type_traits>

namespace apk {

// Brick edge in cells along x, y.  24 x 8 since the end of round 2 (GPU calls 30 - 31, config 3 / config 2, ms per step):
// 12 x 6: 47.4 / 3.29, 12 x 12: 46.7 / 3.23, 16 x 12: 46.4 / 3.15, 12 x 16: 46.4 / 3.17, 24 x 8: 46.3 / 3.15, 8 x 6: 48.1 --
// larger bricks give the partition longer runs of equal keys (scatter 6.9 -> 6.4 ms) and the tile kernel less halo per
// home cell; the tile must stay below the 48 KB of static shared memory.
#ifndef APK_BX
#define APK_BX 24
#endif
#ifndef APK_BY
#define APK_BY 8
#endif
constexpr int BX = APK_BX, BY = APK_BY;
constexpr int BZ = 32;                          // z-lanes of a column = tile cells along z (one warp)
// home cells of a brick along z: a column's 32 lanes are exactly its 32 tile cells -- the home cells, the S - 1 halo
// cells of the window and, for the interlaced pair (PAIR), one more: the twin's home cell is the same cell or the
// NEXT one along each axis, so ONE filing of every particle (under the brick of its mesh-0 home cell) serves both
// meshes when the tile is one cell longer per axis.  29 / 30 (TSC), 30 / 31 (CIC).
template <int S, bool PAIR> struct BrickZ { static constexpr int CELLS = BZ - (S - 1) - (PAIR ? 1 : 0); };
struct P3 { float x, y, z; };
struct P4 { float x, y, z, m; };

struct BrickGrid {
    int nbx, nby, nbz;   // bricks per axis (x counts local planes for slab plans)
    int nbricks;
    int zcells;          // home cells of a brick along z
    float edge[3];       // brick edge per axis, as floats, with 1 / edge and 0.5 / edge - 0.5 (see brick_keys_f32)
    float inv_edge[3], half_edge[3];
};

static inline BrickGrid make_brick_grid(const DepositGeom &G, int S, bool pair) {
    BrickGrid B;
    B.zcells = BZ - (S - 1) - (pair ? 1 : 0);
    B.nbx = (G.nplanes + BX - 1) / BX;
    B.nby = (G.N + BY - 1) / BY;
    B.nbz = (G.N + B.zcells - 1) / B.zcells;
    B.nbricks = B.nbx * B.nby * B.nbz;
    const int e[3] = {BX, BY, B.zcells};
    for (int d = 0; d < 3; ++d) {
        B.edge[d] = (float)e[d];
        B.inv_edge[d] = 1.f / (float)e[d];
        B.half_edge[d] = 0.5f / (float)e[d] - 0.5f;
    }
    return B;
}

// Payload convention (both paths below): l[d] = the particle's coordinate relative to its brick, in cells, such that
// the home cell of mesh 0 inside the brick is rint(l) for TSC and rint(l - 0.5) for CIC, up to ties -- a particle
// within rounding of a cell boundary may be filed under either neighbour, and under the neighbouring BRICK at a brick
// boundary; the tile kernel clamps the home cell to the brick, and the window polynomials are continuous across the
// boundary, so the deposited weights differ by O(eps^2).  The interlaced twin (mesh 1) uses l + 0.5.

// float64 positions (and float32 ones far outside the box): g = x * scale + shift as the oracle forms it.
template <int S>
__device__ __forceinline__ unsigned int brick_of(const double (&x)[3], const DepositGeom &G,
                                                 const BrickGrid &B, float (&l)[3]) {
    if (!owned_by_slab(__dmul_rn(x[0], G.scale), G)) return 0xffffffffu;         // slab plans: not this rank's particle
    int b[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const double g = grid_coord(x[d], G);
        const double r = rint(S == 2 ? g - 0.5 : g);                    // anchor: mesh 0's home cell
        int hl = wrap_index((long long)r, G.N);
        if (d == 0 && G.slab) {
            hl -= G.plane0;
            if (hl < 0) hl += G.N; else if (hl >= G.N) hl -= G.N;
            if (hl >= G.nplanes) hl = 0;                                // unreachable for owned particles
        }
        const int edge = d == 0 ? BX : (d == 1 ? BY : B.zcells);
        b[d] = hl / edge;
        l[d] = (float)(g - r) + (float)(hl - b[d] * edge);
    }
    return (unsigned int)((b[0] * B.nby + b[1]) * B.nbz + b[2]);
}

// float32 positions without any float64, conversion or integer-division instruction (the partition kernels are
// issue-bound): ~20 FP32 instructions per axis.
//   g = x * scale is carried as p + e, p = fl(x * s0), e = the exact rounding error of p plus x * (s1 + s2)
//     (scale = s0 + s1 + s2): an error-free product good to ~2^-70;
//   anchor r = rint(p + shift') by the magic-constant add (ties irrelevant, see above); p - r is exact;
//   periodic wrap a mod N by one more rint (any |g| < 2^20; beyond that -> false, float64 path);
//   brick b = rint((a + 0.5) / edge - 0.5) = floor((a + 0.5) / edge): the argument is never within 0.5 / edge of a tie;
//   all indices are small integers held exactly in float registers; the key needs nbricks < 2^23.
// Returns false if the particle has to take the float64 path.
template <int S>
__device__ __forceinline__ bool brick_keys_f32(const float *x, const DepositGeom &G, const BrickGrid &B,
                                               unsigned int &key, float (&l)[3]) {
    const float M = 12582912.f;                      // 1.5 * 2^23: (v + M) - M = rint(v) for |v| < 2^22
    const float Nf = (float)G.N, invN = 1.f / Nf, hN = 0.5f * invN - 0.5f;
    const float shift = G.t32 - (S == 2 ? 0.f : 0.5f);
    const float tt = G.t32 - 0.5f;                   // anchor = rint(g + tt): floor(g + shift + 0.5) TSC, floor(g + shift) CIC
    bool far = false, owned = true;
    float b[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) {
        const float p = __fmul_rn(x[d], G.s0);       // intrinsics: never contracted into an FMA
        float e = fmaf(x[d], G.s0, -p);
        e = fmaf(x[d], G.s1, e);
        e = fmaf(x[d], G.s2, e);
        const float r = __fsub_rn(__fadd_rn(__fadd_rn(p, tt), M), M);
        // periodic wrap for positions any number of box lengths outside the box (folded boxes: x -> 2^f x mod L):
        // a -= N * floor((a + 0.5) / N), the floor again as rint(. - 0.5) (never within 0.5 / N of a tie; the
        // float error of the quotient stays below that for |a| < 2^20)
        far |= !(fabsf(p) < 1048576.f);
        float a = fmaf(-Nf, __fsub_rn(__fadd_rn(fmaf(r, invN, hN), M), M), r);
        if (d == 0 && G.slab) {
            const float h = floorf(p);               // ownership: floor of the UNSHIFTED coordinate
            const int hu = (int)(h + floorf(__fadd_rn(__fsub_rn(p, h), e)));
            const int rel = wrap_near(hu, G.N, far) - G.own0;
            owned = rel >= 0 && rel < G.nown;
            a -= (float)G.plane0;                    // local plane index
            a = a < 0.f ? a + Nf : a;
            a = a >= Nf ? a - Nf : a;
            a = a >= (float)G.nplanes ? 0.f : a;     // unreachable for owned particles
        }
        const float bq = __fsub_rn(__fadd_rn(fmaf(a, B.inv_edge[d], B.half_edge[d]), M), M);
        b[d] = bq;
        l[d] = fmaf(-B.edge[d], bq, a) + __fadd_rn(__fsub_rn(p, r), __fadd_rn(shift, e));
    }
    const float k = fmaf(fmaf(b[0], (float)B.nby, b[1]), (float)B.nbz, b[2]);
    key = owned ? (__float_as_uint(__fadd_rn(k, 8388608.f)) & 0x7fffffu) : 0xffffffffu;
    return !far;
}

// key and brick-local coordinates of one particle
template <int S, typename PT>
__device__ __forceinline__ void brick_keys(const PT *x, const DepositGeom &G, const BrickGrid &B, unsigned int &key,
                                           float (&l)[3]) {
    if constexpr (std::is_same<PT, float>::value) {
        if (G.t32 >= 0.f && B.nbricks < (1 << 23)) {
            if (brick_keys_f32<S>(x, G, B, key, l)) return;
        }
    }
    const double xd[3] = {(double)x[0], (double)x[1], (double)x[2]};
    key = brick_of<S>(xd, G, B, l);
}

// raw coordinates of this thread's 4 particles of a tile, v[3*k + d]: slice k of the tile is the
// PART_THREADS consecutive particles base + k*PART_THREADS + tid, so the 32 lanes of a warp always hold 32
// CONSECUTIVE particles (long runs of equal brick keys, coalesced 4-byte loads).  All 12 loads are
// issued up front; indices are clamped to np-1 and masked by the caller.
template <typename PT> struct Raw4 { PT v[12]; };

template <typename PT, bool SOA>
__device__ __forceinline__ void load4(const PT *__restrict__ p0, const PT *__restrict__ p1,
                                      const PT *__restrict__ p2, long long first, int stride, long long np,
                                      Raw4<PT> &r) {
    if (first - threadIdx.x + 4LL * stride <= np) {        // whole tile inside the set (uniform): one 64-bit address
        if (SOA) {                                         // per array, the four slices at immediate offsets
            const PT *a0 = p0 + first, *a1 = p1 + first, *a2 = p2 + first;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                r.v[3 * k] = __ldcs(a0 + k * stride); r.v[3 * k + 1] = __ldcs(a1 + k * stride); r.v[3 * k + 2] = __ldcs(a2 + k * stride);
            }
        } else {
            const PT *a0 = p0 + 3 * first;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                r.v[3 * k] = __ldcs(a0 + 3 * k * stride); r.v[3 * k + 1] = __ldcs(a0 + 3 * k * stride + 1); r.v[3 * k + 2] = __ldcs(a0 + 3 * k * stride + 2);
            }
        }
        return;
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const long long p = min(first + (long long)k * stride, np - 1);
        if (SOA) { r.v[3 * k] = __ldcs(p0 + p); r.v[3 * k + 1] = __ldcs(p1 + p); r.v[3 * k + 2] = __ldcs(p2 + p); }
        else     { r.v[3 * k] = __ldcs(p0 + 3 * p); r.v[3 * k + 1] = __ldcs(p0 + 3 * p + 1); r.v[3 * k + 2] = __ldcs(p0 + 3 * p + 2); }
    }
}

// run-length aggregation inside a warp: lanes holding the same key as their left neighbour form a
// run; returns the run's head lane and this lane's offset in it (keys of a snapshot are coherent,
// so runs are long; for random keys every lane is its own run)
__device__ __forceinline__ void warp_runs(unsigned int key, int lane, int &head, int &offset, int &length) {
    const unsigned int prev = __shfl_up_sync(0xffffffffu, key, 1);
    const unsigned int heads = __ballot_sync(0xffffffffu, lane == 0 || key != prev);
    const unsigned int below = heads & ((2u << lane) - 1u);          // heads at or below this lane
    head = 31 - __clz(below);
    offset = lane - head;
    const unsigned int above = heads & ~((2u << lane) - 1u);          // heads above this lane
    const int next = above ? __ffs(above) - 1 : 32;
    length = next - head;
}

// a brick partition of a particle set, left in the plan workspace by the count, scan and scatter kernels
// (deposit_sorted.cu): payload records (P3 / P4) filed by brick, brick_start[nbricks + 1], the non-empty bricks
// filled[0 .. *nfilled).
// Fixed-slot layout (slots != 0): brick b's records are [b slots, b slots + fixed_count[b]) unless the device word
// fixed_count[B.nbricks] is set -- then a brick held more than `slots` particles and brick_start describes the
// partition as above.
struct BrickPartition {
    const void *vals;
    const unsigned int *brick_start, *filled, *nfilled;
    BrickGrid B;
    const unsigned int *fixed_count = nullptr;
    unsigned int slots = 0;
};

constexpr int PART_THREADS = 256;
constexpr int PART_ITEMS = 4;    // consecutive particles per thread per tile

}  // namespace apk
