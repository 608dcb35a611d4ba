// Particle -> mesh mass assignment, sorted / shared-memory-tiled variant (APK_DEPOSIT_SORTED).
//
// Replaces pm.paint(pos, mass=, resampler=) as astrild calls it at
//   /root/reference/src/astrild/particles/hutils/stats_subfind.py:130-131
// (pmesh 0.1.55 CIC / TSC windows, see deposit_common.cuh).
//
// Bound: HBM.  Algorithmic bytes = Np*(12 + 4*[mass]) + 4*N^3 (SURVEY.md section 8d); the sort
// traffic is real but not credited.
//
// Pipeline (all on one stream, no host sync):
//   1. brick_count_kernel   every particle -> key of the brick (24 x 8 x 29..31 home cells) that holds its mesh-0 HOME
//                           cell; per-brick counts with one RED per warp-run of equal keys (snapshot order is spatially
//                           coherent).  float32 positions: ~40 FP32 instructions per particle, no float64, no
//                           conversions, no integer division (brick_keys_f32); float64 positions: the oracle's expression.
//   2. brick_scan_kernel    exclusive scan of the counts -> brick_start[], cursors, list of non-empty bricks.
//   3. brick_scatter_kernel keys are recomputed (never stored); each run of equal keys claims its slots with ONE
//                           atomicAdd on the brick's cursor and writes its payload = brick-local coordinates as
//                           3 floats (+ mass), contiguously.  One read and one write of the particles replace a
//                           multi-pass radix sort; order inside a brick is arbitrary (the deposit does not care).
//                           (One array per coordinate instead of 12-byte records, round 2 call 34: the tile kernel's
//                           loads become one wavefront each, 20.5 -> 20.2 ms, but the scatter writes three streams of
//                           short runs: 6.4 -> 11.1 ms.  Records kept.)
//      Interlaced pair (apk_deposit_interlaced): the SAME partition and the same 12-byte payload serve both meshes --
//      the twin's home cell is the same cell or the next one per axis, so its tile is one cell longer per axis
//      (bricks hold one z-cell less) and its coordinates are the payload's + 0.5.  No second copies, no flags.
//   4. brick_tile_kernel    one CTA per non-empty brick, one THREAD per particle, the brick's window of the mesh as
//                           fixed-point integers in shared memory, native ATOMS.ADD, bank-aware walking order (see
//                           the kernel's comment).
//      Tried and removed in round 2 (profiles/r02_measurements.md): a one-pass partition into paged buckets (21.7 ms
//      against 7.5 + 9.4 ms for count + scatter at 1024^3, and it can dead-lock on randomly ordered input); filing the
//      twin's boundary particles twice with sign flags (14 % more payload, ~110 more instructions per particle in
//      each partition pass).
#include "brick_common.cuh"
#include <algorithm>
#include <cstdint>
#include <type_traits>

namespace apk {


template <int S, typename PT, bool SOA>
__global__ void __launch_bounds__(PART_THREADS)
brick_count_kernel(const PT *__restrict__ p0, const PT *__restrict__ p1, const PT *__restrict__ p2, long long np,
                   DepositGeom G, BrickGrid B, unsigned int *__restrict__ counts) {
    const int lane = threadIdx.x & 31;
    const long long tile = (long long)PART_THREADS * PART_ITEMS;
    const long long step = (long long)gridDim.x * tile;
    long long base = (long long)blockIdx.x * tile;
    Raw4<PT> nxt;
    if (base < np) load4<PT, SOA>(p0, p1, p2, base + threadIdx.x, PART_THREADS, np, nxt);
    for (; base < np; base += step) {
        const long long first = base + threadIdx.x;
        const Raw4<PT> cur = nxt;
        if (base + step < np) load4<PT, SOA>(p0, p1, p2, first + step, PART_THREADS, np, nxt);   // next tile in flight
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float l[3];
            unsigned int key;
            brick_keys<S, PT>(cur.v + 3 * k, G, B, key, l);
            if (first + (long long)k * PART_THREADS >= np) key = 0xffffffffu;
            int head, offset, length;
            warp_runs(key, lane, head, offset, length);
            if (key != 0xffffffffu && offset == 0) atomicAdd(counts + key, (unsigned int)length);
        }
    }
}

// exclusive scan of counts[0..n) -> start[0..n], cursor[0..n) = start, in two launches of n / SCAN_SEG CTAs:
// per-segment totals, then every CTA sums the totals below it and scans its own segment (n is 10^4..10^7)
constexpr int SCAN_PER = 8, SCAN_SEG = 1024 * SCAN_PER;

__device__ __forceinline__ unsigned int block_exclusive_scan_1024(unsigned int s, unsigned int *wsum, unsigned int &total) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    unsigned int incl = s;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const unsigned int w = wsum[lane];
        unsigned int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        wsum[lane] = wi - w;
        if (lane == 31) wsum[32] = wi;
    }
    __syncthreads();
    total = wsum[32];
    const unsigned int excl = wsum[warp] + incl - s;
    __syncthreads();
    return excl;
}

__global__ void __launch_bounds__(1024)
brick_segsum_kernel(const unsigned int *__restrict__ counts, int n, unsigned int *__restrict__ seg_total,
                    unsigned int *__restrict__ seg_filled) {
    __shared__ unsigned int wsum[33];
    const int a = min(blockIdx.x * SCAN_SEG + threadIdx.x * SCAN_PER, n), b = min(a + SCAN_PER, n);
    unsigned int s = 0, f = 0;
    for (int i = a; i < b; ++i) { const unsigned int c = counts[i]; s += c; f += c != 0u; }
    unsigned int total, filled;
    block_exclusive_scan_1024(s, wsum, total);
    block_exclusive_scan_1024(f, wsum, filled);
    if (threadIdx.x == 0) { seg_total[blockIdx.x] = total; seg_filled[blockIdx.x] = filled; }
}

// also lists the non-empty bricks (filled[0..nfilled), ascending) so that the deposit kernel never visits an
// empty one: slab plans, halo catalogues and the particles received from other ranks leave most bricks empty
__global__ void __launch_bounds__(1024)
brick_scan_kernel(const unsigned int *__restrict__ counts, int n, const unsigned int *__restrict__ seg_total,
                  const unsigned int *__restrict__ seg_filled, unsigned int *__restrict__ start,
                  unsigned int *__restrict__ cursor, unsigned int *__restrict__ filled, unsigned int *__restrict__ nfilled) {
    __shared__ unsigned int wsum[33];
    unsigned int below = 0, fbelow = 0, base, fbase, total, ftotal;
    for (int i = threadIdx.x; i < (int)blockIdx.x; i += 1024) { below += seg_total[i]; fbelow += seg_filled[i]; }
    block_exclusive_scan_1024(below, wsum, base);       // base = sum of the segments below this one
    block_exclusive_scan_1024(fbelow, wsum, fbase);
    const int a = min(blockIdx.x * SCAN_SEG + threadIdx.x * SCAN_PER, n), b = min(a + SCAN_PER, n);
    unsigned int v[SCAN_PER], s = 0, f = 0;
#pragma unroll
    for (int k = 0; k < SCAN_PER; ++k) { v[k] = a + k < b ? counts[a + k] : 0u; s += v[k]; f += v[k] != 0u; }
    unsigned int run = base + block_exclusive_scan_1024(s, wsum, total);
    unsigned int frun = fbase + block_exclusive_scan_1024(f, wsum, ftotal);
#pragma unroll
    for (int k = 0; k < SCAN_PER; ++k)
        if (a + k < b) {
            start[a + k] = run; cursor[a + k] = run; run += v[k];
            if (v[k] != 0u) filled[frun++] = (unsigned int)(a + k);
        }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 1023) { start[n] = base + total; *nfilled = fbase + ftotal; }
}

// float32 positions: 4 CTAs per SM (64 registers, no spills; measured 6.9 against 7.2 ms at 1024^3 with 3); float64: 3
#ifndef APK_SCATTER_MIN_CTAS
#define APK_SCATTER_MIN_CTAS (sizeof(PT) == 4 ? 4 : 3)
#endif
template <int S, typename PT, bool SOA, bool MASS, typename VT>
__global__ void __launch_bounds__(PART_THREADS, APK_SCATTER_MIN_CTAS)
brick_scatter_kernel(const PT *__restrict__ p0, const PT *__restrict__ p1, const PT *__restrict__ p2,
                     const void *__restrict__ mass, int mass_f64, long long np, DepositGeom G,
                     BrickGrid B, unsigned int *__restrict__ cursor, VT *__restrict__ vals) {
    const int lane = threadIdx.x & 31;
    const long long tile = (long long)PART_THREADS * PART_ITEMS;
    const long long step = (long long)gridDim.x * tile;
    long long base = (long long)blockIdx.x * tile;
    Raw4<PT> nxt;
    if (base < np) load4<PT, SOA>(p0, p1, p2, base + threadIdx.x, PART_THREADS, np, nxt);
    for (; base < np; base += step) {
        const long long first = base + threadIdx.x;
        const Raw4<PT> cur = nxt;
        if (base + step < np) load4<PT, SOA>(p0, p1, p2, first + step, PART_THREADS, np, nxt);   // next tile in flight
        // Software pipeline of depth one: item k claims its slots (returning atomics, ~600 cycles) and item k-1,
        // whose slots have arrived meanwhile, is stored.
        VT pv = {};
        unsigned int pslot = 0;
        int phead = 0, poffset = 0;
        bool plive = false;
#pragma unroll
        for (int k = 0; k <= 4; ++k) {
            VT v = {};
            unsigned int slot = 0;
            int head = 0, offset = 0, length = 0;
            bool live = false;
            if (k < 4) {
                const long long p = first + (long long)k * PART_THREADS;
                float l[3];
                unsigned int key;
                brick_keys<S, PT>(cur.v + 3 * k, G, B, key, l);
                if (p >= np) key = 0xffffffffu;
                live = key != 0xffffffffu;
                v.x = l[0]; v.y = l[1]; v.z = l[2];
                if constexpr (MASS) {
                    const long long pc = min(p, np - 1);
                    v.m = mass_f64 ? (float)((const double *)mass)[pc] : ((const float *)mass)[pc];
                }
                warp_runs(key, lane, head, offset, length);
                if (live && offset == 0) slot = atomicAdd(cursor + key, (unsigned int)length);
            }
            if (k > 0) {
                const unsigned int ps = __shfl_sync(0xffffffffu, pslot, phead) + poffset;
                if (plive) vals[ps] = pv;
            }
            pv = v; pslot = slot; phead = head; poffset = offset; plive = live;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Tile kernel: one CTA per brick, one THREAD per particle.  The brick's window of the mesh lives in shared memory as
// 32-bit FIXED-POINT integers and every one of the S^3 weights goes there with a native integer ATOMS.ADD (measured on
// B200, tools/ubench/atoms.cu: 0.7 cycles per warp-instruction and SM when the 32 lanes hit 32 banks, 0.7 k when k lanes
// share a bank -- the SAME address counts like any other bank conflict -- and ~1.9 for random cells; the float atomicAdd
// is a CAS loop at 3.5 - 9.6).  No in-brick sort, no per-cell loop: all 32 lanes work on every instruction, whatever the
// cell occupancy.  ncu (profiles/): the shared-memory pipe is what bounds this kernel (88 - 92 % busy, 85 % of its
// wavefronts are the ATOMS'); its time follows the number of ATOMS wavefronts, i.e. the largest number of lanes on one
// bank per instruction: 3.1 - 3.3 when every lane walks its window in the same order (input order, shuffled and
// cell-sorted sets within 10 %, the cell-sorted one slowest).
//   Rotation (TSC; round 2, GPU calls 24 - 29): lanes whose windows START on the same bank collide on all 27 updates.
//   They are ranked with one MATCH.ANY + POPC per particle, and the k-th of them walks the x-planes of its window
//   starting with plane k mod 3; the tile's x-planes are 11 banks apart (bank = z + 11 x), so those lanes now sit on
//   different banks at every step.  2.59 wavefronts per ATOMS (from 3.3 at 512^3), 20.7 ms for both meshes of config 3
//   (from 24.1).  Measured and not kept: the rank from five ballots instead of MATCH (same time); skews 3, 5, 9, 13
//   (within 2 %); rotating the y-rows as well by the next digit of the rank, on a tile skewed (9 x + 3 y + z) (25.1 ms:
//   the 9 extra selects); k-th lane -> plane min(k, 2) or k & 1 (22.3 - 23.1 ms); 7 - 8 CTAs per SM at 32 registers, 128
//   or 512 threads per brick (+- 0.5 %); CIC, with 8 updates per particle, loses to the vote (0.70 -> 0.95 ms at 512^3)
//   and keeps the plain order.  A CPU model of the bench set (max lanes per bank over the 27 steps, particles in the
//   scatter's arrival order) gives 3.13 -> 2.13 for this rule and 2.06 for a greedy choice among all 27 digit-wise
//   rotations: the family is exhausted; only a cyclic walk (lane L on bank L + t at step t) would be conflict-free, and
//   that needs the 27 weights indexed by a per-lane offset, i.e. dynamic register indexing.
//   Quantum: 2^-s of the largest |mass| in the chunk (1 for unit masses), s chosen PER CHUNK of <= TILE_FLUSH particles
//   as large as 32 bits allow if every particle of the chunk put its largest possible weight (1 for CIC, 0.75^3 for
//   TSC) into one cell: s = 20 for the ~5600 particles of a brick at one particle per cell (TSC), 20 for a full
//   chunk, up to 24 for sparse bricks.
//   Unit masses: the float -> fixed conversion costs nothing.  The three axis weights carry the factors 2^-40, 2^-40 and
//   2^(s - 69), so the product of the three is w * 2^(s - 149): a SUBNORMAL float whose bit pattern IS the integer
//   rint(w * 2^s) (the one rounding of the last FMUL is to the subnormal grid, round-to-nearest-even; no intermediate is
//   subnormal).  One FMUL + one ATOMS.ADD per cell.  (Needs denormal support: the library is built without -ftz.)
//   Per-particle masses: FMUL + F2I (signed; the scale comes from the chunk's sum of |mass|).
//   Integer adds commute: a brick's contribution to the mesh does not depend on the order in which the partition
//   filed its particles.
//   The tile goes to the mesh as one coalesced 128-byte RED.ADD.F32 per (x,y) column, zeros skipped.
//   A conflict-free variant was built and measured (round 2, commit "Experiment: bank-queue tile kernel"): tile skewed so
//   that bank = (11 x + 5 y + z) mod 32, each chunk counting-sorted in shared memory into 32 queues by the bank of the
//   window's first cell, lane L working through queue L -- every ATOMS then hits 32 different banks.  Correct, but
//   28.8 against 24.0 ms for both meshes at 1024^3: the sort's own shared-memory traffic (a returning ATOMS, three
//   scattered STS and LDS per particle), its five barriers per chunk and the idle lanes of the shorter queues
//   (utilisation 0.72) cost more than the conflicts.  Removed.
#ifndef APK_TILE_FLUSH
#define APK_TILE_FLUSH 8191
#endif
constexpr int TILE_FLUSH = APK_TILE_FLUSH;            // particles between two flushes of the tile
#ifndef APK_TILE_THREADS
#define APK_TILE_THREADS 256
#endif
constexpr int TILE_THREADS = APK_TILE_THREADS;
#ifndef APK_TILE_CTAS
#define APK_TILE_CTAS 5
#endif

// APK_TILE_ROT (TSC only): 0 = every lane walks its window in the same order; 1 = lanes whose windows start on the same
// shared-memory bank walk the x-planes of their windows in rotated order, on a tile whose x-planes are APK_TILE_XSKEW
// banks apart (see the kernel's comment; 24.1 -> 21.2 ms for both meshes of config 3).
#ifndef APK_TILE_ROT
#define APK_TILE_ROT 1
#endif
#ifndef APK_TILE_XSKEW
#define APK_TILE_XSKEW 11
#endif
// The tile is [TX][TY] columns of TZ = 32 cells along z, YS = 32 words apart, x-planes XS words apart.  Without rotation
// XS = TY * 32: the bank of a cell is its z alone.  (Measured at 1024^3 without rotation: a column stride of 33 words is
// 15 % slower on snapshot-ordered input, 27.2 against 23.7 ms for both meshes, and so are larger bricks, 16 x 16 and
// 24 x 12: 25.8 - 27 ms.)  With rotation XS = XSKEW (mod 32): bank = (z + XSKEW * x) mod 32.
template <int S, bool PAIR> struct Tile {
    static constexpr int OFF = (S == 3) ? 1 : 0;      // window origin = home cell - OFF
    static constexpr int ROT = (S == 3) ? APK_TILE_ROT : 0;   // CIC: 8 updates per particle do not pay for the vote (0.70 -> 0.95 ms at 512^3)
    static constexpr int TX = BX + S - 1 + (PAIR ? 1 : 0), TY = BY + S - 1 + (PAIR ? 1 : 0), TZ = BZ, YS = 32;
    static constexpr int XS = TY * YS + (ROT ? ((APK_TILE_XSKEW - TY * YS) % 32 + 32) % 32 : 0);
    static constexpr int CELLS = (TX * XS + 3) & ~3;
    static constexpr bool PLANE_FLUSH = (S == 3);     // how the tile goes to the mesh (see the kernel)
};

// fractional bits for a chunk of n unit-mass particles: n * wmax * 2^s < 2^32, s <= SMAX (a single weight must stay
// below 2^24 quanta, where float bit patterns stop being linear in the value)
template <int S>
__device__ __forceinline__ int tile_frac_bits(int n) {
    constexpr float WMAX = (S == 3) ? 0.43f : 1.001f;          // 0.75^3 = 0.4219 / 1, padded for the rounding
    constexpr int SMAX = (S == 3) ? 24 : 23;
    const float room = (4294967296.f / WMAX) / (float)n;
    const int s = ((__float_as_int(room) >> 23) & 0xff) - 127;  // floor(log2(room))
    return min(s, SMAX);
}

// nearest brick-local home cell of coordinate l on one axis (clamped to the brick) as int, and the offset
// d = l - home: [-0.5, 0.5] for TSC, [0, 1] for CIC (ties land on either side; the windows are continuous there)
template <int S>
__device__ __forceinline__ void tile_home(float l, float last, float &d, int &h) {
    const float M = 12582912.f;                       // 1.5 * 2^23: adding it rounds to the nearest integer
    float t = (S == 2 ? l - 0.5f : l) + M;
    t = fminf(fmaxf(t, M), M + last);
    h = __float_as_int(t) & 0x3fffff;
    d = l - (t - M);
    // CIC: a coordinate within rounding of the brick's faces may leave [0, 1] by ~1e-5; the weights d and 1 - d must not
    // turn negative (the unit-mass path reads the bit pattern of the product as an unsigned integer).  TSC's are
    // squares and 0.75 - d^2: positive for any |d| < 0.86.
    if (S == 2) d = fminf(fmaxf(d, 0.f), 1.f);
}

// SEL: 0 = mesh 0 (or the only mesh), 1 = the interlaced twin (coordinates + 0.5, home cells one further); a template
// parameter so that the clamps and the shift are immediates (as a kernel argument they were re-derived per particle)
template <int S, bool MASS, bool PAIR, int SEL, typename VT>
__global__ void __launch_bounds__(TILE_THREADS, APK_TILE_CTAS)
brick_tile_kernel(const VT *__restrict__ vals, const unsigned int *__restrict__ brick_start,
                  const unsigned int *__restrict__ filled, const unsigned int *__restrict__ nfilled_ptr,
                  DepositGeom G, BrickGrid B, float *__restrict__ mesh) {
    static_assert(SEL == 0 || PAIR, "the twin exists only for the interlaced pair");
    using T = Tile<S, PAIR>;
    constexpr int ZC = BrickZ<S, PAIR>::CELLS;
    __shared__ __align__(16) unsigned int tile[T::CELLS];
    __shared__ float red_s[TILE_THREADS / 32];
    __shared__ double red_sd[TILE_THREADS / 32];
    __shared__ long long xoff[T::PLANE_FLUSH ? 1 : T::TX];   // table flush: mesh offset of the tile's x-planes (-1: outside the slab)
    __shared__ int yoff[T::PLANE_FLUSH ? 1 : T::TY];         // ... and of its y-rows
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned int lanes_below = (1u << lane) - 1u;
    constexpr float twin = SEL > 0 ? 0.5f : 0.f;
    constexpr float lastx = (float)(BX - 1 + (SEL > 0)), lasty = (float)(BY - 1 + (SEL > 0)), lastz = (float)(ZC - 1 + (SEL > 0));

    // One CTA per non-empty brick, in list order (x-major: neighbouring windows meet in L2).  CTAs retire all the
    // time, so kernels of a higher-priority stream (the slab path's FFT / transpose of the first mesh) get SMs while
    // this one runs.
    const unsigned int nfilled = *nfilled_ptr;
    for (unsigned int slot = blockIdx.x; slot < nfilled; slot += gridDim.x) {
        const unsigned int brick = filled[slot];
        const unsigned int pbeg = brick_start[brick], pend = brick_start[brick + 1];
        const int bz = brick % B.nbz;
        const int by = (brick / B.nbz) % B.nby;
        const int bx = brick / (B.nbz * B.nby);

        __syncthreads();                              // (persistent grids) the previous brick's flush is complete
        for (int i = tid; i < T::CELLS / 4; i += TILE_THREADS) reinterpret_cast<uint4 *>(tile)[i] = make_uint4(0u, 0u, 0u, 0u);
        int bad_home = -1;                            // home cell of this thread's last non-finite particle (x << 16 | y << 8 | z)
        if constexpr (!T::PLANE_FLUSH) {
            if (tid < T::TX) {
                int px = bx * BX - T::OFF + tid;
                bool ok = true;
                if (G.slab) ok = px >= 0 && px < G.nplanes;
                else px = wrap_index32(px, G.N);
                xoff[tid] = ok ? (long long)px * G.N * G.ldz : -1LL;
            } else if (tid < T::TX + T::TY) {
                yoff[tid - T::TX] = wrap_index32(by * BY - T::OFF + tid - T::TX, G.N) * G.ldz;
            }
        }
        __syncthreads();

        for (unsigned int c0 = pbeg; c0 < pend; c0 += TILE_FLUSH) {
            const unsigned int c1 = min(c0 + (unsigned int)TILE_FLUSH, pend);
            // ---- masses: unit = the power of two at or above the chunk's largest |mass| (scaling by it is exact), and
            //      the fixed-point scale from the chunk's sum of |mass|: no cell can overflow 31 bits + sign even if
            //      every particle put its largest weight into it.
            float unit = 1.f, inv_unit = 1.f, mscale = 1.f;
            int frac_bits = 0;
            if constexpr (MASS) {
                // NaN / inf masses count as 0 here (the particle loop sends them to the mesh as NaN); the sum is float64:
                // 8191 masses near FLT_MAX sum to ~3e42
                float top = 0.f;
                double sum = 0.0;
                for (unsigned int p = c0 + tid; p < c1; p += TILE_THREADS) {
                    const float m = fabsf(vals[p].m), a = m <= 3.4028235e38f ? m : 0.f;
                    top = fmaxf(top, a);
                    sum += (double)a;
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    top = fmaxf(top, __shfl_xor_sync(0xffffffffu, top, o));
                    sum += __shfl_xor_sync(0xffffffffu, sum, o);
                }
                if (lane == 0) { red_s[warp] = top; red_sd[warp] = sum; }
                __syncthreads();
                top = red_s[0]; sum = red_sd[0];
#pragma unroll
                for (int i = 1; i < TILE_THREADS / 32; ++i) { top = fmaxf(top, red_s[i]); sum += red_sd[i]; }
                // 2^ceil(log2(top)), clamped to normal numbers whose reciprocal is normal too
                int e = ((__float_as_int(top) >> 23) & 0xff) + ((__float_as_int(top) & 0x7fffff) ? 1 : 0);
                e = min(max(e, 2), 252);
                unit = __int_as_float(e << 23);
                inv_unit = __int_as_float((254 - e) << 23);
                if (!(top > 0.f)) { unit = 1.f; inv_unit = 0.f; sum = 1.0; }   // all-zero masses: nothing to add
                constexpr float WMAX = (S == 3) ? 0.43f : 1.001f;
                const float room = 2147483648.f / (WMAX * fmaxf((float)(sum * (double)inv_unit), 1.f));   // sum |m'| <= n, >= 1 when top > 0
                frac_bits = min(((__float_as_int(room) >> 23) & 0xff) - 127, 30);
                mscale = __int_as_float((127 + frac_bits) << 23);
            } else {
                frac_bits = tile_frac_bits<S>((int)(c1 - c0));
            }
            const float quantum = __int_as_float((127 - frac_bits) << 23) * unit;                         // 2^-s mass units
            // unit masses: axis factors 2^-40 (x), 2^-40 (y), 2^(s - 69) (z); masses: 1, 1, m * 2^s
            const float KXY = MASS ? 1.f : __int_as_float((127 - 40) << 23);
            const float KZ = MASS ? 1.f : __int_as_float((127 + frac_bits - 69) << 23);

            // ---- one thread per particle; the next particle's loads are in flight while this one is deposited ----
            // (with the rotation every lane of a warp makes the same number of trips: it votes across the warp)
            // (measured, call 36: the warp's 96 payload words loaded as three coalesced words per lane and handed to their
            // owners with three shuffles -- 3 + 3 instead of 3 x 2.2 wavefronts -- is slower, 20.76 against 20.25 ms for
            // both meshes: SHFL goes through the same pipe)
            unsigned int p = c0 + tid;
            VT nxt = {};
            if (p < c1) nxt = vals[p];
            for (; T::ROT ? p - lane < c1 : p < c1; p += TILE_THREADS) {
                const bool live = T::ROT ? p < c1 : true;
                const VT v = nxt;
                const unsigned int q = p + TILE_THREADS;
                if (q < c1) nxt = vals[q];
                float dx, dy, dz;
                int hx, hy, hz;
                tile_home<S>(v.x + twin, lastx, dx, hx);
                tile_home<S>(v.y + twin, lasty, dy, hy);
                tile_home<S>(v.z + twin, lastz, dz, hz);
                float kz = KZ;
                if constexpr (MASS) kz = (v.m * inv_unit) * mscale;              // |m / unit| <= 1, exact; times 2^s
                float wx[S], wy[S], wz[S];
                if (S == 2) {
                    wx[S - 1] = dx * KXY; wx[0] = KXY - wx[S - 1];
                    wy[S - 1] = dy * KXY; wy[0] = KXY - wy[S - 1];
                    wz[S - 1] = dz * kz;  wz[0] = kz - wz[S - 1];
                } else {
                    const float ax = 0.5f - dx, cx = 0.5f + dx, ay = 0.5f - dy, cy = 0.5f + dy, az = 0.5f - dz, cz = 0.5f + dz;
                    const float hxy = 0.5f * KXY, hz2 = 0.5f * kz;
                    wx[0] = (ax * hxy) * ax; wx[S / 2] = fmaf(-dx, dx, 0.75f) * KXY; wx[S - 1] = (cx * hxy) * cx;
                    wy[0] = (ay * hxy) * ay; wy[S / 2] = fmaf(-dy, dy, 0.75f) * KXY; wy[S - 1] = (cy * hxy) * cy;
                    wz[0] = (az * hz2) * az; wz[S / 2] = fmaf(-dz, dz, 0.75f) * kz;  wz[S - 1] = (cz * hz2) * cz;
                }
                const int origin = hx * T::XS + hy * T::YS + hz;                // window origin (home - OFF) in tile coordinates
                unsigned int *plane[S];
                if constexpr (T::ROT != 0) {
                    // Lanes whose windows start on the same bank collide on every one of the S^3 updates.  The k-th of
                    // them (MATCH.ANY + POPC) starts with x-plane k mod S of its window instead, XSKEW banks further per
                    // plane: the x weights and the plane pointers are rotated once per particle by selects (no dynamic
                    // register index), the S^3 updates keep their immediate offsets.
                    const unsigned int same = __match_any_sync(0xffffffffu, live ? (origin & 31) : 32 + lane);
                    const unsigned int rank = (unsigned int)__popc(same & lanes_below);                 // <= 31
                    const int rot = S == 3 ? (int)(rank - 3u * ((rank * 11u) >> 5)) : (int)(rank % (unsigned int)S);   // rank mod 3
                    float r[S];
#pragma unroll
                    for (int a = 0; a < S; ++a) {
                        float v = wx[a];
                        int xa = a;
#pragma unroll
                        for (int k = 1; k < S; ++k)
                            if (rot == k) { v = wx[(a + k) % S]; xa = (a + k) % S; }
                        r[a] = v;
                        plane[a] = tile + origin + xa * T::XS;
                    }
#pragma unroll
                    for (int a = 0; a < S; ++a) wx[a] = r[a];
                } else {
#pragma unroll
                    for (int a = 0; a < S; ++a) plane[a] = tile + origin + a * T::XS;
                }
                // A NaN or inf coordinate (its payload is NaN) or mass stays out of the integer tile, where it would
                // spoil the brick's other particles; the thread notes its home cell and puts a NaN there once the brick
                // is done.  Tested by comparison, never by how NaN converts to an integer (0 on the GPU, INT_MIN on x86).
                const bool finite = fabsf(v.x) + fabsf(v.y) + fabsf(v.z) + fabsf(kz) <= 3.4028235e38f;   // kz: m 2^s / unit
                if (live && !finite) bad_home = (hx << 16) | (hy << 8) | hz;
                if (live && finite) {
#pragma unroll
                    for (int a = 0; a < S; ++a)
#pragma unroll
                        for (int b = 0; b < S; ++b) {
                            const float wxy = wx[a] * wy[b];
#pragma unroll
                            for (int c = 0; c < S; ++c) {
                                const unsigned int fx = MASS ? (unsigned int)__float2int_rn(wxy * wz[c])
                                                             : __float_as_uint(__fmul_rn(wxy, wz[c]));
                                atomicAdd(plane[a] + b * T::YS + c, fx);
                            }
                        }
                }
            }
            __syncthreads();   // every particle of the chunk is in the tile

            // ---- tile -> mesh: one coalesced 128-byte RED per (x,y) column, zeros skipped; the tile is cleared on the way.
            float *mz = mesh + wrap_index32(bz * ZC - T::OFF + lane, G.N);
            const bool more = c1 < pend;
            if constexpr (T::PLANE_FLUSH) {
                // A warp takes whole x-planes of the tile and walks their y-rows with a running mesh pointer: one LDS --
                // the tile's own -- and a dozen instructions per column, all offsets immediate.  (Offsets from the
                // shared-memory tables below cost three more LDS per column on the pipe the TSC kernel runs out of:
                // 21.2 -> 20.7 ms for both meshes of config 3.  Equal column ranges per warp with running pointers: 21.3.)
                const int py0 = wrap_index32(by * BY - T::OFF, G.N);
                for (int u = warp; u < T::TX; u += TILE_THREADS / 32) {
                    int px = bx * BX - T::OFF + u;
                    bool ok = true;
                    if (G.slab) ok = px >= 0 && px < G.nplanes;
                    else px = wrap_index32(px, G.N);
                    unsigned int *t = tile + u * T::XS + lane;
                    float *row = mz + ((long long)px * G.N + py0) * G.ldz;
                    int py = py0;
#pragma unroll
                    for (int w = 0; w < T::TY; ++w) {
                        const unsigned int fx = t[w * T::YS];
                        if (more) t[w * T::YS] = 0u;
                        if (fx != 0u && ok) {
                            const float val = MASS ? (float)(int)fx * quantum : (float)fx * quantum;
                            atomicAdd(row, val);
                        }
                        row += G.ldz;
                        if (++py == G.N) { py = 0; row -= (long long)G.N * G.ldz; }
                    }
                }
            } else {
                // CIC (8 updates per particle, 13 - 14 planes for 8 warps): columns dealt to the warps one by one, offsets
                // from the tables (0.70 ms at 512^3 against 0.74 by planes)
                for (int col = warp; col < T::TX * T::TY; col += TILE_THREADS / 32) {
                    const int u = col / T::TY, w = col - u * T::TY;
                    const unsigned int fx = tile[u * T::XS + w * T::YS + lane];
                    if (more) tile[u * T::XS + w * T::YS + lane] = 0u;
                    const long long xo = xoff[u];
                    if (fx != 0u && xo >= 0) {
                        const float val = MASS ? (float)(int)fx * quantum : (float)fx * quantum;
                        atomicAdd(mz + xo + yoff[w], val);
                    }
                }
            }
            __syncthreads();
        }
        // this thread's (last) non-finite particle of the brick: NaN at its home cell, so that the mesh shows it.  A
        // plain store: NaN + anything is NaN, so the REDs of other bricks cannot undo it in either order.
        if (bad_home >= 0) {
            int px = bx * BX + (bad_home >> 16);
            const int py = wrap_index32(by * BY + ((bad_home >> 8) & 0xff), G.N), pz = wrap_index32(bz * ZC + (bad_home & 0xff), G.N);
            const bool ok = G.slab ? px < G.nplanes : true;
            if (!G.slab) px = wrap_index32(px, G.N);
            if (ok) mesh[((long long)px * G.N + py) * G.ldz + pz] = __int_as_float(0x7fc00000);
        }
    }
}

static size_t max_bricks(const apk_plan *P) {
    return (size_t)((P->N + 3 + BX - 1) / BX) * ((P->N + BY - 1) / BY) * ((P->N + 28) / 29);
}
static size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

// pair: the interlaced twins share one partition and one payload -- no extra room needed
size_t deposit_sorted_workspace_bytes(const apk_plan *P, long long np, int with_mass, int /*pair*/) {
    if (np <= 0) return 0;
    const size_t vs = with_mass ? sizeof(P4) : sizeof(P3);
    return align256(vs * (size_t)np) + 4 * align256(4 * (max_bricks(P) + 2)) +
           2 * align256(4 * (max_bricks(P) / SCAN_SEG + 2)) + 256;
}

// mesh1 != nullptr: interlaced pair -- G is the shift-0 geometry, mesh1 gets the shift-0.5 twin
template <int S, typename PT, bool SOA, bool MASS, bool PAIR>
static int run_sorted(apk_plan *P, const void *p0, const void *p1, const void *p2, const void *mass,
                      int mass_dtype, long long np, const DepositGeom &G, float *mesh, float *mesh1, cudaStream_t st) {
    using VT = typename std::conditional<MASS, P4, P3>::type;
    const BrickGrid B = make_brick_grid(G, S, PAIR);
    const size_t need = deposit_sorted_workspace_bytes(P, np, MASS, PAIR);
    // the cuFFT work areas live in the last fft_work_bytes of the same workspace and may be in use on another stream
    APK_REQUIRE(P->workspace && P->workspace_bytes >= need + P->fft_work_bytes + 256,
                "apk_deposit: sorted path needs %zu workspace bytes (+ %zu of cuFFT work area), %zu set "
                "(apk_plan_workspace_bytes / apk_plan_set_workspace)", need, P->fft_work_bytes + 256, P->workspace_bytes);
    APK_REQUIRE(np < 0xffffffffLL, "apk_deposit: more than 2^32-1 particles on one device");
    APK_REQUIRE((size_t)B.nbricks <= max_bricks(P), "apk_deposit: brick tables too small (internal)");
    unsigned char *w = (unsigned char *)P->workspace;
    VT *vals = (VT *)w; w += align256(sizeof(VT) * (size_t)np);
    const size_t tab = align256(4 * (max_bricks(P) + 2));
    unsigned int *counts = (unsigned int *)w; w += tab;
    unsigned int *brick_start = (unsigned int *)w; w += tab;
    unsigned int *cursor = (unsigned int *)w; w += tab;
    unsigned int *filled = (unsigned int *)w; w += tab;
    unsigned int *seg_total = (unsigned int *)w; w += align256(4 * (max_bricks(P) / SCAN_SEG + 2));
    unsigned int *seg_filled = (unsigned int *)w; w += align256(4 * (max_bricks(P) / SCAN_SEG + 2));
    unsigned int *counter = (unsigned int *)w;          // [1] number of non-empty bricks

    const long long tile = (long long)PART_THREADS * PART_ITEMS;
    const int pb = (int)std::min<long long>((np + tile - 1) / tile, (long long)P->num_sms * 8);
    P->mark(0, st);
    APK_CUDA(cudaMemsetAsync(counts, 0, 4 * (size_t)(B.nbricks + 1), st));
    brick_count_kernel<S, PT, SOA><<<pb, PART_THREADS, 0, st>>>((const PT *)p0, (const PT *)p1, (const PT *)p2, np, G, B, counts);
    APK_CUDA(cudaGetLastError());
    P->mark(1, st);
    const int nseg = (B.nbricks + SCAN_SEG - 1) / SCAN_SEG;
    brick_segsum_kernel<<<nseg, 1024, 0, st>>>(counts, B.nbricks, seg_total, seg_filled);
    APK_CUDA(cudaGetLastError());
    brick_scan_kernel<<<nseg, 1024, 0, st>>>(counts, B.nbricks, seg_total, seg_filled, brick_start, cursor, filled, counter + 1);
    APK_CUDA(cudaGetLastError());
    P->mark(2, st);
    brick_scatter_kernel<S, PT, SOA, MASS, VT><<<pb, PART_THREADS, 0, st>>>(
        (const PT *)p0, (const PT *)p1, (const PT *)p2, mass, mass_dtype == APK_F64, np, G, B, cursor, vals);
    APK_CUDA(cudaGetLastError());

    // one CTA per brick (CTAs beyond the number of non-empty bricks, which only the device knows, exit at once)
    const int ctas = B.nbricks;
    P->mark(3, st);
    brick_tile_kernel<S, MASS, PAIR, 0, VT><<<ctas, TILE_THREADS, 0, st>>>(vals, brick_start, filled, counter + 1, G, B, mesh);
    APK_CUDA(cudaGetLastError());
    if constexpr (PAIR) {
        if (P->first_mesh_event) APK_CUDA(cudaEventRecord(P->first_mesh_event, st));
        brick_tile_kernel<S, MASS, PAIR, 1, VT><<<ctas, TILE_THREADS, 0, st>>>(vals, brick_start, filled, counter + 1, G, B, mesh1);
        APK_CUDA(cudaGetLastError());
    }
    P->mark(4, st);
    if (P->timing) { P->dep_timed = true; P->dep_sorted = true; }
    return 0;
}

template <int S, typename PT, bool SOA>
static int dispatch_mass(apk_plan *P, const void *p0, const void *p1, const void *p2, const void *mass,
                         int mass_dtype, long long np, const DepositGeom &G, float *mesh, float *mesh1, cudaStream_t st) {
    if (mesh1)
        return mass ? run_sorted<S, PT, SOA, true, true>(P, p0, p1, p2, mass, mass_dtype, np, G, mesh, mesh1, st)
                    : run_sorted<S, PT, SOA, false, true>(P, p0, p1, p2, mass, mass_dtype, np, G, mesh, mesh1, st);
    return mass ? run_sorted<S, PT, SOA, true, false>(P, p0, p1, p2, mass, mass_dtype, np, G, mesh, nullptr, st)
                : run_sorted<S, PT, SOA, false, false>(P, p0, p1, p2, mass, mass_dtype, np, G, mesh, nullptr, st);
}

template <int S>
static int dispatch_layout(apk_plan *P, const void *p0, const void *p1, const void *p2, int layout, int pos_dtype,
                           const void *mass, int mass_dtype, long long np, const DepositGeom &G, float *mesh,
                           float *mesh1, cudaStream_t st) {
    if (pos_dtype == APK_F32)
        return layout == APK_SOA ? dispatch_mass<S, float, true>(P, p0, p1, p2, mass, mass_dtype, np, G, mesh, mesh1, st)
                                 : dispatch_mass<S, float, false>(P, p0, p1, p2, mass, mass_dtype, np, G, mesh, mesh1, st);
    return layout == APK_SOA ? dispatch_mass<S, double, true>(P, p0, p1, p2, mass, mass_dtype, np, G, mesh, mesh1, st)
                             : dispatch_mass<S, double, false>(P, p0, p1, p2, mass, mass_dtype, np, G, mesh, mesh1, st);
}

int deposit_atomic_launch(const void *, const void *, const void *, int, int, const void *, int, long long,
                          int, const DepositGeom &, float *, int, cudaStream_t);

// mesh1 != nullptr: also deposit the interlaced twin (shift + 0.5) from the same partition (CIC / TSC only)
int deposit_sorted_launch(apk_plan *P, const void *p0, const void *p1, const void *p2, int layout, int pos_dtype,
                          const void *mass, int mass_dtype, long long np, int resampler, const DepositGeom &G,
                          float *mesh, float *mesh1, cudaStream_t st) {
    if (np == 0) return 0;
    if (resampler == APK_CIC) return dispatch_layout<2>(P, p0, p1, p2, layout, pos_dtype, mass, mass_dtype, np, G, mesh, mesh1, st);
    if (resampler == APK_TSC) return dispatch_layout<3>(P, p0, p1, p2, layout, pos_dtype, mass, mass_dtype, np, G, mesh, mesh1, st);
    // NGP has no halo and no arithmetic worth tiling: one RED per particle
    return deposit_atomic_launch(p0, p1, p2, layout, pos_dtype, mass, mass_dtype, np, resampler, G, mesh, P->num_sms, st);
}

}  // namespace apk
