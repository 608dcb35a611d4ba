// Taylor-Fourier (TF) mesh of Colombi et al. (2009), POWMES' `norder`: a window-free delta(k) from NGP moment grids.
//
//   M_alpha[h] = sum_{p with home h} m_p dx^a dy^b dz^c     (h = nearest grid point, d = g - h in [-1/2, 1/2]^3,
//                                                            every alpha = (a, b, c) with |alpha| <= n)
//   c_TF(k)    = sum_alpha (-i)^|alpha| (wx^a wy^b wz^c / (a! b! c!)) r2c(M_alpha)(k),  w = 2 pi freq_index / N
//              = sum_h e^{-i w.h} sum_p m_p T_n(w.d_p),      T_n = degree-n Taylor polynomial of e^{-i theta}
//
// so |c_TF(k) - sum_p m_p e^{-i w.g_p}| <= sum_p |m_p| (|w|_1 / 2)^{n+1} / (n+1)!: no window, no aliasing beyond that.
// Multi-indices are in graded order (|alpha| = 0, 1, ..., then a, then b descending), so the moments of order n are a
// prefix of those of order n + 1.
//
// Pipeline (one stream, no host sync):
//   1. the sorted deposit's brick partition, S = 1 (deposit_sorted.cu, sorted_partition_ngp): bricks of 24 x 8 x 32
//      home cells, payload = brick-local coordinates (+ mass) in the plan workspace.  Once per field.
//   2. per pass of `group` moments (the caller's scratch holds `group` padded meshes):
//      tf_moment_tile_kernel  one CTA per non-empty brick, one thread per particle; up to TF_TILE_G = 8 moment tiles of
//                             the brick (24 KB each) in shared memory as 32-bit fixed-point integers, native ATOMS.ADD
//                             (the float32 shared-memory atomicAdd is a CAS loop on sm_100a), one RED per column to
//                             the moment meshes.  Order 3 (20 moments) takes three walks over the payload.
//      cuFFT r2c              each moment mesh in place, the plan's own r2c.
//      tf_combine_kernel      one pass over the half grid: the pass's transformed moments times the per-axis tables
//                             w^a / a!, rotated by (-i)^|alpha|, written (first pass) or added into the output mesh.
#include "brick_common.cuh"
#include <algorithm>
#include <cmath>
#include <vector>

namespace apk {

constexpr int TF_MAX_ORDER = 4, TF_MAX_MOM = 35;
constexpr int TF_TILE_G = 8;                          // moment tiles per CTA: 8 x 24 KB = 192 KB of shared memory
constexpr int TF_TILE_THREADS = 1024;                // 32 warps: the one CTA per SM (192 KB of tiles) hides the latency alone
constexpr int TF_FLUSH = 8191;                        // particles between two flushes (as the TSC / CIC tile kernel)
constexpr int TF_YS = BZ, TF_XS = BY * BZ;            // tile [BX][BY][32]: bank = z
constexpr int TF_CELLS = BX * BY * BZ;                // 6144 cells = 24 KB per moment
constexpr int TF_COMBINE_THREADS = 256;

__host__ __device__ constexpr int tf_nmom(int n) { return (n + 1) * (n + 2) * (n + 3) / 6; }

// exponent of axis `axis` in multi-index k (graded order)
__host__ __device__ constexpr int tf_exp(int k, int axis) {
    int i = 0;
    for (int t = 0; t <= TF_MAX_ORDER; ++t)
        for (int a = t; a >= 0; --a)
            for (int b = t - a; b >= 0; --b) {
                if (i == k) return axis == 0 ? a : (axis == 1 ? b : t - a - b);
                ++i;
            }
    return 0;
}

// nearest brick-local home cell of coordinate l on one axis (clamped to the brick) and d = l - home in [-1/2, 1/2]
// (a particle filed under the neighbouring brick at a rounding tie is clamped: |d| exceeds 1/2 by ~1e-5 at most)
__device__ __forceinline__ void tf_home(float l, float last, float &d, int &h) {
    const float M = 12582912.f;                       // 1.5 * 2^23: adding it rounds to the nearest integer
    float t = l + M;
    t = fminf(fmaxf(t, M), M + last);
    h = __float_as_int(t) & 0x3fffff;
    d = l - (t - M);
}

struct TfTileArgs {
    int N, ldz;
    BrickGrid B;
    int k0, G;                                        // moments k0 .. k0 + G - 1 (G <= TF_TILE_G)
    unsigned int degs;                                // |alpha| of moment k0 + j in bits 3 j .. 3 j + 2
    float *mesh;                                      // moment k0 + j -> mesh + j * mstride (padded meshes)
    long long mstride;
};

// Fixed point, per chunk of <= TF_FLUSH particles: unit = the power of two at or above the chunk's largest |mass|,
// s = the largest number of fractional bits with (sum |m| / unit) 2^s < 2^31 (float64 sum, padded by 0.1 %), and
// moment alpha is held in units of 2^-(s + |alpha|) unit: since |d^alpha| <= 2^-|alpha|, no cell can overflow.  The
// product m / unit * 2^s * (2 dx)^a (2 dy)^b (2 dz)^c (|2 d| <= 1) goes to the tile with one F2I + ATOMS.ADD.
template <int ORDER, bool MASS, typename VT>
__global__ void __launch_bounds__(TF_TILE_THREADS, 1)
tf_moment_tile_kernel(const VT *__restrict__ vals, const unsigned int *__restrict__ brick_start,
                      const unsigned int *__restrict__ filled, const unsigned int *__restrict__ nfilled_ptr, TfTileArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned int *tile = reinterpret_cast<unsigned int *>(smem_raw);          // [G][TF_CELLS]
    __shared__ float red_s[TF_TILE_THREADS / 32];
    __shared__ double red_sd[TF_TILE_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int k0 = A.k0, G = A.G, N = A.N;
    const BrickGrid B = A.B;
    const unsigned int nfilled = *nfilled_ptr;
    for (unsigned int slot = blockIdx.x; slot < nfilled; slot += gridDim.x) {
        const unsigned int brick = filled[slot];
        const unsigned int pbeg = brick_start[brick], pend = brick_start[brick + 1];
        const int bz = brick % B.nbz;
        const int by = (brick / B.nbz) % B.nby;
        const int bx = brick / (B.nbz * B.nby);
        __syncthreads();                              // (persistent grids) the previous brick's flush is complete
        for (int i = tid; i < G * TF_CELLS / 4; i += TF_TILE_THREADS) reinterpret_cast<uint4 *>(tile)[i] = make_uint4(0u, 0u, 0u, 0u);
        int bad_home = -1;                            // home cell of this thread's last non-finite particle (x << 16 | y << 8 | z)
        __syncthreads();

        for (unsigned int c0 = pbeg; c0 < pend; c0 += TF_FLUSH) {
            const unsigned int c1 = min(c0 + (unsigned int)TF_FLUSH, pend);
            float unit = 1.f, inv_unit = 1.f;
            double sum = (double)(c1 - c0);
            if constexpr (MASS) {
                // NaN / inf masses count as 0 here (the particle loop sends them to the mesh as NaN)
                float top = 0.f;
                sum = 0.0;
                for (unsigned int p = c0 + tid; p < c1; p += TF_TILE_THREADS) {
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
                for (int i = 1; i < TF_TILE_THREADS / 32; ++i) { top = fmaxf(top, red_s[i]); sum += red_sd[i]; }
                int e = ((__float_as_int(top) >> 23) & 0xff) + ((__float_as_int(top) & 0x7fffff) ? 1 : 0);
                e = min(max(e, 2), 252);
                unit = __int_as_float(e << 23);
                inv_unit = __int_as_float((254 - e) << 23);
                if (!(top > 0.f)) { unit = 1.f; inv_unit = 0.f; sum = 1.0; }   // all-zero masses: nothing to add
                sum *= (double)inv_unit;
            }
            const float room = 2147483648.f / (1.001f * fmaxf((float)sum, 1.f));
            const int frac_bits = min(((__float_as_int(room) >> 23) & 0xff) - 127, 30);
            const float mscale = __int_as_float((127 + frac_bits) << 23);

            unsigned int p = c0 + tid;
            VT nxt = {};
            if (p < c1) nxt = vals[p];
            for (; p < c1; p += TF_TILE_THREADS) {
                const VT v = nxt;
                const unsigned int q = p + TF_TILE_THREADS;
                if (q < c1) nxt = vals[q];
                float dx, dy, dz;
                int hx, hy, hz;
                tf_home(v.x, (float)(BX - 1), dx, hx);
                tf_home(v.y, (float)(BY - 1), dy, hy);
                tf_home(v.z, (float)(BZ - 1), dz, hz);
                float km = mscale;
                if constexpr (MASS) km = (v.m * inv_unit) * mscale;             // |m / unit| <= 1, exact; times 2^s
                // a NaN or inf coordinate or mass stays out of the integer tile (see brick_tile_kernel)
                const bool finite = fabsf(v.x) + fabsf(v.y) + fabsf(v.z) + fabsf(km) <= 3.4028235e38f;
                if (!finite) { bad_home = (hx << 16) | (hy << 8) | hz; continue; }
                float px[ORDER + 1], py[ORDER + 1], pz[ORDER + 1];
                px[0] = km; py[0] = 1.f; pz[0] = 1.f;
#pragma unroll
                for (int j = 1; j <= ORDER; ++j) {
                    px[j] = px[j - 1] * (2.f * dx); py[j] = py[j - 1] * (2.f * dy); pz[j] = pz[j - 1] * (2.f * dz);
                }
                unsigned int *cell = tile + hx * TF_XS + hy * TF_YS + hz;
                // the multi-indices in graded order (tf_exp), every exponent an immediate once the loops are unrolled
                int k = 0;
#pragma unroll
                for (int t = 0; t <= ORDER; ++t)
#pragma unroll
                    for (int a = t; a >= 0; --a)
#pragma unroll
                        for (int b = t - a; b >= 0; --b, ++k)
                            if (k >= k0 && k < k0 + G) {
                                const float val = (px[a] * py[b]) * pz[t - a - b];
                                atomicAdd(cell + (k - k0) * TF_CELLS, (unsigned int)__float2int_rn(val));
                            }
            }
            __syncthreads();   // every particle of the chunk is in the tiles

            // ---- tiles -> meshes: one coalesced 128-byte RED per (moment, x, y) column, zeros skipped; the tiles are
            //      cleared on the way if more chunks follow
            const bool more = c1 < pend;
            const int pz = wrap_index32(bz * BZ + lane, N);
            for (int col = warp; col < G * BX * BY; col += TF_TILE_THREADS / 32) {
                const int j = col / (BX * BY), u = (col / BY) % BX, w = col % BY;
                unsigned int *t = tile + j * TF_CELLS + u * TF_XS + w * TF_YS + lane;
                const unsigned int fx = *t;
                if (more) *t = 0u;
                if (fx != 0u) {
                    const int deg = (int)((A.degs >> (3 * j)) & 7u);
                    const float quantum = __int_as_float((127 - frac_bits - deg) << 23) * unit;
                    const int px = wrap_index32(bx * BX + u, N), py = wrap_index32(by * BY + w, N);
                    atomicAdd(A.mesh + j * A.mstride + ((long long)px * N + py) * A.ldz + pz, (float)(int)fx * quantum);
                }
            }
            __syncthreads();
        }
        // this thread's (last) non-finite particle of the brick: NaN at its home cell in every moment mesh of the pass
        if (bad_home >= 0) {
            const int px = wrap_index32(bx * BX + (bad_home >> 16), N), py = wrap_index32(by * BY + ((bad_home >> 8) & 0xff), N);
            const int pz = wrap_index32(bz * BZ + (bad_home & 0xff), N);
            for (int j = 0; j < G; ++j) A.mesh[j * A.mstride + ((long long)px * N + py) * A.ldz + pz] = __int_as_float(0x7fc00000);
        }
    }
}

struct TfCombineArgs {
    const float2 *mom;                                // transformed moment k0 + j at mom + j * mstride ([N][N][Nk])
    long long mstride;
    const float *tw;                                  // [TF_MAX_ORDER + 1][N]: w_i^a / a! (float64 on the host, then float32)
    int N, Nk, G, accumulate;
    int ea[TF_MAX_MOM], eb[TF_MAX_MOM], ec[TF_MAX_MOM];   // exponents of the pass's moment j
    float2 *out;                                      // [N][N][Nk], the caller's padded mesh
};

// (-i)^t v
__device__ __forceinline__ float2 tf_rot(float2 v, int t) {
    switch (t & 3) {
        case 0: return v;
        case 1: return make_float2(v.y, -v.x);
        case 2: return make_float2(-v.x, -v.y);
        default: return make_float2(-v.y, v.x);
    }
}

__global__ void __launch_bounds__(TF_COMBINE_THREADS)
tf_combine_kernel(TfCombineArgs A) {
    const long long total = (long long)A.N * A.N * A.Nk;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x; m < total; m += stride) {
        const int iz = (int)(m % A.Nk);
        const long long r = m / A.Nk;
        const int ib = (int)(r % A.N), ia = (int)(r / A.N);
        float re = 0.f, im = 0.f;
        for (int j = 0; j < A.G; ++j) {
            const int a = A.ea[j], b = A.eb[j], c = A.ec[j];
            const float cf = (A.tw[a * A.N + ia] * A.tw[b * A.N + ib]) * A.tw[c * A.N + iz];
            const float2 v = tf_rot(A.mom[j * A.mstride + m], a + b + c);
            re = fmaf(cf, v.x, re);
            im = fmaf(cf, v.y, im);
        }
        if (A.accumulate) { const float2 o = A.out[m]; re += o.x; im += o.y; }
        A.out[m] = make_float2(re, im);
    }
}

int sorted_partition_ngp(apk_plan *P, const void *p0, const void *p1, const void *p2, int layout, int pos_dtype,
                         const void *mass, int mass_dtype, long long np, const DepositGeom &G, BrickPartition &out,
                         cudaStream_t st);

}  // namespace apk

using namespace apk;

struct apk_tf {
    apk_plan *plan = nullptr;
    int order = 0, nmom = 1;
    float *tw = nullptr;                              // device [TF_MAX_ORDER + 1][N]
    std::vector<cudaEvent_t> ev;                      // partition | per pass: tiles, r2c, combine
    int npass = 0;
    bool timed = false;
};

namespace {

size_t tf_mesh_bytes(const apk_plan *P) { return sizeof(float) * (size_t)P->N * P->N * P->ldz; }

bool tf_overlaps(const void *a, size_t na, const void *b, size_t nb) {
    if (!a || !b) return false;
    const char *x = (const char *)a, *y = (const char *)b;
    return x < y + nb && y < x + na;
}

template <int ORDER>
int tf_tiles(const BrickPartition &part, bool mass, const TfTileArgs &A, cudaStream_t st) {
    const size_t smem = sizeof(unsigned int) * (size_t)A.G * TF_CELLS;
    auto go = [&](auto kern, const auto *vals) -> int {
        APK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(unsigned int) * TF_TILE_G * TF_CELLS)));
        // one CTA per brick (CTAs beyond the number of non-empty bricks exit at once)
        kern<<<part.B.nbricks, TF_TILE_THREADS, smem, st>>>(vals, part.brick_start, part.filled, part.nfilled, A);
        APK_CUDA(cudaGetLastError());
        return 0;
    };
    if (mass) return go(tf_moment_tile_kernel<ORDER, true, P4>, (const P4 *)part.vals);
    return go(tf_moment_tile_kernel<ORDER, false, P3>, (const P3 *)part.vals);
}

int tf_tiles_dispatch(int order, const BrickPartition &part, bool mass, const TfTileArgs &A, cudaStream_t st) {
    switch (order) {
        case 0: return tf_tiles<0>(part, mass, A, st);
        case 1: return tf_tiles<1>(part, mass, A, st);
        case 2: return tf_tiles<2>(part, mass, A, st);
        case 3: return tf_tiles<3>(part, mass, A, st);
        default: return tf_tiles<4>(part, mass, A, st);
    }
}

}  // namespace

extern "C" {

int apk_tf_create(apk_tf **out, apk_plan *P, int order) {
    APK_REQUIRE(out && P, "apk_tf_create: null argument");
    APK_REQUIRE(P->n0 == P->N, "apk_tf_create: single-GPU plans only (slab plans have no Taylor-Fourier path)");
    APK_REQUIRE(order >= 0 && order <= TF_MAX_ORDER, "apk_tf_create: order must be 0 .. %d, got %d", TF_MAX_ORDER, order);
    DeviceGuard guard(P->device);
    const int N = P->N;
    // w_i^a / a! per axis in float64 (w = 2 pi freq_index(i) / N, -N/2 for the Nyquist index of even N), then float32
    std::vector<float> host((size_t)(TF_MAX_ORDER + 1) * N);
    for (int i = 0; i < N; ++i) {
        const int n = 2 * i < N ? i : i - N;
        const double w = (double)n * (2.0 * M_PI / (double)N);
        double v = 1.0;
        for (int a = 0; a <= TF_MAX_ORDER; ++a) {
            host[(size_t)a * N + i] = (float)v;
            v = v * w / (double)(a + 1);
        }
    }
    apk_tf *T = new apk_tf();
    T->plan = P; T->order = order; T->nmom = tf_nmom(order);
    if (cudaMalloc(&T->tw, sizeof(float) * host.size()) != cudaSuccess) {
        delete T; set_error("apk_tf_create: cudaMalloc of the coefficient tables failed"); return 1;
    }
    if (cudaMemcpy(T->tw, host.data(), sizeof(float) * host.size(), cudaMemcpyHostToDevice) != cudaSuccess) {
        apk_tf_destroy(T); set_error("apk_tf_create: table upload failed"); return 1;
    }
    *out = T;
    return 0;
}

int apk_tf_destroy(apk_tf *T) {
    if (!T) return 0;
    DeviceGuard guard(T->plan->device);
    if (T->tw) cudaFree(T->tw);
    for (auto &e : T->ev) cudaEventDestroy(e);
    delete T;
    return 0;
}

int apk_tf_scratch_bytes(const apk_tf *T, int group, size_t *bytes) {
    APK_REQUIRE(T && bytes, "apk_tf_scratch_bytes: null argument");
    APK_REQUIRE(group >= 1 && group <= T->nmom, "apk_tf_scratch_bytes: group must be 1 .. %d moments, got %d", T->nmom, group);
    *bytes = (size_t)group * tf_mesh_bytes(T->plan);
    return 0;
}

int apk_tf_field(apk_tf *T, const void *p0, const void *p1, const void *p2, int layout, int pos_dtype, double pos_scale,
                 const void *mass, int mass_dtype, int64_t np, int group, void *scratch, size_t bytes, float *out_mesh,
                 void *stream) {
    APK_REQUIRE(T && out_mesh, "apk_tf_field: null tf object or output mesh");
    APK_REQUIRE(np >= 0, "apk_tf_field: negative particle count");
    APK_REQUIRE(np == 0 || p0, "apk_tf_field: null positions");
    APK_REQUIRE(layout == APK_AOS || layout == APK_SOA, "apk_tf_field: bad layout %d", layout);
    APK_REQUIRE(layout == APK_AOS || (p1 && p2) || np == 0, "apk_tf_field: SoA layout needs three pointers");
    APK_REQUIRE(pos_dtype == APK_F32 || pos_dtype == APK_F64, "apk_tf_field: bad position dtype %d", pos_dtype);
    APK_REQUIRE(!mass || mass_dtype == APK_F32 || mass_dtype == APK_F64, "apk_tf_field: bad mass dtype %d", mass_dtype);
    APK_REQUIRE(std::isfinite(pos_scale) && pos_scale != 0.0, "apk_tf_field: pos_scale must be finite and non-zero");
    APK_REQUIRE(np < 0xffffffffLL, "apk_tf_field: more than 2^32-1 particles on one device");
    APK_REQUIRE(group >= 1 && group <= T->nmom, "apk_tf_field: group must be 1 .. %d moments, got %d", T->nmom, group);
    apk_plan *P = T->plan;
    const size_t mb = tf_mesh_bytes(P), need = (size_t)group * mb;
    APK_REQUIRE(scratch && bytes >= need, "apk_tf_field: scratch of %zu bytes needed for %d moment meshes, %zu given "
                "(apk_tf_scratch_bytes)", need, group, scratch ? bytes : (size_t)0);
    APK_REQUIRE(!tf_overlaps(scratch, need, out_mesh, mb), "apk_tf_field: the output mesh overlaps the scratch");
    DeviceGuard guard(P->device);
    cudaStream_t st = (cudaStream_t)stream;
    const int npass = (T->nmom + group - 1) / group;
    const bool timing = P->timing;
    if (timing) {
        while (T->ev.size() < (size_t)(2 + 3 * npass)) {
            cudaEvent_t e;
            APK_CUDA(cudaEventCreate(&e));
            T->ev.push_back(e);
        }
        APK_CUDA(cudaEventRecord(T->ev[0], st));
    }
    T->timed = false;

    DepositGeom G;
    G.N = P->N; G.ldz = P->ldz; G.scale = pos_scale * (double)P->N; G.shift = 0.0;
    G.slab = 0; G.plane0 = 0; G.nplanes = P->N; G.own0 = 0; G.nown = P->N;
    G.s0 = (float)G.scale;
    G.s1 = (float)(G.scale - (double)G.s0);
    G.s2 = (float)(G.scale - (double)G.s0 - (double)G.s1);
    G.t32 = (fabs(G.scale) < 1e30 && fabs(G.scale) > 1e-30) ? 0.5f : -1.f;        // NGP rounding, as apk_deposit
    BrickPartition part{};
    if (np > 0)
        if (int rc = sorted_partition_ngp(P, p0, p1, p2, layout, pos_dtype, mass, mass_dtype, np, G, part, st)) return rc;
    if (timing) APK_CUDA(cudaEventRecord(T->ev[1], st));

    for (int pass = 0, k0 = 0; k0 < T->nmom; ++pass, k0 += group) {
        const int g = std::min(group, T->nmom - k0);
        float *meshes = (float *)scratch;
        const long long mstride = (long long)P->N * P->N * P->ldz;
        APK_CUDA(cudaMemsetAsync(meshes, 0, (size_t)g * mb, st));
        for (int sub = 0; np > 0 && sub < g; sub += TF_TILE_G) {
            TfTileArgs A;
            A.N = P->N; A.ldz = P->ldz; A.B = part.B;
            A.k0 = k0 + sub; A.G = std::min(TF_TILE_G, g - sub);
            A.degs = 0u;
            for (int j = 0; j < A.G; ++j)
                A.degs |= (unsigned int)(tf_exp(A.k0 + j, 0) + tf_exp(A.k0 + j, 1) + tf_exp(A.k0 + j, 2)) << (3 * j);
            A.mesh = meshes + sub * mstride; A.mstride = mstride;
            if (int rc = tf_tiles_dispatch(T->order, part, mass != nullptr, A, st)) return rc;
        }
        if (timing) APK_CUDA(cudaEventRecord(T->ev[2 + 3 * pass], st));
        for (int j = 0; j < g; ++j)
            if (int rc = apk_fft_r2c(P, meshes + j * mstride, stream)) return rc;
        if (timing) APK_CUDA(cudaEventRecord(T->ev[3 + 3 * pass], st));
        TfCombineArgs C;
        C.mom = (const float2 *)meshes; C.mstride = mstride / 2; C.tw = T->tw;
        C.N = P->N; C.Nk = P->Nk; C.G = g; C.accumulate = pass > 0;
        for (int j = 0; j < g; ++j) { C.ea[j] = tf_exp(k0 + j, 0); C.eb[j] = tf_exp(k0 + j, 1); C.ec[j] = tf_exp(k0 + j, 2); }
        C.out = (float2 *)out_mesh;
        const long long modes = (long long)P->N * P->N * P->Nk;
        const int blocks = (int)std::min<long long>((modes + TF_COMBINE_THREADS - 1) / TF_COMBINE_THREADS, (long long)P->num_sms * 16);
        tf_combine_kernel<<<blocks, TF_COMBINE_THREADS, 0, st>>>(C);
        APK_CUDA(cudaGetLastError());
        if (timing) APK_CUDA(cudaEventRecord(T->ev[4 + 3 * pass], st));
    }
    T->npass = npass;
    T->timed = timing;
    return 0;
}

int apk_tf_last_ms(apk_tf *T, float ms[4]) {
    APK_REQUIRE(T && ms, "apk_tf_last_ms: null argument");
    APK_REQUIRE(T->timed, "apk_tf_last_ms: no timed apk_tf_field on this object (apk_plan_enable_timing)");
    DeviceGuard guard(T->plan->device);
    APK_CUDA(cudaEventSynchronize(T->ev[1 + 3 * T->npass]));
    APK_CUDA(cudaEventElapsedTime(&ms[0], T->ev[0], T->ev[1]));
    ms[1] = ms[2] = ms[3] = 0.f;
    for (int pass = 0; pass < T->npass; ++pass)
        for (int s = 0; s < 3; ++s) {
            float t = 0.f;
            APK_CUDA(cudaEventElapsedTime(&t, T->ev[1 + 3 * pass + s], T->ev[2 + 3 * pass + s]));
            ms[1 + s] += t;
        }
    return 0;
}

}  // extern "C"
