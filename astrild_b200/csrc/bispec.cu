// Bispectrum B(k1, k2, k3) of one field by the FFT (shell-field) estimator, with exact triangle counts.
//
//   F_b(x) = sum_{q in shell b} c(q) e^{i q.x}          (un-normalised c2r of the k-grid masked to shell b)
//   T_F(i,j,l) = sum_x F_i F_j F_l,   T_D(i,j,l) = the same with c == 1 = N^3 N_tri
//   B = (L^6 s^3 / N^9) T_F / T_D                        (V^2 <delta delta delta> in pmesh's normalisation)
//
// Shells are those of the 1-D binning (bin_power.cu / bin_kmu.cu): k^2 = (ka^2 + kb^2) + kz^2 in float64 from the
// host-built tables, numpy.digitize(k^2, kedges^2) by a float guess fixed with float64 compares; the k = 0 mode is in no
// shell.  Triples i <= j <= l are skipped only when they provably hold no triangle: lo_l >= hi_i + hi_j (no closure)
// and hi_i + hi_j + hi_l <= 2 k_Nyquist (no closure modulo the grid).  kmax is at most k_Nyquist, so no shell holds a
// Nyquist-index mode and every masked k-grid is exactly Hermitian.
//
// Kernels
//   bk_fill_kernel     one pass over the half-complex grid: interlace-combine and window deconvolution as in
//                      bin_power.cu (compensation tables hold 1 / comp), one write of each mode into its shell's
//                      field (pre-zeroed); indicator variant (c == 1) in float64 for the counts.
//   cuFFT              C2R (spectrum) / Z2D (counts), in place in the padded mesh layout, batched over shells.
//   bk_reduce_kernel   C_i[j][l] = sum_x (F_i F_j)(x) F_l(x): a CTA stages a chunk of BK_P points of all shells in
//                      shared memory ([point][shell], padding floats of the rows skipped) with cp.async, double
//                      buffered; each thread owns one tile = (i, TJ consecutive j, TD consecutive d = l - j) and keeps
//                      its TJ x TD sums in registers: per point one LDS for F_i, TJ/4 LDS.128 for F_j, (TJ + TD)/4
//                      LDS.128 for the l-run, TJ FMUL and TJ TD FFMA.  The tiles follow the band l <= i + j + 1 of
//                      the kept triples; tiles whose triples are all skipped are not computed.
//                      float: sums over at most BK_SEG_POINTS points per thread in float32, then added to the CTA's
//                      float64 slot; double: float64 throughout.
//   bk_fold_kernel     per kept triple: the CTAs' float64 slots in a fixed order (deterministic).
#include "apk_common.cuh"
#include <algorithm>
#include <cmath>
#include <utility>
#include <vector>

namespace apk {

constexpr int BK_MAX_BINS = 128;           // shells; also bounds the shared-memory row (128 + 12 floats)
constexpr int BK_P = 64;                   // points per staged chunk
constexpr int BK_SEG_CHUNKS = 16;          // float32 partial sums span at most BK_SEG_CHUNKS * BK_P points ...
constexpr int BK_SEG_POINTS = BK_SEG_CHUNKS * BK_P;   // ... = 1024, then go to float64
static_assert(BK_SEG_POINTS == 1024, "the float32 error model of the tests assumes 1024-point partial sums");
constexpr int BK_MAX_THREADS = 512;        // tiles per CTA (one per thread)
constexpr int BK_FILL_THREADS = 256;

// register tile (j-run x d-run) of the two instantiations
template <typename T> struct BkTile;
template <> struct BkTile<float> { static constexpr int TJ = 8, TD = 4; };
template <> struct BkTile<double> { static constexpr int TJ = 4, TD = 4; };

struct BkFillArgs {
    const float2 *c1, *c1s;
    const double *ka2, *kb2, *kz2, *edges2;
    const float *ic_a, *ic_b, *ic_z;           // 1 / comp (NULL: no compensation)
    const float2 *ph_a, *ph_b, *ph_z;          // exp(i phase) (NULL: not interlaced)
    int N, Nk, nedges;
    long long field_cplx;                      // complex elements per field (N * N * Nk)
    float kmin_f, inv_dk_f;
    void *fields;                              // float2 or double2 [nbins][N][N][Nk]
};

__device__ __forceinline__ float2 bk_cmul(float2 a, float2 b) {
    return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}

// IND: indicator fields (c == 1) as double2; otherwise the field as float2
template <bool IND, bool INTERLACED, bool COMP>
__global__ void __launch_bounds__(BK_FILL_THREADS)
bk_fill_kernel(BkFillArgs A) {
    const long long total = (long long)A.N * A.N * A.Nk;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const int nedges = A.nedges;
    const double e2_first = A.edges2[0], e2_last = A.edges2[nedges - 1];
    for (long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x; m < total; m += stride) {
        const int iz = (int)(m % A.Nk);
        const long long r = m / A.Nk;
        const int ib = (int)(r % A.N), ia = (int)(r / A.N);
        if (ia == 0 && ib == 0 && iz == 0) continue;                 // k = 0: in no shell
        const double k2 = __dadd_rn(__dadd_rn(A.ka2[ia], A.kb2[ib]), A.kz2[iz]);
        if (k2 >= e2_last || k2 < e2_first) continue;                // outside the edges
        // numpy.digitize(k2, kedges^2): float guess, fixed by float64 compares (bin_kmu.cu)
        const double knorm = sqrt(k2);
        int bin = (int)(((float)knorm - A.kmin_f) * A.inv_dk_f) + 1;
        bin = max(1, min(bin, nedges - 1));
        while (k2 < A.edges2[bin - 1]) --bin;
        while (k2 >= A.edges2[bin]) ++bin;
        const size_t dst = (size_t)(bin - 1) * A.field_cplx + (size_t)m;
        if (IND) {
            reinterpret_cast<double2 *>(A.fields)[dst] = make_double2(1.0, 0.0);
        } else {
            float2 a = __ldcs(A.c1 + m);
            if (INTERLACED) {
                const float2 ph = bk_cmul(bk_cmul(A.ph_a[ia], A.ph_z[iz]), A.ph_b[ib]);
                const float2 s = bk_cmul(__ldcs(A.c1s + m), ph);
                a = make_float2(0.5f * (a.x + s.x), 0.5f * (a.y + s.y));
            }
            if (COMP) {
                const float ic = (A.ic_a[ia] * A.ic_z[iz]) * A.ic_b[ib];
                a.x *= ic; a.y *= ic;
            }
            reinterpret_cast<float2 *>(A.fields)[dst] = a;
        }
    }
}

struct BkReduceArgs {
    const void *fields;             // T [nbins][N][N][ldz] (real, after the c2r)
    long long field_elems;          // N * N * ldz
    int N, ldz, nbins;
    int row;                        // shared-memory row length (elements, multiple of 4): >= nbins + TJ + TD
    long long npoints;              // N^3
    long long nchunks;              // ceil(npoints / BK_P)
    const int4 *tiles;              // (i, j0, d0, -) per tile
    int ntiles;                     // tiles of this launch (all tile groups)
    double *slots;                  // [gridDim.x][ntiles][TJ * TD] float64
};

__device__ __forceinline__ void bk_cp_async(void *smem, const void *gmem, int bytes) {
#ifdef APK_SIMT
    memcpy(smem, gmem, bytes);
#else
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    if (bytes == 4) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gmem) : "memory");
    else asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem) : "memory");
#endif
}
__device__ __forceinline__ void bk_cp_commit() {
#ifndef APK_SIMT
    asm volatile("cp.async.commit_group;" ::: "memory");
#endif
}
template <int PENDING>
__device__ __forceinline__ void bk_cp_wait() {
#ifndef APK_SIMT
    asm volatile("cp.async.wait_group %0;" ::"n"(PENDING) : "memory");
#endif
}

// vector of 4 elements from shared memory (LDS.128 for float, 2 x LDS.128 for double)
template <typename T> struct BkVec4;
template <> struct BkVec4<float> {
    static __device__ __forceinline__ void load(const float *p, float *v) {
        const float4 q = *reinterpret_cast<const float4 *>(p);
        v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    }
};
template <> struct BkVec4<double> {
    static __device__ __forceinline__ void load(const double *p, double *v) {
        const double2 a = reinterpret_cast<const double2 *>(p)[0], b = reinterpret_cast<const double2 *>(p)[1];
        v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
    }
};

// stage chunk `c` (BK_P points of all shells) into buffer `buf` ([BK_P][row]); points past the end are zero
template <typename T>
__device__ __forceinline__ void bk_stage(const BkReduceArgs &A, T *buf, long long c) {
    const int nthr = blockDim.x;
    const long long p0 = c * BK_P;
    for (int e = threadIdx.x; e < BK_P * A.nbins; e += nthr) {
        const int b = e / BK_P, p = e - b * BK_P;             // consecutive threads: consecutive points of one shell
        const long long pt = p0 + p;
        T *dst = buf + p * A.row + b;
        if (pt < A.npoints) {
            const long long rr = pt / A.N;                         // mesh row (x, y); the two padding floats are skipped
            const int z = (int)(pt - rr * A.N);
            const T *src = reinterpret_cast<const T *>(A.fields) + (size_t)b * A.field_elems + (size_t)rr * A.ldz + z;
            bk_cp_async(dst, src, (int)sizeof(T));
        } else {
            *dst = T(0);
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(BK_MAX_THREADS, 1)
bk_reduce_kernel(BkReduceArgs A) {
    constexpr int TJ = BkTile<T>::TJ, TD = BkTile<T>::TD, NL = TJ + TD;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *buf0 = reinterpret_cast<T *>(smem_raw);
    T *buf1 = buf0 + BK_P * A.row;

    // zero both buffers once: the columns nbins .. row-1 stay zero (they feed j, l >= nbins, which are discarded)
    for (int e = threadIdx.x; e < 2 * BK_P * A.row; e += blockDim.x) buf0[e] = T(0);
    __syncthreads();

    const int tile_id = blockIdx.y * BK_MAX_THREADS + threadIdx.x;
    const bool active = threadIdx.x < BK_MAX_THREADS && tile_id < A.ntiles;
    int4 tile = make_int4(0, 0, 0, 0);
    if (active) tile = A.tiles[tile_id];
    const int ti = tile.x, j0 = tile.y, l0 = tile.y + tile.z;

    const long long c_begin = A.nchunks * blockIdx.x / gridDim.x, c_end = A.nchunks * (blockIdx.x + 1) / gridDim.x;
    double *slot = A.slots + ((size_t)blockIdx.x * A.ntiles + (active ? tile_id : 0)) * (TJ * TD);
    T acc[TJ][TD];
#pragma unroll
    for (int a = 0; a < TJ; ++a)
#pragma unroll
        for (int d = 0; d < TD; ++d) acc[a][d] = T(0);
    bool first_flush = true;

    if (c_begin < c_end) bk_stage<T>(A, buf0, c_begin);
    bk_cp_commit();
    int seg = 0;
    for (long long c = c_begin; c < c_end; ++c) {
        T *cur = ((c - c_begin) & 1) ? buf1 : buf0;
        T *nxt = ((c - c_begin) & 1) ? buf0 : buf1;
        if (c + 1 < c_end) bk_stage<T>(A, nxt, c + 1);      // nxt was last read before the barrier that ended c - 1
        bk_cp_commit();
        bk_cp_wait<1>();                                      // chunk c has landed (for this thread's copies) ...
        __syncthreads();                                      // ... and for everybody's
        if (active) {
            const T *rowp = cur;
#pragma unroll 2
            for (int p = 0; p < BK_P; ++p, rowp += A.row) {
                const T fi = rowp[ti];
                T fj[TJ], fl[NL];
#pragma unroll
                for (int a = 0; a < TJ; a += 4) BkVec4<T>::load(rowp + j0 + a, fj + a);
#pragma unroll
                for (int a = 0; a < NL; a += 4) BkVec4<T>::load(rowp + l0 + a, fl + a);
#pragma unroll
                for (int a = 0; a < TJ; ++a) {
                    const T g = fi * fj[a];
#pragma unroll
                    for (int d = 0; d < TD; ++d) acc[a][d] = fma(g, fl[a + d], acc[a][d]);
                }
            }
        }
        __syncthreads();                                      // cur may be overwritten from the next iteration on
        if (++seg == BK_SEG_CHUNKS || c + 1 == c_end) {
            seg = 0;
            if (active) {                                     // float32 partials of <= BK_SEG_POINTS points -> float64
#pragma unroll
                for (int a = 0; a < TJ; ++a)
#pragma unroll
                    for (int d = 0; d < TD; ++d) {
                        const double prev = first_flush ? 0.0 : slot[a * TD + d];
                        slot[a * TD + d] = prev + (double)acc[a][d];
                        acc[a][d] = T(0);
                    }
            }
            first_flush = false;
        }
    }
    if (active && first_flush)                                // a CTA without points still owns its slot
        for (int e = 0; e < TJ * TD; ++e) slot[e] = 0.0;
}

// one thread per kept triple: sum of the CTAs' slots, fixed order
__global__ void __launch_bounds__(256)
bk_fold_kernel(const double *slots, const int *slot_of, int ntriples, int ctas, long long slot_stride, double *out) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= ntriples) return;
    const int s = slot_of[t];
    double acc = 0.0;
    for (int c = 0; c < ctas; ++c) acc += slots[(size_t)c * slot_stride + s];
    out[t] = acc;
}

}  // namespace apk

using namespace apk;

struct BkTiling {
    int ntiles = 0;
    int4 *tiles = nullptr;          // device
    int *slot_of = nullptr;         // device, per kept triple
    int groups = 0, threads = 0, ctas = 0;
    double *slots = nullptr;        // device [ctas][ntiles][TJ * TD]
};

struct apk_bispec {
    apk_plan *plan = nullptr;
    int nedges = 0, nbins = 0;
    bool interlaced = false, has_comp = false;
    std::vector<double> edges;
    std::vector<int> triples;       // [ntriples][3]
    int ntriples = 0;
    void *tables = nullptr;
    double *ka2 = nullptr, *kb2 = nullptr, *kz2 = nullptr, *edges2 = nullptr;
    float *ic_a = nullptr, *ic_b = nullptr, *ic_z = nullptr;
    float2 *ph_a = nullptr, *ph_b = nullptr, *ph_z = nullptr;
    cufftHandle fft_f = 0, fft_d = 0;
    bool has_fft_f = false, has_fft_d = false;
    int batch = 1;                  // shells per cuFFT execution
    size_t ws_f = 0, ws_d = 0;
    BkTiling tf, td;                // float (spectrum) and double (counts) tilings
    bool counted = false;
    std::vector<int64_t> ntri;
    double residual = 0.0;
    cudaEvent_t ev[5] = {};
    bool ev_ready = false, timed = false;
};

namespace {

size_t bk_fields_bytes(const apk_bispec *K) {
    const apk_plan *P = K->plan;
    return sizeof(double) * (size_t)K->nbins * P->N * P->N * P->ldz;      // the float64 indicator fields (the larger)
}

size_t bk_row(int nbins, int TJ, int TD) { return (size_t)((nbins + TJ + TD + 3) & ~3); }

template <typename T>
int bk_make_tiling(apk_bispec *K, BkTiling &Tg) {
    constexpr int TJ = BkTile<T>::TJ, TD = BkTile<T>::TD;
    const int nb = K->nbins;
    // slot of each kept triple inside its tile; tiles with no kept triple are never made
    std::vector<int> index((size_t)nb * nb * nb, -1);
    for (int t = 0; t < K->ntriples; ++t) {
        const int *q = &K->triples[3 * (size_t)t];
        index[((size_t)q[0] * nb + q[1]) * nb + q[2]] = t;
    }
    std::vector<int4> tiles;
    std::vector<int> slot_of(K->ntriples, -1);
    for (int i = 0; i < nb; ++i)
        for (int j0 = (i / TJ) * TJ; j0 < nb; j0 += TJ)
            for (int d0 = 0; j0 + d0 < nb; d0 += TD) {
                std::vector<std::pair<int, int>> hits;
                for (int a = 0; a < TJ; ++a)
                    for (int d = 0; d < TD; ++d) {
                        const int j = j0 + a, l = j0 + a + d0 + d;
                        if (j < i || j >= nb || l >= nb) continue;
                        const int t = index[((size_t)i * nb + j) * nb + l];
                        if (t >= 0) hits.push_back({t, a * TD + d});
                    }
                if (hits.empty()) continue;
                for (auto &h : hits) slot_of[h.first] = (int)tiles.size() * (TJ * TD) + h.second;
                tiles.push_back(make_int4(i, j0, d0, 0));
            }
    for (int s : slot_of) APK_REQUIRE(s >= 0, "apk_bispec_create: internal error (a kept triple has no tile)");
    Tg.ntiles = (int)tiles.size();
    Tg.groups = (Tg.ntiles + BK_MAX_THREADS - 1) / BK_MAX_THREADS;
    const int per = (Tg.ntiles + Tg.groups - 1) / Tg.groups;
    Tg.threads = std::min(BK_MAX_THREADS, ((per + 31) / 32) * 32);
    // the tiles of group g are g * BK_MAX_THREADS + [0, threads): re-pack so that each group holds `per` tiles
    std::vector<int4> packed((size_t)Tg.groups * BK_MAX_THREADS, make_int4(0, 0, 0, 0));
    std::vector<int> where(tiles.size());
    for (size_t t = 0; t < tiles.size(); ++t) {
        const int g = (int)(t / per), k = (int)(t % per);
        packed[(size_t)g * BK_MAX_THREADS + k] = tiles[t];
        where[t] = g * BK_MAX_THREADS + k;
    }
    Tg.ntiles = Tg.groups * BK_MAX_THREADS;                       // tile ids of the launch (holes are inactive)
    std::vector<char> used(Tg.ntiles, 0);
    for (size_t t = 0; t < tiles.size(); ++t) used[where[t]] = 1;
    for (int &s : slot_of) s = where[s / (TJ * TD)] * (TJ * TD) + s % (TJ * TD);
    // holes: mark inactive by giving them the id range past the real ones -> the kernel tests tile_id < ntiles only,
    // so holes compute a harmless (0, 0, 0) tile whose slots nobody reads
    (void)used;
    // resident CTAs: one wave of persistent CTAs over the chunks, per tile group
    const size_t smem = 2 * BK_P * bk_row(nb, TJ, TD) * sizeof(T);
    APK_CUDA(cudaFuncSetAttribute(bk_reduce_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    APK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bk_reduce_kernel<T>, Tg.threads, smem));
    if (per_sm < 1) per_sm = 1;
    Tg.ctas = std::max(1, (K->plan->num_sms * per_sm + Tg.groups - 1) / Tg.groups);
    const long long nchunks = ((long long)K->plan->N * K->plan->N * K->plan->N + BK_P - 1) / BK_P;
    if (Tg.ctas > nchunks) Tg.ctas = (int)nchunks;
    APK_CUDA(cudaMalloc(&Tg.tiles, sizeof(int4) * packed.size()));
    APK_CUDA(cudaMemcpy(Tg.tiles, packed.data(), sizeof(int4) * packed.size(), cudaMemcpyHostToDevice));
    APK_CUDA(cudaMalloc(&Tg.slot_of, sizeof(int) * std::max<size_t>(1, slot_of.size())));
    if (!slot_of.empty())
        APK_CUDA(cudaMemcpy(Tg.slot_of, slot_of.data(), sizeof(int) * slot_of.size(), cudaMemcpyHostToDevice));
    APK_CUDA(cudaMalloc(&Tg.slots, sizeof(double) * (size_t)Tg.ctas * Tg.ntiles * (TJ * TD)));
    return 0;
}

void bk_free_tiling(BkTiling &Tg) {
    if (Tg.tiles) cudaFree(Tg.tiles);
    if (Tg.slot_of) cudaFree(Tg.slot_of);
    if (Tg.slots) cudaFree(Tg.slots);
    Tg = BkTiling();
}

int bk_make_fft(apk_bispec *K, bool dbl) {
    apk_plan *P = K->plan;
    cufftHandle &h = dbl ? K->fft_d : K->fft_f;
    APK_CUFFT(cufftCreate(&h));
    (dbl ? K->has_fft_d : K->has_fft_f) = true;
    APK_CUFFT(cufftSetAutoAllocation(h, 0));
    long long n[3] = {P->N, P->N, P->N};
    long long inembed[3] = {P->N, P->N, P->Nk}, onembed[3] = {P->N, P->N, P->ldz};
    const long long idist = (long long)P->N * P->N * P->Nk, odist = (long long)P->N * P->N * P->ldz;
    size_t ws = 0;
    APK_CUFFT(cufftMakePlanMany64(h, 3, n, inembed, 1, idist, onembed, 1, odist, dbl ? CUFFT_Z2D : CUFFT_C2R, K->batch, &ws));
    (dbl ? K->ws_d : K->ws_f) = (ws + 255) & ~(size_t)255;
    return 0;
}

template <typename T>
int bk_reduce(apk_bispec *K, BkTiling &Tg, const void *fields, double *out, cudaStream_t st, bool timing) {
    constexpr int TJ = BkTile<T>::TJ, TD = BkTile<T>::TD;
    apk_plan *P = K->plan;
    BkReduceArgs A;
    A.fields = fields;
    A.field_elems = (long long)P->N * P->N * P->ldz;
    A.N = P->N; A.ldz = P->ldz; A.nbins = K->nbins;
    A.row = (int)bk_row(K->nbins, TJ, TD);
    A.npoints = (long long)P->N * P->N * P->N;
    A.nchunks = (A.npoints + BK_P - 1) / BK_P;
    A.tiles = Tg.tiles; A.ntiles = Tg.ntiles; A.slots = Tg.slots;
    const size_t smem = 2 * BK_P * (size_t)A.row * sizeof(T);
    // the attribute belongs to the kernel, not to this object: another object may have set a smaller one since
    APK_CUDA(cudaFuncSetAttribute(bk_reduce_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    bk_reduce_kernel<T><<<dim3(Tg.ctas, Tg.groups), Tg.threads, smem, st>>>(A);
    APK_CUDA(cudaGetLastError());
    if (timing) APK_CUDA(cudaEventRecord(K->ev[3], st));
    if (K->ntriples > 0) {
        bk_fold_kernel<<<(K->ntriples + 255) / 256, 256, 0, st>>>(Tg.slots, Tg.slot_of, K->ntriples, Tg.ctas,
                                                                  (long long)Tg.ntiles * (TJ * TD), out);
        APK_CUDA(cudaGetLastError());
    }
    return 0;
}

// zero the fields, fill the shells, c2r: the Nb shell fields of `c1` (or the indicators) in the scratch
int bk_fields(apk_bispec *K, const void *c1, const void *c1s, void *scratch, cudaStream_t st, bool dbl, bool timing) {
    apk_plan *P = K->plan;
    const size_t per = (size_t)P->N * P->N * P->ldz * (dbl ? sizeof(double) : sizeof(float));
    APK_CUDA(cudaMemsetAsync(scratch, 0, per * K->nbins, st));
    BkFillArgs F;
    F.c1 = (const float2 *)c1; F.c1s = (const float2 *)c1s;
    F.ka2 = K->ka2; F.kb2 = K->kb2; F.kz2 = K->kz2; F.edges2 = K->edges2;
    F.ic_a = K->ic_a; F.ic_b = K->ic_b; F.ic_z = K->ic_z;
    F.ph_a = K->ph_a; F.ph_b = K->ph_b; F.ph_z = K->ph_z;
    F.N = P->N; F.Nk = P->Nk; F.nedges = K->nedges;
    F.field_cplx = (long long)P->N * P->N * P->Nk;
    F.kmin_f = (float)K->edges[0]; F.inv_dk_f = (float)(1.0 / (K->edges[1] - K->edges[0]));
    F.fields = scratch;
    const long long modes = (long long)P->N * P->N * P->Nk;
    const int blocks = (int)std::min<long long>((modes + BK_FILL_THREADS - 1) / BK_FILL_THREADS, (long long)P->num_sms * 16);
    const bool inter = c1s != nullptr, comp = K->has_comp;
    if (dbl) bk_fill_kernel<true, false, false><<<blocks, BK_FILL_THREADS, 0, st>>>(F);
    else if (inter && comp) bk_fill_kernel<false, true, true><<<blocks, BK_FILL_THREADS, 0, st>>>(F);
    else if (inter) bk_fill_kernel<false, true, false><<<blocks, BK_FILL_THREADS, 0, st>>>(F);
    else if (comp) bk_fill_kernel<false, false, true><<<blocks, BK_FILL_THREADS, 0, st>>>(F);
    else bk_fill_kernel<false, false, false><<<blocks, BK_FILL_THREADS, 0, st>>>(F);
    APK_CUDA(cudaGetLastError());
    if (timing) APK_CUDA(cudaEventRecord(K->ev[1], st));
    cufftHandle h = dbl ? K->fft_d : K->fft_f;
    APK_CUFFT(cufftSetStream(h, st));
    const size_t ws = dbl ? K->ws_d : K->ws_f;
    if (ws) APK_CUFFT(cufftSetWorkArea(h, (char *)scratch + ((bk_fields_bytes(K) + 255) & ~(size_t)255)));
    for (int b = 0; b < K->nbins; b += K->batch) {
        char *f = (char *)scratch + per * b;
        if (dbl) APK_CUFFT(cufftExecZ2D(h, (cufftDoubleComplex *)f, (cufftDoubleReal *)f));
        else APK_CUFFT(cufftExecC2R(h, (cufftComplex *)f, (cufftReal *)f));
    }
    if (timing) APK_CUDA(cudaEventRecord(K->ev[2], st));
    return 0;
}

int bk_check_scratch(const apk_bispec *K, void *scratch, size_t bytes, const char *who) {
    size_t need = 0;
    apk_bispec_scratch_bytes(K, &need);
    APK_REQUIRE(scratch && bytes >= need, "%s: scratch of %zu bytes needed, %zu given (apk_bispec_scratch_bytes)", who, need, bytes);
    return 0;
}

}  // namespace

extern "C" {

int apk_bispec_create(apk_bispec **out, apk_plan *P, double kmin, double dk, double kmax, int k_dtype, int resampler,
                      int interlaced) {
    APK_REQUIRE(out && P, "apk_bispec_create: null argument");
    APK_REQUIRE(P->n0 == P->N, "apk_bispec_create: single-GPU plans only (slab plans have no bispectrum path)");
    APK_REQUIRE(k_dtype == APK_F32 || k_dtype == APK_F64, "apk_bispec_create: bad k_dtype %d", k_dtype);
    APK_REQUIRE(resampler == 0 || resampler == APK_CIC || resampler == APK_TSC,
                "apk_bispec_create: compensation needs CIC or TSC (0 = none), got %d", resampler);
    const int N = P->N, Nk = P->Nk;
    const double L = P->L, pi = 3.141592653589793, knyq = pi * (double)N / L;
    if (!(dk > 0.0)) dk = 2.0 * pi / L;
    if (!(kmax > 0.0)) kmax = 2.0 / 3.0 * knyq;                  // every triangle free of aliasing
    APK_REQUIRE(kmax <= knyq * (1.0 + 1e-12), "apk_bispec_create: kmax %g is beyond the Nyquist wavenumber %g", kmax, knyq);
    int ne = 0;
    if (int rc = apk_tables_k_edges(N, L, kmin, dk, kmax, nullptr, 0, &ne)) return rc;
    APK_REQUIRE(ne >= 2, "apk_bispec_create: the binning needs at least two k edges (kmin %g, dk %g, kmax %g)", kmin, dk, kmax);
    APK_REQUIRE(ne - 1 <= BK_MAX_BINS, "apk_bispec_create: %d shells, at most %d (increase dk)", ne - 1, BK_MAX_BINS);
    std::vector<double> edges(ne);
    if (int rc = apk_tables_k_edges(N, L, kmin, dk, kmax, edges.data(), ne, &ne)) return rc;
    APK_REQUIRE(edges[0] >= 0.0, "apk_bispec_create: kmin must be non-negative");
    APK_REQUIRE(edges[ne - 1] < knyq, "apk_bispec_create: the last edge %g reaches the Nyquist wavenumber %g", edges[ne - 1], knyq);
    DeviceGuard guard(P->device);

    apk_bispec *K = new apk_bispec();
    K->plan = P; K->nedges = ne; K->nbins = ne - 1; K->edges = edges;
    K->interlaced = interlaced != 0; K->has_comp = resampler != 0;
    // kept triples i <= j <= l: skipped only when no triangle can close, directly or modulo the grid
    const int nb = K->nbins;
    for (int i = 0; i < nb; ++i)
        for (int j = i; j < nb; ++j)
            for (int l = j; l < nb; ++l) {
                const double hij = edges[i + 1] + edges[j + 1];
                if (edges[l] >= hij && hij + edges[l + 1] <= 2.0 * knyq) continue;
                K->triples.push_back(i); K->triples.push_back(j); K->triples.push_back(l);
            }
    K->ntriples = (int)(K->triples.size() / 3);

    // tables: k^2 per axis (squares of the library's k table), edges^2, 1 / comp, exp(i phase)
    std::vector<double> k(N), comp, phase;
    apk_tables_k_axis(N, L, k_dtype, k.data());
    const size_t nd = (size_t)N + N + Nk + ne, nf = K->has_comp ? (size_t)N + N + Nk : 0, nc = K->interlaced ? (size_t)N + N + Nk : 0;
    const size_t bytes = nd * 8 + nc * 8 + ((nf + 1) & ~(size_t)1) * 4;
    std::vector<unsigned char> host(bytes);
    double *hd = (double *)host.data();
    float2 *hc = (float2 *)(hd + nd);
    float *hf = (float *)(hc + nc);
    size_t o = 0;
    for (int i = 0; i < N; ++i) hd[o++] = k[i] * k[i];
    for (int i = 0; i < N; ++i) hd[o++] = k[i] * k[i];
    for (int i = 0; i < Nk; ++i) hd[o++] = k[i] * k[i];
    for (int i = 0; i < ne; ++i) hd[o++] = edges[i] * edges[i];
    if (K->has_comp) {
        comp.resize(N);
        apk_tables_compensation(resampler, interlaced, N, comp.data());
        o = 0;
        for (int i = 0; i < N; ++i) hf[o++] = (float)(1.0 / comp[i]);
        for (int i = 0; i < N; ++i) hf[o++] = (float)(1.0 / comp[i]);
        for (int i = 0; i < Nk; ++i) hf[o++] = (float)(1.0 / comp[i]);
    }
    if (K->interlaced) {
        phase.resize(N);
        apk_tables_interlace_phase(N, L, phase.data());
        o = 0;
        for (int d = 0; d < 3; ++d)
            for (int i = 0; i < (d == 2 ? Nk : N); ++i) hc[o++] = make_float2((float)cos(phase[i]), (float)sin(phase[i]));
    }
    int rc = 0;
    if (cudaMalloc(&K->tables, bytes) != cudaSuccess) { set_error("apk_bispec_create: cudaMalloc(%zu) failed", bytes); rc = 1; }
    if (!rc && cudaMemcpy(K->tables, host.data(), bytes, cudaMemcpyHostToDevice) != cudaSuccess) {
        set_error("apk_bispec_create: table upload failed"); rc = 1;
    }
    if (!rc) {
        double *dd = (double *)K->tables;
        K->ka2 = dd; K->kb2 = dd + N; K->kz2 = K->kb2 + N; K->edges2 = K->kz2 + Nk;
        float2 *dc = (float2 *)(dd + nd);
        if (K->interlaced) { K->ph_a = dc; K->ph_b = dc + N; K->ph_z = K->ph_b + N; }
        float *df = (float *)(dc + nc);
        if (K->has_comp) { K->ic_a = df; K->ic_b = df + N; K->ic_z = K->ic_b + N; }
        // shells per cuFFT execution: a divisor of Nb, at most 2^24 points per execution
        const long long pts = (long long)N * N * N;
        for (int b = 1; b <= nb; ++b)
            if (nb % b == 0 && (long long)b * pts <= (1LL << 24)) K->batch = b;
        rc = bk_make_fft(K, false);
        if (!rc) rc = bk_make_fft(K, true);
        if (!rc) rc = bk_make_tiling<float>(K, K->tf);
        if (!rc) rc = bk_make_tiling<double>(K, K->td);
    }
    if (rc) { apk_bispec_destroy(K); return rc; }
    *out = K;
    return 0;
}

int apk_bispec_destroy(apk_bispec *K) {
    if (!K) return 0;
    DeviceGuard guard(K->plan->device);
    if (K->has_fft_f) cufftDestroy(K->fft_f);
    if (K->has_fft_d) cufftDestroy(K->fft_d);
    if (K->tables) cudaFree(K->tables);
    bk_free_tiling(K->tf);
    bk_free_tiling(K->td);
    if (K->ev_ready) for (auto &e : K->ev) cudaEventDestroy(e);
    delete K;
    return 0;
}

int apk_bispec_triples(const apk_bispec *K, int *ijl_host, int capacity, int *ntriples) {
    APK_REQUIRE(K && ntriples, "apk_bispec_triples: null argument");
    *ntriples = K->ntriples;
    if (ijl_host) {
        APK_REQUIRE(capacity >= K->ntriples, "apk_bispec_triples: %d triples, room for %d", K->ntriples, capacity);
        for (size_t i = 0; i < K->triples.size(); ++i) ijl_host[i] = K->triples[i];
    }
    return 0;
}

int apk_bispec_scratch_bytes(const apk_bispec *K, size_t *bytes) {
    APK_REQUIRE(K && bytes, "apk_bispec_scratch_bytes: null argument");
    *bytes = ((bk_fields_bytes(K) + 255) & ~(size_t)255) + std::max(K->ws_f, K->ws_d) + 256;
    return 0;
}

int apk_bispec_count(apk_bispec *K, void *scratch, size_t bytes, int64_t *ntri_dev, double *residual_host, void *stream) {
    APK_REQUIRE(K && ntri_dev, "apk_bispec_count: null argument");
    DeviceGuard guard(K->plan->device);
    cudaStream_t st = (cudaStream_t)stream;
    if (!K->counted) {
        if (int rc = bk_check_scratch(K, scratch, bytes, "apk_bispec_count")) return rc;
        if (int rc = bk_fields(K, nullptr, nullptr, scratch, st, true, false)) return rc;
        double *td = nullptr;
        APK_CUDA(cudaMalloc(&td, sizeof(double) * std::max(1, K->ntriples)));
        int rc = bk_reduce<double>(K, K->td, scratch, td, st, false);
        std::vector<double> host(K->ntriples);
        if (!rc && K->ntriples && cudaMemcpyAsync(host.data(), td, sizeof(double) * K->ntriples, cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = 1;
        if (!rc && cudaStreamSynchronize(st) != cudaSuccess) rc = 1;
        cudaFree(td);
        if (rc == 1 && !*apk_last_error()) set_error("apk_bispec_count: copying the counts to the host failed");
        if (rc) return rc;
        const double cells = (double)K->plan->N * K->plan->N * K->plan->N;
        std::vector<int64_t> n(K->ntriples);
        double res = 0.0;
        for (int t = 0; t < K->ntriples; ++t) {
            const double v = host[t] / cells;
            n[t] = (int64_t)std::rint(v);
            res = std::max(res, std::fabs(v - (double)n[t]));
        }
        APK_REQUIRE(res <= 0.1, "apk_bispec_count: the float64 triangle counts are off an integer by %g (> 0.1): precision "
                    "lost at this mesh size", res);
        K->ntri = n; K->residual = res; K->counted = true;
    }
    if (residual_host) *residual_host = K->residual;
    if (K->ntriples) {
        APK_CUDA(cudaMemcpyAsync(ntri_dev, K->ntri.data(), sizeof(int64_t) * K->ntriples, cudaMemcpyHostToDevice, st));
        APK_CUDA(cudaStreamSynchronize(st));             // the host vector is pageable: keep the copy ordered and done
    }
    return 0;
}

int apk_bispec_measure(apk_bispec *K, const void *c1, const void *c1s, void *scratch, size_t bytes, double *tsum_dev,
                       void *stream) {
    APK_REQUIRE(K && c1 && tsum_dev, "apk_bispec_measure: null argument");
    APK_REQUIRE((c1s != nullptr) == K->interlaced, "apk_bispec_measure: an interlaced twin is given iff the object was "
                "created with interlaced != 0");
    if (int rc = bk_check_scratch(K, scratch, bytes, "apk_bispec_measure")) return rc;
    DeviceGuard guard(K->plan->device);
    cudaStream_t st = (cudaStream_t)stream;
    const bool timing = K->plan->timing;
    if (timing && !K->ev_ready) {
        for (auto &e : K->ev) APK_CUDA(cudaEventCreate(&e));
        K->ev_ready = true;
    }
    if (timing) APK_CUDA(cudaEventRecord(K->ev[0], st));
    if (int rc = bk_fields(K, c1, c1s, scratch, st, false, timing)) return rc;
    if (int rc = bk_reduce<float>(K, K->tf, scratch, tsum_dev, st, timing)) return rc;
    if (timing) APK_CUDA(cudaEventRecord(K->ev[4], st));
    K->timed = timing;
    return 0;
}

int apk_bispec_last_ms(apk_bispec *K, float ms[4]) {
    APK_REQUIRE(K && ms, "apk_bispec_last_ms: null argument");
    APK_REQUIRE(K->timed, "apk_bispec_last_ms: no timed apk_bispec_measure on this object (apk_plan_enable_timing)");
    DeviceGuard guard(K->plan->device);
    APK_CUDA(cudaEventSynchronize(K->ev[4]));
    for (int i = 0; i < 4; ++i) APK_CUDA(cudaEventElapsedTime(&ms[i], K->ev[i], K->ev[i + 1]));
    return 0;
}

}  // extern "C"
