// Two-point correlation function xi(r) by the FFT estimator: FFTCorr(mode="1d" | "2d", poles=) on the device.
//
//   p(k) = c1(k) conj(c2(k)), k = 0 zeroed            (c = r2c of the mesh, interlace-combined and divided by the
//                                                      window as in bin_power.cu; c2 = c1 for an auto correlation)
//   xi(r_n) = Re sum_{stored k} w(k) p(k) e^{i k.r_n}  (w = 2 on the non-singular z planes, 1 on iz = 0 and iz = N/2)
//
// cuFFT's C2R extends the half grid by p(-k) := conj p(k).  On the self-paired planes (iz = 0 and, for even N, iz = N/2)
// interlacing makes the stored p non-Hermitian, and cuFFT does not define its result for such input; there the fill
// writes the Hermitian part H(k) = (p(k) + conj p(k')) / 2, k' = ((N - ia) % N, (N - ib) % N, iz).  Both members of a
// pair compute p(k) and p(k') with the same code and no FMA contraction, so they are exact conjugates in floating point
// and self-paired points get an exactly zero imaginary part: the C2R of the filled half grid is then exactly the sum
// above.  The fill writes into the caller's output buffer (never in place: a thread would read a partner that another
// thread has already overwritten, and the caller's fields stay untouched), scaled by a power of two 2^-e with
// e = round(log2 N^3), so that the C2R's sum over N^3 modes stays as large as its inputs, not N^3 times larger.
//
// Binning (nbodykit project_to_basis on the real grid): every one of the N^3 points has weight 1;
// r^2 = (ra^2 + rb^2) + rz^2 from the host-built squares of r_axis = freq_index(N) * (L / N) (two DADDs, no squaring on
// the device), numpy.digitize(r^2, edges^2) by a float guess fixed with float64 compares; mu = (r . los) / |r| (0 at
// r = 0) and numpy.digitize(|mu|, linspace(0, 1, Nmu + 1)) as in bin_kmu.cu, the mu = 1 column folded into the last one;
// multipoles (2 ell + 1) L_ell(mu) xi with SIGNED mu.  r = 0 is an ordinary point (the shot-noise spike lands in the
// first bin when rmin = 0).  Points outside [edges[0], edges[-1]) are neither read nor accumulated.
//
// Kernels
//   xi_fill_kernel   one pass over the half grid: c1 (+ twin), c2 (+ twin) -> p -> plane-symmetrised, scaled output.
//   cuFFT C2R        single mesh, in place in the output buffer; plan owned by the object, work area in caller scratch.
//   xi_bin_kernel    GEO: counts, sum |r|, sum |mu| -- they depend on the binning alone, so they are computed once per
//                    object with REDs into private global histograms and cached.  DATA (per call): a warp takes 32
//                    consecutive z of a row and walks y (coalesced loads); a thread keeps the sums of its current bin in
//                    registers and adds them to the CTA's float64 shared-memory histogram when the bin changes; the CTA
//                    sends its histogram to one of XI_NCOPY private global copies with REDs at the end.
//   xi_fold_kernel   the copies in a fixed order, the mu = 1 column folded, the data sums divided by 2^-e (exact).
#include "apk_common.cuh"
#include <algorithm>
#include <cmath>
#include <vector>

namespace apk {

constexpr int XI_FILL_THREADS = 256, XI_BIN_THREADS = 256, XI_NCOPY = 32, XI_MAXL = 8, XI_SEG = 32;
constexpr long long XI_MAX_HIST = 25600;          // float64 entries of the per-CTA histogram (200 KB of shared memory)

struct XiFillArgs {
    const float2 *c1, *c1s, *c2, *c2s;
    const float *ic_a, *ic_b, *ic_z;              // 1 / comp^2 (NULL: no compensation)
    const float2 *ph_a, *ph_b, *ph_z;             // exp(i phase) (NULL: not interlaced)
    int N, Nk;
    float fac;                                    // 2^-e
    float2 *out;                                  // [N][N][Nk] (the caller's padded mesh)
};

// no contraction: the two threads of a mirrored pair must get bit-identical products
__device__ __forceinline__ float2 xi_cmul(float2 a, float2 b) {
    return make_float2(__fsub_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y)), __fadd_rn(__fmul_rn(a.x, b.y), __fmul_rn(a.y, b.x)));
}

// p = c1 conj(c2) of mode (ia, ib, iz): interlace-combine, product and 1 / comp^2 in bin_power.cu's expression order
template <bool INTERLACED, bool CROSS, bool COMP>
__device__ __forceinline__ float2 xi_product(const XiFillArgs &A, int ia, int ib, int iz) {
    if (ia == 0 && ib == 0 && iz == 0) return make_float2(0.f, 0.f);
    const size_t idx = ((size_t)ia * A.N + ib) * A.Nk + iz;
    float2 a = A.c1[idx];
    float2 ph = make_float2(1.f, 0.f);
    if (INTERLACED) {
        ph = xi_cmul(xi_cmul(A.ph_a[ia], A.ph_z[iz]), A.ph_b[ib]);
        const float2 s = xi_cmul(A.c1s[idx], ph);
        a = make_float2(__fmul_rn(0.5f, __fadd_rn(a.x, s.x)), __fmul_rn(0.5f, __fadd_rn(a.y, s.y)));
    }
    float pre, pim;
    if (CROSS) {
        float2 b = A.c2[idx];
        if (INTERLACED) {
            const float2 s = xi_cmul(A.c2s[idx], ph);
            b = make_float2(__fmul_rn(0.5f, __fadd_rn(b.x, s.x)), __fmul_rn(0.5f, __fadd_rn(b.y, s.y)));
        }
        pre = __fadd_rn(__fmul_rn(a.x, b.x), __fmul_rn(a.y, b.y));
        pim = __fsub_rn(__fmul_rn(a.y, b.x), __fmul_rn(a.x, b.y));
    } else {
        pre = __fadd_rn(__fmul_rn(a.x, a.x), __fmul_rn(a.y, a.y));
        pim = 0.f;
    }
    if (COMP) {
        const float ic = __fmul_rn(__fmul_rn(A.ic_a[ia], A.ic_z[iz]), A.ic_b[ib]);
        pre = __fmul_rn(pre, ic); pim = __fmul_rn(pim, ic);
    }
    return make_float2(pre, pim);
}

template <bool INTERLACED, bool CROSS, bool COMP>
__global__ void __launch_bounds__(XI_FILL_THREADS)
xi_fill_kernel(XiFillArgs A) {
    const long long total = (long long)A.N * A.N * A.Nk;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x; m < total; m += stride) {
        const int iz = (int)(m % A.Nk);
        const long long r = m / A.Nk;
        const int ib = (int)(r % A.N), ia = (int)(r / A.N);
        float2 p = xi_product<INTERLACED, CROSS, COMP>(A, ia, ib, iz);
        if (iz == 0 || 2 * iz == A.N) {                          // self-paired plane: the Hermitian part
            const float2 q = xi_product<INTERLACED, CROSS, COMP>(A, (A.N - ia) % A.N, (A.N - ib) % A.N, iz);
            p = make_float2(__fmul_rn(0.5f, __fadd_rn(p.x, q.x)), __fmul_rn(0.5f, __fsub_rn(p.y, q.y)));
        }
        A.out[m] = make_float2(__fmul_rn(p.x, A.fac), __fmul_rn(p.y, A.fac));
    }
}

struct XiBinArgs {
    const float *grid;                // [N][N][ldz] real (after the C2R)
    const double *r, *r2, *edges2, *muedges;
    int N, ldz, nedges, nmu, nell;
    int ells[XI_MAXL], lmax;
    double inv_n1[17];                // 1 / (n + 1)
    double los[3];
    float rmin_f, inv_dr_f;
    long long nbins;                  // (nedges + 1) * (nmu + 2)
    double *copies;                   // GEO: [XI_NCOPY][3][nbins] (rsum, musum, count as u64); DATA: [XI_NCOPY][nell][nbins]
};

__device__ __forceinline__ void xi_red_f64(double *addr, double v) {
    asm volatile("red.global.add.f64 [%0], %1;" ::"l"(addr), "d"(v) : "memory");
}
__device__ __forceinline__ void xi_red_u64(unsigned long long *addr, unsigned long long v) {
    asm volatile("red.global.add.u64 [%0], %1;" ::"l"(addr), "l"(v) : "memory");
}

// MU: (r, mu) bins and multipoles (otherwise every point is in mu column 1: the 1-D fast path).  GEO: the geometry
// sums (no grid read); otherwise the data sums.
template <bool MU, bool GEO>
__global__ void __launch_bounds__(XI_BIN_THREADS)
xi_bin_kernel(XiBinArgs A) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double *s_hist = reinterpret_cast<double *>(smem_raw);       // DATA: [nell][nbins], this CTA's sums
    const long long nbins = A.nbins;
    const int nell = A.nell, nmu = A.nmu, nedges = A.nedges, N = A.N;
    if (!GEO) {
        for (long long i = threadIdx.x; i < nell * nbins; i += blockDim.x) s_hist[i] = 0.0;
        __syncthreads();
    }
    double *copy = A.copies + (size_t)(blockIdx.x % XI_NCOPY) * (GEO ? 3 : nell) * nbins;
    const int lane = threadIdx.x & 31;
    const long long warps_total = (long long)gridDim.x * (blockDim.x / 32);
    const long long warp_id = (long long)blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    const int n_zc = (N + 31) / 32, n_sb = (N + XI_SEG - 1) / XI_SEG;
    const long long n_items = (long long)N * n_sb * n_zc;
    const double e2_first = A.edges2[0], e2_last = A.edges2[nedges - 1];

    for (long long item = warp_id; item < n_items; item += warps_total) {
        const int zc = (int)(item % n_zc);
        const long long rr = item / n_zc;
        const int sb = (int)(rr % n_sb), ia = (int)(rr / n_sb);
        const int iz = zc * 32 + lane;
        if (iz >= N) continue;
        const double ra2 = A.r2[ia], rz2 = A.r2[iz];
        double ral = 0.0, rzl = 0.0;
        if (MU) { ral = __dmul_rn(A.r[ia], A.los[0]); rzl = __dmul_rn(A.r[iz], A.los[2]); }
        const float *row = A.grid + (size_t)ia * N * A.ldz + iz;
        long long cur = -1;
        double ax = 0.0, am = 0.0, ay[XI_MAXL];
        unsigned int an = 0;
#pragma unroll
        for (int i = 0; i < XI_MAXL; ++i) ay[i] = 0.0;
        auto flush = [&]() {
            if (cur < 0) return;
            if (GEO) {
                xi_red_f64(copy + cur, ax);
                if (MU) xi_red_f64(copy + nbins + cur, am);
                xi_red_u64(reinterpret_cast<unsigned long long *>(copy + 2 * nbins) + cur, (unsigned long long)an);
                ax = 0.0; am = 0.0; an = 0;
            } else {
#pragma unroll
                for (int i = 0; i < XI_MAXL; ++i)
                    if (i < (MU ? nell : 1)) { atomicAdd(s_hist + i * nbins + cur, ay[i]); ay[i] = 0.0; }
            }
        };
        const int ib1 = min((sb + 1) * XI_SEG, N);
        for (int ib = sb * XI_SEG; ib < ib1; ++ib) {
            const double r2 = __dadd_rn(__dadd_rn(ra2, A.r2[ib]), rz2);
            if (r2 >= e2_last || r2 < e2_first) continue;           // outside the edges: neither read nor accumulated
            // ---- r bin: numpy.digitize(r2, edges^2) ----
            int rbin = (int)((sqrtf((float)r2) - A.rmin_f) * A.inv_dr_f) + 1;
            rbin = max(1, min(rbin, nedges - 1));
            while (r2 < A.edges2[rbin - 1]) --rbin;
            while (r2 >= A.edges2[rbin]) ++rbin;
            // ---- mu and its bin: numpy.digitize(|mu|, linspace(0, 1, Nmu + 1)) -> 1 .. Nmu + 1 ----
            int mbin = 1;
            double mu = 0.0, amu = 0.0;
            if (MU) {
                const double rdl = __dadd_rn(__dadd_rn(ral, __dmul_rn(A.r[ib], A.los[1])), rzl);
                const double rnorm = sqrt(r2);
                mu = rnorm > 0.0 ? rdl / rnorm : 0.0;
                amu = fabs(mu);
                mbin = min(max((int)(amu * nmu) + 1, 1), nmu + 1);
                while (mbin > 1 && amu < A.muedges[mbin - 1]) --mbin;
                while (mbin <= nmu && amu >= A.muedges[mbin]) ++mbin;
            }
            const long long bin = (long long)rbin * (nmu + 2) + mbin;
            if (bin != cur) { flush(); cur = bin; }
            if (GEO) {
                ax += sqrt(r2);
                am += amu;
                ++an;
            } else {
                const double v = (double)row[(size_t)ib * A.ldz];
                if (MU) {
                    // P_0 .. P_lmax by Bonnet's recursion; the division by n + 1 is a multiplication by the host's
                    // reciprocal (a double division's slow path is a call, whose register save would spill)
                    double p0 = 1.0, p1 = mu;
                    for (int n = 0; n <= A.lmax; ++n) {
                        const double pn = n == 0 ? 1.0 : p1;
#pragma unroll
                        for (int i = 0; i < XI_MAXL; ++i)
                            if (i < nell && A.ells[i] == n) ay[i] += (2.0 * n + 1.0) * pn * v;
                        if (n >= 1) {
                            const double t = ((2 * n + 1) * mu * p1 - n * p0) * A.inv_n1[n];
                            p0 = p1; p1 = t;
                        }
                    }
                } else {
                    ay[0] += v;
                }
            }
        }
        flush();
    }
    if (!GEO) {
        __syncthreads();
        for (long long i = threadIdx.x; i < nell * nbins; i += blockDim.x)
            if (s_hist[i] != 0.0) xi_red_f64(copy + i, s_hist[i]);
    }
}

// out[arr][b] = sum over the copies in a fixed order (row u64_row as uint64), the internal mu == 1 column (Nmu + 1)
// added to the last visible one; float64 rows are multiplied by `scale`
__global__ void __launch_bounds__(256)
xi_fold_kernel(const double *copies, int narr, long long nbins, int nmu, int u64_row, double scale, double *out) {
    const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nbins) return;
    const int m = (int)(b % (nmu + 2));
    for (int arr = 0; arr < narr; ++arr) {
        double s = 0.0;
        unsigned long long n = 0;
        for (int c = 0; c < XI_NCOPY; ++c) {
            const double *src = copies + ((size_t)c * narr + arr) * nbins;
            for (int part = 0; part < 2; ++part) {
                if (part == 1 && m != nmu) break;
                if (arr == u64_row) n += reinterpret_cast<const unsigned long long *>(src)[b + part];
                else s += src[b + part];
            }
        }
        if (arr == u64_row) reinterpret_cast<unsigned long long *>(out)[(size_t)arr * nbins + b] = n;
        else out[(size_t)arr * nbins + b] = s * scale;
    }
}

}  // namespace apk

using namespace apk;

struct apk_xi {
    apk_plan *plan = nullptr;
    int nedges = 0, nmu = 1, nell = 1;
    int ells[XI_MAXL] = {};
    double los[3] = {0, 0, 1};
    bool mu_path = false, interlaced = false, has_comp = false;
    std::vector<double> edges;
    double fac = 1.0;                 // 2^-e: the output grid holds fac * sum w p e^{ikr} of the un-normalised fields
    void *tables = nullptr;
    double *r = nullptr, *r2 = nullptr, *edges2 = nullptr, *muedges = nullptr;
    float *ic_a = nullptr, *ic_b = nullptr, *ic_z = nullptr;
    float2 *ph_a = nullptr, *ph_b = nullptr, *ph_z = nullptr;
    double *copies = nullptr;         // [XI_NCOPY][max(3, nell)][nbins]
    double *geo = nullptr;            // [3][nbins], once per object
    bool geo_done = false;
    cufftHandle fft = 0;
    bool has_fft = false;
    size_t ws = 0;
    cudaEvent_t ev[4] = {};
    bool ev_ready = false, timed = false;
};

namespace {

long long xi_nbins(const apk_xi *X) { return (long long)(X->nedges + 1) * (X->nmu + 2); }
size_t xi_hist_bytes(const apk_xi *X) { return sizeof(double) * (size_t)X->nell * (size_t)xi_nbins(X); }
size_t xi_grid_bytes(const apk_plan *P) { return sizeof(float) * (size_t)P->N * P->N * P->ldz; }

bool overlaps(const void *a, const void *b, size_t bytes) {
    if (!a || !b) return false;
    const char *x = (const char *)a, *y = (const char *)b;
    return x < y + bytes && y < x + bytes;
}

int xi_bin_launch(apk_xi *X, const float *grid, bool geo, cudaStream_t st) {
    apk_plan *P = X->plan;
    XiBinArgs A;
    A.grid = grid;
    A.r = X->r; A.r2 = X->r2; A.edges2 = X->edges2; A.muedges = X->muedges;
    A.N = P->N; A.ldz = P->ldz; A.nedges = X->nedges; A.nmu = X->nmu; A.nell = X->nell;
    A.lmax = 0;
    for (int i = 0; i < XI_MAXL; ++i) { A.ells[i] = X->ells[i]; if (i < X->nell) A.lmax = std::max(A.lmax, X->ells[i]); }
    for (int n = 0; n < 17; ++n) A.inv_n1[n] = 1.0 / (n + 1);
    for (int d = 0; d < 3; ++d) A.los[d] = X->los[d];
    A.rmin_f = (float)X->edges[0]; A.inv_dr_f = (float)(1.0 / (X->edges[1] - X->edges[0]));
    A.nbins = xi_nbins(X);
    A.copies = X->copies;
    const int narr = geo ? 3 : X->nell;
    APK_CUDA(cudaMemsetAsync(X->copies, 0, sizeof(double) * XI_NCOPY * narr * (size_t)A.nbins, st));
    const size_t smem = geo ? 0 : xi_hist_bytes(X);
    auto kern = geo ? (X->mu_path ? xi_bin_kernel<true, true> : xi_bin_kernel<false, true>)
                    : (X->mu_path ? xi_bin_kernel<true, false> : xi_bin_kernel<false, false>);
    APK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    APK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, XI_BIN_THREADS, smem));
    const int ctas = P->num_sms * std::max(1, std::min(per_sm, 8));
    kern<<<ctas, XI_BIN_THREADS, smem, st>>>(A);
    APK_CUDA(cudaGetLastError());
    return 0;
}

int xi_fold(apk_xi *X, bool geo, double *out, cudaStream_t st) {
    const long long nb = xi_nbins(X);
    xi_fold_kernel<<<(unsigned)((nb + 255) / 256), 256, 0, st>>>(X->copies, geo ? 3 : X->nell, nb, X->nmu, geo ? 2 : -1,
                                                                  geo ? 1.0 : 1.0 / X->fac, out);
    APK_CUDA(cudaGetLastError());
    return 0;
}

}  // namespace

extern "C" {

int apk_xi_create(apk_xi **out, apk_plan *P, double rmin, double dr, double rmax, int nmu, const int *ells, int nell,
                  const double *los3, int resampler, int interlaced) {
    APK_REQUIRE(out && P && los3, "apk_xi_create: null argument");
    APK_REQUIRE(P->n0 == P->N, "apk_xi_create: single-GPU plans only (slab plans have no correlation-function path)");
    APK_REQUIRE(resampler == 0 || resampler == APK_CIC || resampler == APK_TSC,
                "apk_xi_create: compensation needs CIC or TSC (0 = none), got %d", resampler);
    APK_REQUIRE(std::isfinite(dr) && dr >= 0.0, "apk_xi_create: dr must be positive (0 = L / N), got %g", dr);
    APK_REQUIRE(std::isfinite(rmin) && rmin >= 0.0, "apk_xi_create: rmin must be non-negative, got %g", rmin);
    APK_REQUIRE(std::isfinite(rmax) && rmax >= 0.0, "apk_xi_create: rmax must be positive (0 = L / 2 + dr / 2), got %g", rmax);
    APK_REQUIRE(rmax == 0.0 || rmax > rmin, "apk_xi_create: rmax %g must exceed rmin %g", rmax, rmin);
    APK_REQUIRE(nmu >= 1 && nmu <= 4096, "apk_xi_create: need 1..4096 mu bins, got %d", nmu);
    APK_REQUIRE(ells && nell >= 1 && nell <= XI_MAXL && ells[0] == 0, "apk_xi_create: 1..%d multipoles, the monopole first",
                XI_MAXL);
    for (int i = 0; i < nell; ++i) APK_REQUIRE(ells[i] >= 0 && ells[i] <= 16, "apk_xi_create: multipole %d out of range", ells[i]);
    for (int d = 0; d < 3; ++d) APK_REQUIRE(std::isfinite(los3[d]), "apk_xi_create: los must be finite");
    const int N = P->N, Nk = P->Nk;
    const double L = P->L;
    int ne = 0;
    if (int rc = apk_tables_r_edges(N, L, rmin, dr, rmax, nullptr, 0, &ne)) return rc;
    APK_REQUIRE(ne >= 2, "apk_xi_create: the binning needs at least two r edges (rmin %g, dr %g, rmax %g: rmax must exceed "
                "rmin + dr)", rmin, dr, rmax);
    std::vector<double> edges(ne);
    if (int rc = apk_tables_r_edges(N, L, rmin, dr, rmax, edges.data(), ne, &ne)) return rc;
    const bool mu_path = !(nmu == 1 && nell == 1);
    const long long nbins = (long long)(ne + 1) * (nmu + 2);
    APK_REQUIRE((mu_path ? nell : 1) * nbins <= XI_MAX_HIST, "apk_xi_create: %lld (r, mu) bins x %d multipoles exceed the "
                "%lld sums of the per-CTA histogram: use a larger dr, fewer mu bins or fewer multipoles", nbins, nell, XI_MAX_HIST);
    DeviceGuard guard(P->device);

    apk_xi *X = new apk_xi();
    X->plan = P; X->nedges = ne; X->nmu = nmu; X->nell = mu_path ? nell : 1; X->edges = edges;
    for (int i = 0; i < nell; ++i) X->ells[i] = ells[i];
    for (int d = 0; d < 3; ++d) X->los[d] = los3[d];
    X->mu_path = mu_path; X->interlaced = interlaced != 0; X->has_comp = resampler != 0;
    X->fac = std::ldexp(1.0, -(int)std::lround(3.0 * std::log2((double)N)));

    // tables: r and r^2 per axis (the library's r table and its squares), edges^2, mu edges, 1 / comp^2, exp(i phase)
    std::vector<double> r(N), comp, phase;
    apk_tables_r_axis(N, L, r.data());
    const size_t nd = (size_t)N + N + ne + nmu + 1, nc = X->interlaced ? (size_t)N + N + Nk : 0;
    const size_t nf = X->has_comp ? (size_t)N + N + Nk : 0;
    const size_t bytes = nd * 8 + nc * 8 + ((nf + 1) & ~(size_t)1) * 4;
    std::vector<unsigned char> host(bytes);
    double *hd = (double *)host.data();
    float2 *hc = (float2 *)(hd + nd);
    float *hf = (float *)(hc + nc);
    size_t o = 0;
    for (int i = 0; i < N; ++i) hd[o++] = r[i];
    for (int i = 0; i < N; ++i) hd[o++] = r[i] * r[i];
    for (int i = 0; i < ne; ++i) hd[o++] = edges[i] * edges[i];
    // numpy.linspace(0, 1, Nmu + 1): i * step with step = 1 / Nmu, the last point set to the stop value
    for (int i = 0; i <= nmu; ++i) hd[o++] = i == nmu ? 1.0 : (double)i * (1.0 / (double)nmu);
    if (X->has_comp) {
        comp.resize(N);
        apk_tables_compensation(resampler, interlaced, N, comp.data());
        o = 0;
        for (int d = 0; d < 3; ++d)
            for (int i = 0; i < (d == 2 ? Nk : N); ++i) hf[o++] = (float)(1.0 / (comp[i] * comp[i]));
    }
    if (X->interlaced) {
        phase.resize(N);
        apk_tables_interlace_phase(N, L, phase.data());
        o = 0;
        for (int d = 0; d < 3; ++d)
            for (int i = 0; i < (d == 2 ? Nk : N); ++i) hc[o++] = make_float2((float)cos(phase[i]), (float)sin(phase[i]));
    }
    const size_t cbytes = sizeof(double) * XI_NCOPY * (size_t)std::max(3, X->nell) * nbins;
    int rc = 0;
    if (cudaMalloc(&X->tables, bytes) != cudaSuccess || cudaMalloc(&X->copies, cbytes) != cudaSuccess ||
        cudaMalloc(&X->geo, sizeof(double) * 3 * nbins) != cudaSuccess) {
        set_error("apk_xi_create: cudaMalloc(%zu + %zu) failed", bytes, cbytes); rc = 1;
    }
    if (!rc && cudaMemcpy(X->tables, host.data(), bytes, cudaMemcpyHostToDevice) != cudaSuccess) {
        set_error("apk_xi_create: table upload failed"); rc = 1;
    }
    if (!rc) {
        double *dd = (double *)X->tables;
        X->r = dd; X->r2 = dd + N; X->edges2 = X->r2 + N; X->muedges = X->edges2 + ne;
        float2 *dc = (float2 *)(dd + nd);
        if (X->interlaced) { X->ph_a = dc; X->ph_b = dc + N; X->ph_z = X->ph_b + N; }
        float *df = (float *)(dc + nc);
        if (X->has_comp) { X->ic_a = df; X->ic_b = df + N; X->ic_z = X->ic_b + N; }
        // C2R of one mesh, in place in the padded layout; work area in the caller's scratch
        rc = [&]() -> int {
            APK_CUFFT(cufftCreate(&X->fft));
            X->has_fft = true;
            APK_CUFFT(cufftSetAutoAllocation(X->fft, 0));
            long long n[3] = {N, N, N};
            long long inembed[3] = {N, N, Nk}, onembed[3] = {N, N, P->ldz};
            size_t ws = 0;
            APK_CUFFT(cufftMakePlanMany64(X->fft, 3, n, inembed, 1, (long long)N * N * Nk, onembed, 1,
                                          (long long)N * N * P->ldz, CUFFT_C2R, 1, &ws));
            X->ws = (ws + 255) & ~(size_t)255;
            return 0;
        }();
    }
    if (rc) { apk_xi_destroy(X); return rc; }
    *out = X;
    return 0;
}

int apk_xi_destroy(apk_xi *X) {
    if (!X) return 0;
    DeviceGuard guard(X->plan->device);
    if (X->has_fft) cufftDestroy(X->fft);
    if (X->tables) cudaFree(X->tables);
    if (X->copies) cudaFree(X->copies);
    if (X->geo) cudaFree(X->geo);
    if (X->ev_ready) for (auto &e : X->ev) cudaEventDestroy(e);
    delete X;
    return 0;
}

int apk_xi_edges(const apk_xi *X, double *edges_host, int capacity, int *n) {
    APK_REQUIRE(X && n, "apk_xi_edges: null argument");
    *n = X->nedges;
    if (edges_host) {
        APK_REQUIRE(capacity >= X->nedges, "apk_xi_edges: %d edges, room for %d", X->nedges, capacity);
        for (int i = 0; i < X->nedges; ++i) edges_host[i] = X->edges[i];
    }
    return 0;
}

int apk_xi_scratch_bytes(const apk_xi *X, size_t *bytes) {
    APK_REQUIRE(X && bytes, "apk_xi_scratch_bytes: null argument");
    *bytes = X->ws;
    return 0;
}

int apk_xi_grid_scale(const apk_xi *X, double *scale) {
    APK_REQUIRE(X && scale, "apk_xi_grid_scale: null argument");
    *scale = X->fac;
    return 0;
}

int apk_xi_measure(apk_xi *X, const void *c1, const void *c1s, const void *c2, const void *c2s, float *grid_out,
                   void *scratch, size_t bytes, double *sums_dev, void *stream) {
    APK_REQUIRE(X && c1 && sums_dev, "apk_xi_measure: null argument");
    APK_REQUIRE(grid_out, "apk_xi_measure: no output grid (a padded mesh of the plan)");
    APK_REQUIRE((c1s != nullptr) == X->interlaced, "apk_xi_measure: an interlaced twin is given iff the object was created "
                "with interlaced != 0");
    APK_REQUIRE(!c2s || c2, "apk_xi_measure: c2s without c2");
    APK_REQUIRE(!c2 || ((c2s != nullptr) == (c1s != nullptr)), "apk_xi_measure: both fields interlaced or neither");
    APK_REQUIRE(bytes >= X->ws && (scratch || X->ws == 0), "apk_xi_measure: scratch of %zu bytes needed, %zu given "
                "(apk_xi_scratch_bytes)", X->ws, scratch ? bytes : (size_t)0);
    apk_plan *P = X->plan;
    const size_t gb = xi_grid_bytes(P);
    for (const void *in : {c1, c1s, c2, c2s})
        APK_REQUIRE(!overlaps(in, grid_out, gb), "apk_xi_measure: the output grid overlaps an input field (the fill is "
                    "never in place)");
    APK_REQUIRE(!overlaps(scratch, grid_out, gb) || X->ws == 0, "apk_xi_measure: the scratch overlaps the output grid");
    DeviceGuard guard(P->device);
    cudaStream_t st = (cudaStream_t)stream;
    const bool timing = P->timing;
    if (timing && !X->ev_ready) {
        for (auto &e : X->ev) APK_CUDA(cudaEventCreate(&e));
        X->ev_ready = true;
    }
    if (!X->geo_done) {                   // counts, sum |r|, sum |mu|: once per object
        if (int rc = xi_bin_launch(X, nullptr, true, st)) return rc;
        if (int rc = xi_fold(X, true, X->geo, st)) return rc;
        X->geo_done = true;
    }
    if (timing) APK_CUDA(cudaEventRecord(X->ev[0], st));
    XiFillArgs F;
    F.c1 = (const float2 *)c1; F.c1s = (const float2 *)c1s; F.c2 = (const float2 *)c2; F.c2s = (const float2 *)c2s;
    F.ic_a = X->ic_a; F.ic_b = X->ic_b; F.ic_z = X->ic_z;
    F.ph_a = X->ph_a; F.ph_b = X->ph_b; F.ph_z = X->ph_z;
    F.N = P->N; F.Nk = P->Nk; F.fac = (float)X->fac;
    F.out = (float2 *)grid_out;
    const long long modes = (long long)P->N * P->N * P->Nk;
    const int blocks = (int)std::min<long long>((modes + XI_FILL_THREADS - 1) / XI_FILL_THREADS, (long long)P->num_sms * 16);
    const bool inter = c1s != nullptr, cross = c2 != nullptr, comp = X->has_comp;
#define APK_XI_GO(I, C, M) xi_fill_kernel<I, C, M><<<blocks, XI_FILL_THREADS, 0, st>>>(F)
    if (inter) { if (cross) { if (comp) APK_XI_GO(true, true, true); else APK_XI_GO(true, true, false); }
                 else { if (comp) APK_XI_GO(true, false, true); else APK_XI_GO(true, false, false); } }
    else { if (cross) { if (comp) APK_XI_GO(false, true, true); else APK_XI_GO(false, true, false); }
           else { if (comp) APK_XI_GO(false, false, true); else APK_XI_GO(false, false, false); } }
#undef APK_XI_GO
    APK_CUDA(cudaGetLastError());
    if (timing) APK_CUDA(cudaEventRecord(X->ev[1], st));
    APK_CUFFT(cufftSetStream(X->fft, st));
    if (X->ws) APK_CUFFT(cufftSetWorkArea(X->fft, scratch));
    APK_CUFFT(cufftExecC2R(X->fft, (cufftComplex *)grid_out, (cufftReal *)grid_out));
    if (timing) APK_CUDA(cudaEventRecord(X->ev[2], st));
    if (int rc = xi_bin_launch(X, grid_out, false, st)) return rc;
    const long long nb = xi_nbins(X);
    if (int rc = xi_fold(X, false, sums_dev + 3 * nb, st)) return rc;
    APK_CUDA(cudaMemcpyAsync(sums_dev, X->geo, sizeof(double) * 3 * nb, cudaMemcpyDeviceToDevice, st));
    if (timing) APK_CUDA(cudaEventRecord(X->ev[3], st));
    X->timed = timing;
    return 0;
}

int apk_xi_last_ms(apk_xi *X, float ms[3]) {
    APK_REQUIRE(X && ms, "apk_xi_last_ms: null argument");
    APK_REQUIRE(X->timed, "apk_xi_last_ms: no timed apk_xi_measure on this object (apk_plan_enable_timing)");
    DeviceGuard guard(X->plan->device);
    APK_CUDA(cudaEventSynchronize(X->ev[3]));
    for (int i = 0; i < 3; ++i) APK_CUDA(cudaEventElapsedTime(&ms[i], X->ev[i], X->ev[i + 1]));
    return 0;
}

}  // extern "C"
