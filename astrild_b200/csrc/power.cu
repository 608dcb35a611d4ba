// Binning tables and the one-call entry points of libastrild_pk.so (host code; SURVEY.md section 8b).
//
// The tables decide which float lands on which side of a bin edge, so they restate -- in IEEE double, expression by
// expression, no FMA contraction (-ffp-contract=off for the host compiler) -- what the reference stack computes on the
// host for the calls astrild makes at
//   /root/reference/src/astrild/power_spectra/power_spectrum_3d.py:181-195   FFTPower(first, mode="1d", kmin=2 pi / L)
//   /root/reference/src/astrild/particles/hutils/stats_subfind.py:142-148
// (pmesh ParticleMesh k tables, nbodykit FFTPower edges and Compensate* factors; SURVEY.md Appendix A.3-A.6).
// astrild_b200/tables.py is the same in NumPy; tests/test_abi.py compares the two bit for bit (k tables, edges, Hermitian
// weights) and to 1e-15 (sin / pow based compensation and phase tables).
//
// apk_power_from_particles / apk_power_from_mesh are what a C, Fortran or ctypes caller binds to get
// (k, P(k), Nmodes) in one call: SubFind.power_spectrum's numerical body (stats_subfind.py:129-150) and
// PowerSpectrum3D._power_spectrum_3d (power_spectrum_3d.py:164-226).
#include "apk_common.cuh"
#include <cmath>
#include <cstring>
#include <map>
#include <tuple>
#include <vector>

namespace apk {

static const double kPi = 3.141592653589793;          // numpy.pi

static inline long long freq_index(int i, int N) { return 2 * (long long)i < N ? i : (long long)i - N; }

static void k_axis(int N, double L, int k_dtype, double *out) {
    if (k_dtype == APK_F32) {                          // pmesh with a float32 index ramp (SURVEY Appendix C, Q1)
        const float f = (float)(2.0 * kPi / N), Nf = (float)N, Lf = (float)L;
        for (int i = 0; i < N; ++i) {
            volatile float w = (float)freq_index(i, N) * f;
            volatile float t = w * Nf;
            out[i] = (double)(float)(t / Lf);
        }
        return;
    }
    const double f = 2.0 * kPi / (double)N;
    for (int i = 0; i < N; ++i) {
        const double w = (double)freq_index(i, N) * f;   // w = n * (2 pi / N)
        const double t = w * (double)N;                  // k = w * N / L, left to right
        out[i] = t / L;
    }
}

// numpy.arange(start, stop, step) for float64: length ceil((stop - start) / step), value i = start + i * delta with
// delta = (start + step) - start (how NumPy fills a float range)
static int arange(double start, double stop, double step, std::vector<double> &out) {
    out.clear();
    if (!(step > 0.0) || !(stop > start)) return 0;
    const double len = std::ceil((stop - start) / step);
    if (!(len < 1e8)) return -1;
    const long long n = (long long)len;
    const double next = start + step;
    const double delta = next - start;
    out.resize((size_t)n);
    for (long long i = 0; i < n; ++i) out[(size_t)i] = start + (double)i * delta;
    return (int)n;
}

static int k_edges(int N, double L, double kmin, double dk, double kmax, std::vector<double> &out) {
    if (!(dk > 0.0)) dk = 2.0 * kPi / L;
    if (!(kmax > 0.0)) kmax = kPi * (double)N / L + dk / 2.0;
    return arange(kmin, kmax, dk, out);
}

static double np_sinc(double x) {                      // numpy.sinc: y = pi * where(x == 0, 1e-20, x); sin(y) / y
    const double y = kPi * (x == 0.0 ? 1.0e-20 : x);
    return std::sin(y) / y;
}

static void compensation_axis(int resampler, int interlaced, int N, double *out) {
    const double f = 2.0 * kPi / (double)N;
    for (int i = 0; i < N; ++i) {
        const double w = (double)freq_index(i, N) * f;
        if (interlaced) {
            const double s = np_sinc(w / (2.0 * kPi));
            out[i] = resampler == APK_CIC ? s * s : std::pow(s, 3.0);
        } else {
            const double h = std::sin(0.5 * w);
            const double s = h * h;
            out[i] = resampler == APK_CIC ? std::sqrt(1.0 - 2.0 / 3.0 * s) : std::sqrt(1.0 - s + 2.0 / 15.0 * s * s);
        }
    }
}

struct BinKey {
    double kmin, dk, kmax;
    int comp, interlaced, k_dtype;
    bool operator<(const BinKey &o) const {
        return std::tie(kmin, dk, kmax, comp, interlaced, k_dtype) < std::tie(o.kmin, o.dk, o.kmax, o.comp, o.interlaced, o.k_dtype);
    }
};

// binning objects of the one-call entry points, kept per plan (plans are not shared between host threads)
static std::map<std::pair<apk_plan *, BinKey>, apk_binning *> g_binnings;

static int get_binning(apk_plan *P, double kmin, double dk, double kmax, int comp_resampler, int interlaced, int k_dtype,
                       apk_binning **out, std::vector<double> *edges_out) {
    const BinKey key{kmin, dk, kmax, comp_resampler, interlaced, k_dtype};
    std::vector<double> edges;
    const int ne = k_edges(P->N, P->L, kmin, dk, kmax, edges);
    APK_REQUIRE(ne >= 2, "apk_power: the binning needs at least two k edges (kmin %g, dk %g, kmax %g)", kmin, dk, kmax);
    if (edges_out) *edges_out = edges;
    auto it = g_binnings.find({P, key});
    if (it != g_binnings.end()) { *out = it->second; return 0; }
    APK_REQUIRE(P->n0 == P->N, "apk_power: single-GPU plans only (slab plans: astrild_b200.distributed)");
    const int N = P->N, Nk = P->Nk;
    std::vector<double> k(N), wz(Nk), comp, phase;
    k_axis(N, P->L, k_dtype, k.data());
    for (int i = 0; i < Nk; ++i) wz[i] = freq_index(i, N) > 0 ? 2.0 : 1.0;
    if (comp_resampler) { comp.resize(N); compensation_axis(comp_resampler, interlaced, N, comp.data()); }
    if (interlaced) {
        std::vector<double> k64(N);
        k_axis(N, P->L, APK_F64, k64.data());
        phase.resize(N);
        for (int i = 0; i < N; ++i) phase[i] = 0.5 * k64[i] * (P->L / (double)N);
    }
    const double *c = comp.empty() ? nullptr : comp.data(), *ph = phase.empty() ? nullptr : phase.data();
    apk_binning *B = nullptr;
    if (int rc = apk_binning_create(&B, P, N, N, Nk, k.data(), k.data(), k.data(), wz.data(), edges.data(), ne, c, c, c, ph, ph, ph, 0, 0))
        return rc;
    g_binnings[{P, key}] = B;
    *out = B;
    return 0;
}

void forget_plan_binnings(apk_plan *P) {
    for (auto it = g_binnings.begin(); it != g_binnings.end();) {
        if (it->first.first == P) { apk_binning_destroy(it->second); it = g_binnings.erase(it); }
        else ++it;
    }
}

// shell sums on the device -> (k, power, modes) on the host, nbodykit's conventions (project_to_basis tail)
static int finish(apk_plan *P, apk_binning *B, const std::vector<double> &edges, const void *c1, const void *c1s, const void *c2,
                  const void *c2s, double scale, double *k_host, double *power_host, int64_t *modes_host, int capacity,
                  int *nbins, cudaStream_t st) {
    const int nb1 = (int)edges.size() + 1, nb = (int)edges.size() - 1;
    if (nbins) *nbins = nb;
    APK_REQUIRE(capacity >= nb, "apk_power: output arrays hold %d bins, %d needed", capacity, nb);
    double *dev = nullptr;
    APK_CUDA(cudaMalloc(&dev, sizeof(double) * 4 * (size_t)nb1));
    int rc = apk_bin_power(B, c1, c1s, c2, c2s, dev, dev + nb1, dev + 2 * nb1, (int64_t *)(dev + 3 * nb1), st);
    std::vector<double> host(4 * (size_t)nb1);
    if (!rc && cudaMemcpyAsync(host.data(), dev, sizeof(double) * host.size(), cudaMemcpyDeviceToHost, st) != cudaSuccess) rc = 1;
    if (!rc && cudaStreamSynchronize(st) != cudaSuccess) rc = 1;
    cudaFree(dev);
    if (rc == 1 && !*apk_last_error()) set_error("apk_power: copying the shell sums to the host failed");
    if (rc) return rc;
    const int64_t *nsum = (const int64_t *)(host.data() + 3 * (size_t)nb1);
    for (int b = 0; b < nb; ++b) {                       // drop digitize's under- and overflow bins
        const double n = (double)nsum[b + 1];
        k_host[b] = host[b + 1] / n;                     // mean |k| of the modes in the bin; NaN if empty
        power_host[b] = host[nb1 + b + 1] * scale / n;
        modes_host[b] = nsum[b + 1];
    }
    return 0;
}

}  // namespace apk

using namespace apk;

extern "C" {

int apk_tables_k_axis(int nmesh, double boxsize, int k_dtype, double *k_host) {
    APK_REQUIRE(nmesh >= 1 && boxsize > 0.0 && k_host, "apk_tables_k_axis: bad argument");
    k_axis(nmesh, boxsize, k_dtype, k_host);
    return 0;
}

int apk_tables_k_edges(int nmesh, double boxsize, double kmin, double dk, double kmax, double *edges_host, int capacity,
                       int *nedges) {
    APK_REQUIRE(nmesh >= 1 && boxsize > 0.0 && nedges, "apk_tables_k_edges: bad argument");
    std::vector<double> e;
    const int n = k_edges(nmesh, boxsize, kmin, dk, kmax, e);
    APK_REQUIRE(n >= 0, "apk_tables_k_edges: too many edges");
    *nedges = n;
    if (edges_host) {
        APK_REQUIRE(capacity >= n, "apk_tables_k_edges: %d edges, room for %d", n, capacity);
        std::memcpy(edges_host, e.data(), sizeof(double) * (size_t)n);
    }
    return 0;
}

int apk_tables_r_axis(int nmesh, double boxsize, double *r_host) {
    APK_REQUIRE(nmesh >= 1 && boxsize > 0.0 && r_host, "apk_tables_r_axis: bad argument");
    const double h = boxsize / (double)nmesh;
    for (int i = 0; i < nmesh; ++i) r_host[i] = (double)freq_index(i, nmesh) * h;
    return 0;
}

int apk_tables_r_edges(int nmesh, double boxsize, double rmin, double dr, double rmax, double *edges_host, int capacity,
                       int *nedges) {
    APK_REQUIRE(nmesh >= 1 && boxsize > 0.0 && nedges, "apk_tables_r_edges: bad argument");
    if (!(dr > 0.0)) dr = boxsize / (double)nmesh;
    if (!(rmax > 0.0)) rmax = boxsize / 2.0 + dr / 2.0;
    std::vector<double> e;
    const int n = arange(rmin, rmax, dr, e);
    APK_REQUIRE(n >= 0, "apk_tables_r_edges: too many edges");
    *nedges = n;
    if (edges_host) {
        APK_REQUIRE(capacity >= n, "apk_tables_r_edges: %d edges, room for %d", n, capacity);
        std::memcpy(edges_host, e.data(), sizeof(double) * (size_t)n);
    }
    return 0;
}

int apk_tables_hermitian_weights(int nmesh, double *w_host) {
    APK_REQUIRE(nmesh >= 1 && w_host, "apk_tables_hermitian_weights: bad argument");
    for (int i = 0; i < nmesh / 2 + 1; ++i) w_host[i] = freq_index(i, nmesh) > 0 ? 2.0 : 1.0;
    return 0;
}

int apk_tables_compensation(int resampler, int interlaced, int nmesh, double *comp_host) {
    APK_REQUIRE(nmesh >= 1 && comp_host, "apk_tables_compensation: bad argument");
    APK_REQUIRE(resampler == APK_CIC || resampler == APK_TSC, "apk_tables_compensation: no window compensation for resampler %d", resampler);
    compensation_axis(resampler, interlaced, nmesh, comp_host);
    return 0;
}

int apk_tables_interlace_phase(int nmesh, double boxsize, double *phase_host) {
    APK_REQUIRE(nmesh >= 1 && boxsize > 0.0 && phase_host, "apk_tables_interlace_phase: bad argument");
    std::vector<double> k((size_t)nmesh);
    k_axis(nmesh, boxsize, APK_F64, k.data());
    for (int i = 0; i < nmesh; ++i) phase_host[i] = 0.5 * k[(size_t)i] * (boxsize / (double)nmesh);
    return 0;
}

int apk_power_scratch_elems(const apk_plan *P, int interlaced, int nfields, int64_t *elems) {
    APK_REQUIRE(P && elems && nfields >= 1 && nfields <= 2, "apk_power_scratch_elems: bad argument");
    *elems = (int64_t)P->n0 * P->N * P->ldz * (interlaced ? 2 : 1) * nfields;
    return 0;
}

int apk_power_from_particles(apk_plan *P, const void *p0, const void *p1, const void *p2, int layout, int pos_dtype,
                             double pos_scale, const void *mass, int mass_dtype, int64_t np, int resampler, int interlaced,
                             int compensated, int normalize, double kmin, double dk, double kmax, float *scratch,
                             double *k_host, double *power_host, int64_t *modes_host, int capacity, int *nbins,
                             double *total_mass, void *stream) {
    APK_REQUIRE(P && scratch && k_host && power_host && modes_host, "apk_power_from_particles: null argument");
    APK_REQUIRE(P->n0 == P->N, "apk_power_from_particles: single-GPU plans only");
    APK_REQUIRE(!compensated || resampler == APK_CIC || resampler == APK_TSC, "apk_power_from_particles: compensation needs CIC or TSC");
    DeviceGuard guard(P->device);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t elems = (size_t)P->N * P->N * P->ldz;
    float *mesh = scratch, *twin = interlaced ? scratch + elems : nullptr;
    int rc = interlaced ? apk_deposit_interlaced(P, p0, p1, p2, layout, pos_dtype, pos_scale, mass, mass_dtype, np, resampler,
                                                 APK_DEPOSIT_AUTO, 1, mesh, twin, stream)
                        : apk_deposit(P, p0, p1, p2, layout, pos_dtype, pos_scale, mass, mass_dtype, np, resampler, 0.0,
                                      APK_DEPOSIT_AUTO, 1, mesh, stream);
    if (rc) return rc;
    double W = 0.0;
    if ((rc = apk_padded_mesh_sum(P, mesh, P->scratch, stream))) return rc;
    APK_CUDA(cudaMemcpyAsync(&W, P->scratch, sizeof(double), cudaMemcpyDeviceToHost, st));
    if ((rc = apk_fft_r2c(P, mesh, stream))) return rc;
    if (twin && (rc = apk_fft_r2c(P, twin, stream))) return rc;
    APK_CUDA(cudaStreamSynchronize(st));
    if (total_mass) *total_mass = W;
    const double N = (double)P->N, L = P->L, cells = N * N * N, dx = L / N;
    const double field = normalize ? cells / W : 1.0 / (dx * dx * dx);            // 1 + delta, or rho = mass / dx^3
    apk_binning *B = nullptr;
    std::vector<double> edges;
    if ((rc = get_binning(P, kmin, dk, kmax, compensated ? resampler : 0, interlaced, APK_F64, &B, &edges))) return rc;
    const double scale = L * L * L * field * field / (cells * cells);
    return finish(P, B, edges, mesh, twin, nullptr, nullptr, scale, k_host, power_host, modes_host, capacity, nbins, st);
}

int apk_power_from_mesh(apk_plan *P, const void *value_map1, const void *value_map2, int dtype, double kmin, double dk,
                        double kmax, float *scratch, double *k_host, double *power_host, int64_t *modes_host, int capacity,
                        int *nbins, void *stream) {
    APK_REQUIRE(P && value_map1 && scratch && k_host && power_host && modes_host, "apk_power_from_mesh: null argument");
    APK_REQUIRE(P->n0 == P->N, "apk_power_from_mesh: single-GPU plans only");
    DeviceGuard guard(P->device);
    cudaStream_t st = (cudaStream_t)stream;
    const size_t elems = (size_t)P->N * P->N * P->ldz;
    const double cells = (double)P->N * P->N * P->N;
    const void *maps[2] = {value_map1, value_map2};
    float *mesh[2] = {scratch, value_map2 ? scratch + elems : nullptr};
    for (int f = 0; f < 2; ++f) {
        if (!maps[f]) continue;
        // the float64 mean only feeds the k = 0 mode, which FFTPower zeroes; removing it keeps the fp32 FFT clean
        double sum = 0.0;
        int rc = apk_mesh_sum(P, maps[f], dtype, P->scratch, stream);
        if (rc) return rc;
        APK_CUDA(cudaMemcpyAsync(&sum, P->scratch, sizeof(double), cudaMemcpyDeviceToHost, st));
        APK_CUDA(cudaStreamSynchronize(st));
        if ((rc = apk_load_mesh(P, maps[f], dtype, sum / cells, mesh[f], stream))) return rc;
        if ((rc = apk_fft_r2c(P, mesh[f], stream))) return rc;
    }
    apk_binning *B = nullptr;
    std::vector<double> edges;
    if (int rc = get_binning(P, kmin, dk, kmax, 0, 0, APK_F64, &B, &edges)) return rc;
    const double L = P->L, scale = L * L * L / (cells * cells);
    return finish(P, B, edges, mesh[0], nullptr, mesh[1], nullptr, scale, k_host, power_host, modes_host, capacity, nbins, st);
}

}  // extern "C"
