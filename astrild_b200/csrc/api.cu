// extern "C" surface of libastrild_pk.so (declared in include/astrild_pk.h).
#include "apk_common.cuh"
#include <cstdlib>
#include "deposit_common.cuh"
#include <algorithm>
#include <cmath>
#include <cstring>

namespace apk {

static thread_local std::string g_last_error;

void set_error(const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
}

// kernels (other translation units)
int deposit_atomic_launch(const void *, const void *, const void *, int, int, const void *, int, long long,
                          int, const DepositGeom &, float *, int, cudaStream_t);
int deposit_sorted_launch(apk_plan *, const void *, const void *, const void *, int, int, const void *, int,
                          long long, int, const DepositGeom &, float *, float *, cudaStream_t);
size_t deposit_sorted_workspace_bytes(const apk_plan *, long long np, int with_mass, int pair);

int mesh_sum_launch(apk_plan *, const void *, int, double *, cudaStream_t);
int padded_mesh_sum_launch(apk_plan *, const float *, double *, cudaStream_t);
int load_mesh_launch(apk_plan *, const void *, int, double, float *, cudaStream_t);
int store_mesh_launch(apk_plan *, const float *, double, double *, cudaStream_t);
int route_launch(apk_plan *, const void *, const void *, const void *, int, int, double, const void *, int, long long,
                 int, unsigned long long *, long long, void *, void *, cudaStream_t);
int accumulate_launch(apk_plan *, float *, const float *, long long, cudaStream_t);
int transpose_p2p_launch(apk_plan *, const void *, const unsigned long long *, long long, int, cudaStream_t);
int bin_power_launch(apk_binning *, const void *, const void *, const void *, const void *, double *,
                     double *, double *, int64_t *, cudaStream_t);

void forget_plan_binnings(apk_plan *P);

static int make_fft3d(apk_plan *P) {
    if (P->has_fft3d) return 0;
    APK_CUFFT(cufftCreate(&P->fft3d));
    APK_CUFFT(cufftSetAutoAllocation(P->fft3d, 0));
    long long n[3] = {P->N, P->N, P->N};
    size_t ws = 0;
    APK_CUFFT(cufftMakePlanMany64(P->fft3d, 3, n, nullptr, 1, 0, nullptr, 1, 0, CUFFT_R2C, 1, &ws));
    P->fft_ws[0] = (ws + 255) & ~(size_t)255;
    P->fft_work_bytes = P->fft_ws[0] + P->fft_ws[1] + P->fft_ws[2];
    P->has_fft3d = true;
    return 0;
}

static int make_fft2d(apk_plan *P) {
    if (P->has_fft2d) return 0;
    APK_CUFFT(cufftCreate(&P->fft2d));
    APK_CUFFT(cufftSetAutoAllocation(P->fft2d, 0));
    long long n[2] = {P->N, P->N};
    size_t ws = 0;
    APK_CUFFT(cufftMakePlanMany64(P->fft2d, 2, n, nullptr, 1, 0, nullptr, 1, 0, CUFFT_R2C, P->n0, &ws));
    P->fft_ws[1] = (ws + 255) & ~(size_t)255;
    P->fft_work_bytes = P->fft_ws[0] + P->fft_ws[1] + P->fft_ws[2];
    P->has_fft2d = true;
    return 0;
}

static int make_fft1d(apk_plan *P, int ny_local) {
    if (P->has_fft1d && P->fft1d_ny == ny_local) return 0;
    if (P->has_fft1d) { cufftDestroy(P->fft1d); P->has_fft1d = false; }
    APK_CUFFT(cufftCreate(&P->fft1d));
    APK_CUFFT(cufftSetAutoAllocation(P->fft1d, 0));
    long long n[1] = {P->N};
    long long embed[1] = {P->N};
    const long long stride = (long long)ny_local * P->Nk;
    size_t ws = 0;
    APK_CUFFT(cufftMakePlanMany64(P->fft1d, 1, n, embed, stride, 1, embed, stride, 1, CUFFT_C2C, stride, &ws));
    P->fft_ws[2] = (ws + 255) & ~(size_t)255;
    P->fft_work_bytes = P->fft_ws[0] + P->fft_ws[1] + P->fft_ws[2];
    P->has_fft1d = true;
    P->fft1d_ny = ny_local;
    return 0;
}

}  // namespace apk

using namespace apk;

extern "C" {

int apk_version(void) { return APK_VERSION; }
const char *apk_last_error(void) { return g_last_error.c_str(); }

int apk_plan_create(apk_plan **out, int nmesh, double boxsize, int x0, int n0, int device) {
    APK_REQUIRE(out != nullptr, "apk_plan_create: null output");
    APK_REQUIRE(nmesh >= 2 && nmesh <= 8192, "apk_plan_create: nmesh %d out of range [2, 8192]", nmesh);
    APK_REQUIRE(boxsize > 0.0, "apk_plan_create: boxsize must be positive");
    APK_REQUIRE(x0 >= 0 && n0 >= 1 && x0 + n0 <= nmesh, "apk_plan_create: slab [%d, %d) outside [0, %d)", x0, x0 + n0, nmesh);
    int ndev = 0;
    APK_CUDA(cudaGetDeviceCount(&ndev));
    APK_REQUIRE(device >= 0 && device < ndev, "apk_plan_create: device %d not available (%d devices)", device, ndev);
    DeviceGuard guard(device);
    apk_plan *P = new apk_plan();
    P->N = nmesh; P->Nk = nmesh / 2 + 1; P->ldz = 2 * P->Nk; P->L = boxsize;
    P->x0 = x0; P->n0 = n0; P->device = device;
    if (n0 < nmesh) { P->ghost_lo = 1; P->ghost_hi = 2; }
    if (P->ghost_lo + P->n0 + P->ghost_hi > nmesh) {
        delete P;
        set_error("apk_plan_create: slab of %d planes plus 3 ghost planes exceeds nmesh %d", n0, nmesh);
        return 2;
    }
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) P->num_sms = prop.multiProcessorCount;
    if (cudaMalloc(&P->scratch, 64 * sizeof(double)) != cudaSuccess) {
        delete P;
        set_error("apk_plan_create: cudaMalloc of plan scratch failed");
        return 1;
    }
    int rc = (n0 == nmesh) ? make_fft3d(P) : make_fft2d(P);
    if (rc) { apk_plan_destroy(P); return rc; }
    *out = P;
    return 0;
}

int apk_plan_destroy(apk_plan *P) {
    if (!P) return 0;
    DeviceGuard guard(P->device);
    forget_plan_binnings(P);                     // binning objects made by apk_power_from_*
    if (P->has_fft3d) cufftDestroy(P->fft3d);
    if (P->has_fft2d) cufftDestroy(P->fft2d);
    if (P->has_fft1d) cufftDestroy(P->fft1d);
    if (P->scratch) cudaFree(P->scratch);
    if (P->ev_ready) for (auto &e : P->ev) cudaEventDestroy(e);
    if (P->ovf_event) cudaEventDestroy(P->ovf_event);
    if (P->ovf_host) cudaFreeHost(P->ovf_host);
    delete P;
    return 0;
}

int apk_plan_mesh_elems(const apk_plan *P, int64_t *elems) {
    APK_REQUIRE(P && elems, "apk_plan_mesh_elems: null argument");
    *elems = (int64_t)P->n0 * P->N * P->ldz;
    return 0;
}

int apk_plan_ghost_planes(const apk_plan *P, int *n_lo, int *n_hi) {
    APK_REQUIRE(P && n_lo && n_hi, "apk_plan_ghost_planes: null argument");
    *n_lo = P->ghost_lo; *n_hi = P->ghost_hi;
    return 0;
}

int apk_plan_workspace_bytes(const apk_plan *P, int64_t max_particles, int with_mass, int interlaced, size_t *bytes) {
    APK_REQUIRE(P && bytes, "apk_plan_workspace_bytes: null argument");
    size_t dep = deposit_sorted_workspace_bytes(P, max_particles, with_mass, interlaced);
    // the cuFFT work areas sit at the END of the workspace, one per plan, disjoint from the deposit's region at
    // its start: a transform may run on another stream while a deposit is in flight
    *bytes = ((dep + 255) & ~(size_t)255) + P->fft_work_bytes + 512;
    return 0;
}

int apk_plan_set_workspace(apk_plan *P, void *workspace, size_t bytes) {
    APK_REQUIRE(P, "apk_plan_set_workspace: null plan");
    P->workspace = workspace;
    P->workspace_bytes = bytes;
    return 0;
}

static int deposit_impl(apk_plan *P, const void *p0, const void *p1, const void *p2, int layout, int pos_dtype,
                        double pos_scale, const void *mass, int mass_dtype, int64_t np, int resampler,
                        double shift, int method, int zero_first, float *mesh, float *mesh1, void *stream) {
    APK_REQUIRE(P && mesh, "apk_deposit: null plan or mesh");
    APK_REQUIRE(np >= 0, "apk_deposit: negative particle count");
    APK_REQUIRE(np == 0 || p0, "apk_deposit: null positions");
    APK_REQUIRE(layout == APK_AOS || (p1 && p2) || np == 0, "apk_deposit: SoA layout needs three pointers");
    APK_REQUIRE(pos_dtype == APK_F32 || pos_dtype == APK_F64, "apk_deposit: bad position dtype %d", pos_dtype);
    APK_REQUIRE(resampler >= APK_NGP && resampler <= APK_TSC, "apk_deposit: bad resampler %d", resampler);
    DeviceGuard guard(P->device);
    cudaStream_t st = (cudaStream_t)stream;
    auto geom = [&](double sh) {
        DepositGeom G;
        G.N = P->N; G.ldz = P->ldz; G.scale = pos_scale * (double)P->N; G.shift = sh;
        G.slab = P->n0 < P->N; G.plane0 = P->x0 - P->ghost_lo; G.nplanes = P->ghost_lo + P->n0 + P->ghost_hi;
        G.own0 = P->x0; G.nown = P->n0;
        G.s0 = (float)G.scale;
        G.s1 = (float)(G.scale - (double)G.s0);
        G.s2 = (float)(G.scale - (double)G.s0 - (double)G.s1);
        G.t32 = -1.f;
        if ((sh == 0.0 || sh == 0.5) && fabs(G.scale) < 1e30 && fabs(G.scale) > 1e-30)
            G.t32 = (float)sh + (resampler == APK_CIC ? 0.f : 0.5f);
        return G;
    };
    const DepositGeom G = geom(shift);
    const size_t mesh_bytes = sizeof(float) * (size_t)G.nplanes * P->N * P->ldz;
    if (zero_first) {
        APK_CUDA(cudaMemsetAsync(mesh, 0, mesh_bytes, st));
        if (mesh1) APK_CUDA(cudaMemsetAsync(mesh1, 0, mesh_bytes, st));
    }
    if (method == APK_DEPOSIT_AUTO) {
        // the sorted path pays per brick (a tile to clear and to flush): it wins once the bricks are populated --
        // more than ~1 particle per 135 cells (measured with 12 x 6 x 30 bricks: 16 per brick) -- and the set is large
        // enough to amortise its launches
        const double bricks = (double)G.nplanes * P->N * P->N / 2160.0;
        method = (np >= (1 << 18) && (double)np >= 16.0 * bricks) ? APK_DEPOSIT_SORTED : APK_DEPOSIT_ATOMIC;
    }
    if (P->timing) P->dep_timed = false;            // an untimed call leaves the last timed deposit's events alone
    if (method == APK_DEPOSIT_SORTED && resampler != APK_NGP && np > 0)
        return deposit_sorted_launch(P, p0, p1, p2, layout, pos_dtype, mass, mass_dtype, np, resampler, G, mesh, mesh1, st);
    if (P->mark(3, st)) { set_error("apk_deposit: event record failed"); return 1; }
    int rc = deposit_atomic_launch(p0, p1, p2, layout, pos_dtype, mass, mass_dtype, np, resampler, G, mesh, P->num_sms, st);
    if (rc) return rc;
    if (mesh1) {
        if (P->first_mesh_event) APK_CUDA(cudaEventRecord(P->first_mesh_event, st));
        rc = deposit_atomic_launch(p0, p1, p2, layout, pos_dtype, mass, mass_dtype, np, resampler, geom(shift + 0.5), mesh1, P->num_sms, st);
        if (rc) return rc;
    }
    if (P->mark(4, st)) { set_error("apk_deposit: event record failed"); return 1; }
    if (P->timing) { P->dep_timed = true; P->dep_sorted = false; }
    return 0;
}

int apk_deposit(apk_plan *P, const void *p0, const void *p1, const void *p2, int layout, int pos_dtype,
                double pos_scale, const void *mass, int mass_dtype, int64_t np, int resampler,
                double shift, int method, int zero_first, float *mesh, void *stream) {
    return deposit_impl(P, p0, p1, p2, layout, pos_dtype, pos_scale, mass, mass_dtype, np, resampler, shift, method,
                        zero_first, mesh, nullptr, stream);
}

int apk_deposit_interlaced(apk_plan *P, const void *p0, const void *p1, const void *p2, int layout, int pos_dtype,
                           double pos_scale, const void *mass, int mass_dtype, int64_t np, int resampler,
                           int method, int zero_first, float *mesh, float *mesh_shifted, void *stream) {
    APK_REQUIRE(mesh_shifted, "apk_deposit_interlaced: null shifted mesh");
    return deposit_impl(P, p0, p1, p2, layout, pos_dtype, pos_scale, mass, mass_dtype, np, resampler, 0.0, method,
                        zero_first, mesh, mesh_shifted, stream);
}

int apk_plan_enable_timing(apk_plan *P, int on) {
    APK_REQUIRE(P, "apk_plan_enable_timing: null plan");
    P->timing = on != 0;
    return 0;
}

int apk_plan_last_deposit_ms(apk_plan *P, float ms[4]) {
    APK_REQUIRE(P && ms, "apk_plan_last_deposit_ms: null argument");
    APK_REQUIRE(P->dep_timed, "apk_plan_last_deposit_ms: no timed deposit on this plan (apk_plan_enable_timing)");
    DeviceGuard guard(P->device);
    APK_CUDA(cudaEventSynchronize(P->ev[4]));
    ms[0] = ms[1] = ms[2] = 0.f;
    if (P->dep_sorted && P->dep_fixed) {         // events: 0 scatter 1 scan (+ refiling) 2 = 3 tile kernels 4
        APK_CUDA(cudaEventElapsedTime(&ms[2], P->ev[0], P->ev[1]));
        APK_CUDA(cudaEventElapsedTime(&ms[1], P->ev[1], P->ev[2]));
    } else if (P->dep_sorted) {                  // events: 0 count 1 scan 2 scatter 3 tile kernels 4
        for (int i = 0; i < 3; ++i) APK_CUDA(cudaEventElapsedTime(&ms[i], P->ev[i], P->ev[i + 1]));
    }
    APK_CUDA(cudaEventElapsedTime(&ms[3], P->ev[3], P->ev[4]));
    return 0;
}

int apk_binning_last_ms(apk_binning *B, float ms[2]) {
    APK_REQUIRE(B && ms, "apk_binning_last_ms: null argument");
    APK_REQUIRE(B->timed, "apk_binning_last_ms: no timed apk_bin_power on this binning (apk_plan_enable_timing)");
    DeviceGuard guard(B->plan->device);
    APK_CUDA(cudaEventSynchronize(B->ev[2]));
    APK_CUDA(cudaEventElapsedTime(&ms[0], B->ev[0], B->ev[1]));
    APK_CUDA(cudaEventElapsedTime(&ms[1], B->ev[1], B->ev[2]));
    return 0;
}

int apk_route_particles(apk_plan *P, const void *p0, const void *p1, const void *p2, int layout, int pos_dtype,
                        double pos_scale, const void *mass, int mass_dtype, int64_t np, int nranks,
                        uint64_t *counts_dev, int64_t capacity, void *out_pos, void *out_mass, void *stream) {
    APK_REQUIRE(P && counts_dev && (np == 0 || p0) && (capacity == 0 || out_pos), "apk_route_particles: null argument");
    APK_REQUIRE(layout == APK_AOS || (p1 && p2) || np == 0, "apk_route_particles: SoA layout needs three pointers");
    APK_REQUIRE(pos_dtype == APK_F32 || pos_dtype == APK_F64, "apk_route_particles: bad position dtype %d", pos_dtype);
    APK_REQUIRE(!mass || out_mass, "apk_route_particles: mass given without out_mass");
    DeviceGuard guard(P->device);
    return route_launch(P, p0, p1, p2, layout, pos_dtype, pos_scale, mass, mass_dtype, np, nranks,
                        (unsigned long long *)counts_dev, capacity, out_pos, out_mass, (cudaStream_t)stream);
}

int apk_slab_transpose_p2p(apk_plan *P, const void *grid, const uint64_t *peer_recv_dev, int64_t peer_offset_bytes,
                           int nranks, void *stream) {
    APK_REQUIRE(P && grid && peer_recv_dev, "apk_slab_transpose_p2p: null argument");
    DeviceGuard guard(P->device);
    return transpose_p2p_launch(P, grid, (const unsigned long long *)peer_recv_dev, peer_offset_bytes, nranks, (cudaStream_t)stream);
}

int apk_mesh_accumulate(apk_plan *P, float *dst, const float *src, int64_t n, void *stream) {
    APK_REQUIRE(P && dst && src, "apk_mesh_accumulate: null argument");
    DeviceGuard guard(P->device);
    return accumulate_launch(P, dst, src, n, (cudaStream_t)stream);
}

int apk_mesh_sum(apk_plan *P, const void *value_map, int dtype, double *sum_dev, void *stream) {
    APK_REQUIRE(P && value_map && sum_dev, "apk_mesh_sum: null argument");
    DeviceGuard guard(P->device);
    return mesh_sum_launch(P, value_map, dtype, sum_dev, (cudaStream_t)stream);
}

int apk_padded_mesh_sum(apk_plan *P, const float *mesh, double *sum_dev, void *stream) {
    APK_REQUIRE(P && mesh && sum_dev, "apk_padded_mesh_sum: null argument");
    DeviceGuard guard(P->device);
    return padded_mesh_sum_launch(P, mesh, sum_dev, (cudaStream_t)stream);
}

int apk_load_mesh(apk_plan *P, const void *value_map, int dtype, double mean_subtract, float *mesh, void *stream) {
    APK_REQUIRE(P && value_map && mesh, "apk_load_mesh: null argument");
    APK_REQUIRE(dtype == APK_F32 || dtype == APK_F64, "apk_load_mesh: bad dtype %d", dtype);
    DeviceGuard guard(P->device);
    return load_mesh_launch(P, value_map, dtype, mean_subtract, mesh, (cudaStream_t)stream);
}

int apk_store_mesh(apk_plan *P, const float *mesh, double scale, double *value_map, void *stream) {
    APK_REQUIRE(P && value_map && mesh, "apk_store_mesh: null argument");
    DeviceGuard guard(P->device);
    return store_mesh_launch(P, mesh, scale, value_map, (cudaStream_t)stream);
}

static int check_work(apk_plan *P, const char *who) {
    APK_REQUIRE(P->fft_work_bytes == 0 || (P->workspace && P->workspace_bytes >= P->fft_work_bytes + 256),
                "%s: workspace of %zu bytes needed, %zu set (apk_plan_set_workspace)", who,
                P->fft_work_bytes + 256, P->workspace_bytes);
    return 0;
}

// work area of plan `which` (0: 3-D, 1: batched 2-D, 2: batched 1-D) at the tail of the workspace
static void *fft_work_area(const apk_plan *P, int which) {
    size_t off = (P->workspace_bytes - P->fft_work_bytes) & ~(size_t)255;
    for (int i = 0; i < which; ++i) off += P->fft_ws[i];
    return (char *)P->workspace + off;
}

int apk_fft_r2c(apk_plan *P, float *mesh, void *stream) {
    APK_REQUIRE(P && mesh, "apk_fft_r2c: null argument");
    APK_REQUIRE(P->n0 == P->N, "apk_fft_r2c: slab plans use apk_fft_r2c_2d / apk_fft_c2c_1d");
    DeviceGuard guard(P->device);
    if (int rc = make_fft3d(P)) return rc;
    if (int rc = check_work(P, "apk_fft_r2c")) return rc;
    APK_CUFFT(cufftSetStream(P->fft3d, (cudaStream_t)stream));
    if (P->fft_ws[0]) APK_CUFFT(cufftSetWorkArea(P->fft3d, fft_work_area(P, 0)));
    APK_CUFFT(cufftExecR2C(P->fft3d, mesh, (cufftComplex *)mesh));
    return 0;
}

int apk_fft_r2c_2d(apk_plan *P, float *mesh, void *stream) {
    APK_REQUIRE(P && mesh, "apk_fft_r2c_2d: null argument");
    DeviceGuard guard(P->device);
    if (int rc = make_fft2d(P)) return rc;
    if (int rc = check_work(P, "apk_fft_r2c_2d")) return rc;
    APK_CUFFT(cufftSetStream(P->fft2d, (cudaStream_t)stream));
    if (P->fft_ws[1]) APK_CUFFT(cufftSetWorkArea(P->fft2d, fft_work_area(P, 1)));
    APK_CUFFT(cufftExecR2C(P->fft2d, mesh, (cufftComplex *)mesh));
    return 0;
}

int apk_plan_prepare_fft1d(apk_plan *P, int ny_local) {
    APK_REQUIRE(P && ny_local >= 1, "apk_plan_prepare_fft1d: bad argument");
    DeviceGuard guard(P->device);
    return make_fft1d(P, ny_local);
}

int apk_plan_prepare_fft2d(apk_plan *P) {
    APK_REQUIRE(P, "apk_plan_prepare_fft2d: null plan");
    DeviceGuard guard(P->device);
    return make_fft2d(P);
}

int apk_plan_set_first_mesh_event(apk_plan *P, void *event) {
    APK_REQUIRE(P, "apk_plan_set_first_mesh_event: null plan");
    P->first_mesh_event = (cudaEvent_t)event;
    return 0;
}

int apk_fft_c2c_1d(apk_plan *P, void *grid, int ny_local, void *stream) {
    APK_REQUIRE(P && grid && ny_local >= 1, "apk_fft_c2c_1d: bad argument");
    DeviceGuard guard(P->device);
    if (int rc = make_fft1d(P, ny_local)) return rc;
    if (int rc = check_work(P, "apk_fft_c2c_1d")) return rc;
    APK_CUFFT(cufftSetStream(P->fft1d, (cudaStream_t)stream));
    if (P->fft_ws[2]) APK_CUFFT(cufftSetWorkArea(P->fft1d, fft_work_area(P, 2)));
    APK_CUFFT(cufftExecC2C(P->fft1d, (cufftComplex *)grid, (cufftComplex *)grid, CUFFT_FORWARD));
    return 0;
}

int apk_binning_create(apk_binning **out, apk_plan *P, int n_a, int n_b, int nz, const double *ka,
                       const double *kb, const double *kz, const double *wz, const double *kedges,
                       int nedges, const double *comp_a, const double *comp_b, const double *comp_z,
                       const double *phase_a, const double *phase_b, const double *phase_z, int dc_a, int dc_b) {
    APK_REQUIRE(out && P && ka && kb && kz && wz && kedges, "apk_binning_create: null argument");
    APK_REQUIRE(n_a >= 1 && n_b >= 1 && nz >= 1, "apk_binning_create: empty grid");
    APK_REQUIRE(nedges >= 2 && nedges <= 65536, "apk_binning_create: need 2..65536 edges, got %d", nedges);
    for (int i = 1; i < nedges; ++i)
        APK_REQUIRE(kedges[i] > kedges[i - 1] && kedges[0] >= 0.0, "apk_binning_create: kedges must be non-negative and increasing");
    const bool has_comp = comp_a || comp_b || comp_z;
    const bool has_phase = phase_a || phase_b || phase_z;
    APK_REQUIRE(!has_comp || (comp_a && comp_b && comp_z), "apk_binning_create: give all three compensation tables or none");
    APK_REQUIRE(!has_phase || (phase_a && phase_b && phase_z), "apk_binning_create: give all three phase tables or none");
    DeviceGuard guard(P->device);

    apk_binning *B = new apk_binning();
    B->plan = P; B->n_a = n_a; B->n_b = n_b; B->nz = nz; B->nedges = nedges;
    B->dc_a = dc_a; B->dc_b = dc_b; B->has_comp = has_comp; B->has_phase = has_phase;
    B->kmin_guess = kedges[0];
    B->inv_dk_guess = 1.0 / (kedges[1] - kedges[0]);

    // one host staging buffer -> one device allocation
    const size_t nd = (size_t)n_a + n_b + nz + nedges;           // doubles
    const size_t nf = (size_t)nz + (has_comp ? n_a + n_b + nz : 0);   // floats
    const size_t nc = has_phase ? (size_t)n_a + n_b + nz : 0;    // float2
    const size_t bytes = nd * 8 + nc * 8 + ((nf + 1) & ~(size_t)1) * 4;
    std::vector<unsigned char> host(bytes);
    double *hd = (double *)host.data();
    float2 *hc = (float2 *)(hd + nd);
    float *hf = (float *)(hc + nc);
    size_t o = 0;
    for (int i = 0; i < n_a; ++i) hd[o++] = ka[i] * ka[i];
    for (int i = 0; i < n_b; ++i) hd[o++] = kb[i] * kb[i];
    for (int i = 0; i < nz; ++i) hd[o++] = kz[i] * kz[i];
    for (int i = 0; i < nedges; ++i) hd[o++] = kedges[i] * kedges[i];
    o = 0;
    if (has_phase) {
        const double *src[3] = {phase_a, phase_b, phase_z};
        const int cnt[3] = {n_a, n_b, nz};
        for (int d = 0; d < 3; ++d)
            for (int i = 0; i < cnt[d]; ++i) hc[o++] = make_float2((float)cos(src[d][i]), (float)sin(src[d][i]));
    }
    o = 0;
    for (int i = 0; i < nz; ++i) hf[o++] = (float)wz[i];
    if (has_comp) {
        const double *src[3] = {comp_a, comp_b, comp_z};
        const int cnt[3] = {n_a, n_b, nz};
        for (int d = 0; d < 3; ++d)
            for (int i = 0; i < cnt[d]; ++i) hf[o++] = (float)(1.0 / (src[d][i] * src[d][i]));
    }
    if (cudaMalloc(&B->tables, bytes) != cudaSuccess) { delete B; set_error("apk_binning_create: cudaMalloc(%zu) failed", bytes); return 1; }
    if (cudaMemcpy(B->tables, host.data(), bytes, cudaMemcpyHostToDevice) != cudaSuccess) {
        cudaFree(B->tables); delete B; set_error("apk_binning_create: table upload failed"); return 1;
    }
    double *dd = (double *)B->tables;
    B->ka2 = dd; B->kb2 = dd + n_a; B->kz2 = B->kb2 + n_b; B->edges2 = B->kz2 + nz;
    float2 *dc = (float2 *)(dd + nd);
    if (has_phase) { B->ph_a = dc; B->ph_b = dc + n_a; B->ph_z = B->ph_b + n_b; }
    float *df = (float *)(dc + nc);
    B->wz = df;
    if (has_comp) { B->icomp2_a = df + nz; B->icomp2_b = B->icomp2_a + n_a; B->icomp2_z = B->icomp2_b + n_b; }

    // the binning PLAN: shell of every mode (uint16), mode counts and sum(w k) per shell are functions of the geometry
    // alone; they are computed on the device by the first apk_bin_power of this object (same float64 digitize) and the
    // data passes then read the table instead of redoing float64 wavenumber arithmetic.  APK_BIN_TABLE=0: one-pass kernel.
    B->use_table = nedges < 65534;
    if (const char *v = getenv("APK_BIN_TABLE")) B->use_table = B->use_table && v[0] != '0';
    B->partial_ctas = P->num_sms * 3;   // = resident CTAs (80 regs, 51 KB smem)
    const size_t pbytes = sizeof(double) * 4 * (size_t)B->partial_ctas * (nedges + 1);
    if (cudaMalloc(&B->partial, pbytes) != cudaSuccess) {
        cudaFree(B->tables); delete B; set_error("apk_binning_create: cudaMalloc(%zu) failed", pbytes); return 1;
    }
    *out = B;
    return 0;
}

int apk_binning_destroy(apk_binning *B) {
    if (!B) return 0;
    DeviceGuard guard(B->plan->device);
    if (B->tables) cudaFree(B->tables);
    if (B->partial) cudaFree(B->partial);
    if (B->bins) cudaFree(B->bins);
    if (B->geo) cudaFree(B->geo);
    if (B->ev_ready) for (auto &e : B->ev) cudaEventDestroy(e);
    delete B;
    return 0;
}

int apk_bin_power(apk_binning *B, const void *c1, const void *c1s, const void *c2, const void *c2s,
                  double *ksum, double *psum_re, double *psum_im, int64_t *nmodes, void *stream) {
    APK_REQUIRE(B && c1 && ksum && psum_re && psum_im && nmodes, "apk_bin_power: null argument");
    DeviceGuard guard(B->plan->device);
    return bin_power_launch(B, c1, c1s, c2, c2s, ksum, psum_re, psum_im, nmodes, (cudaStream_t)stream);
}

}  // extern "C"
