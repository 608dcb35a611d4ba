// Shared declarations of libastrild_pk.so (see include/astrild_pk.h for the ABI).
#pragma once
#include <cuda_runtime.h>
#include <cufft.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>
#include <string>
#include <vector>
#include "astrild_pk.h"

namespace apk {

void set_error(const char *fmt, ...);

#define APK_CUDA(expr)                                                                        \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            apk::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return 1;                                                                         \
        }                                                                                     \
    } while (0)

#define APK_CUFFT(expr)                                                                       \
    do {                                                                                      \
        cufftResult _e = (expr);                                                              \
        if (_e != CUFFT_SUCCESS) {                                                            \
            apk::set_error("%s:%d: %s -> cufft error %d", __FILE__, __LINE__, #expr, (int)_e); \
            return 1;                                                                         \
        }                                                                                     \
    } while (0)

#define APK_REQUIRE(cond, ...)                                                                \
    do {                                                                                      \
        if (!(cond)) {                                                                        \
            apk::set_error(__VA_ARGS__);                                                      \
            return 2;                                                                         \
        }                                                                                     \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { cudaGetDevice(&prev); if (prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

constexpr int kNumSMsFallback = 148;

}  // namespace apk

struct apk_plan {
    int N = 0;          // cells per side
    int Nk = 0;         // N/2+1
    int ldz = 0;        // padded floats per z-row = 2*Nk
    double L = 0.0;
    int x0 = 0, n0 = 0; // owned slab of planes along axis 0
    int ghost_lo = 0, ghost_hi = 0;
    int device = 0;
    int num_sms = apk::kNumSMsFallback;
    cufftHandle fft3d = 0;     bool has_fft3d = false;
    cufftHandle fft2d = 0;     bool has_fft2d = false;
    cufftHandle fft1d = 0;     bool has_fft1d = false;   int fft1d_ny = 0;
    size_t fft_work_bytes = 0;  // sum of fft_ws
    size_t fft_ws[3] = {0, 0, 0};   // cuFFT work areas (3-D, 2-D, 1-D plan), 256-byte multiples, at the tail of the workspace
    cudaEvent_t first_mesh_event = nullptr;   // apk_plan_set_first_mesh_event
    void *workspace = nullptr;
    size_t workspace_bytes = 0;
    double *scratch = nullptr;   // small device scratch for reductions (plan-owned)
    bool timing = false;
    cudaEvent_t ev[6] = {};      // deposit: 0..4, created on first use
    bool ev_ready = false;
    bool dep_timed = false;      // events of the last deposit are valid
    bool dep_sorted = false;
    bool dep_fixed = false;      // ... and it partitioned in the fixed-slot layout (no count pass)
    // fixed-slot partition (deposit_sorted.cu): its overflow word, copied to pinned host memory behind ovf_event and
    // read only once that event has completed; ovf_seen: a brick overflowed, partition in two passes from then on
    unsigned int *ovf_host = nullptr;
    cudaEvent_t ovf_event = nullptr;
    bool ovf_pending = false, ovf_seen = false;

    int mark(int i, cudaStream_t st) {
        if (!timing) return 0;
        if (!ev_ready) {
            for (auto &e : ev) if (cudaEventCreate(&e) != cudaSuccess) return 1;
            ev_ready = true;
        }
        return cudaEventRecord(ev[i], st) != cudaSuccess;
    }
};

struct apk_binning {
    apk_plan *plan = nullptr;
    int n_a = 0, n_b = 0, nz = 0, nedges = 0;
    int dc_a = -1, dc_b = -1;
    bool has_comp = false, has_phase = false;
    // device tables (one allocation)
    void *tables = nullptr;
    double *ka2 = nullptr, *kb2 = nullptr, *kz2 = nullptr, *edges2 = nullptr;
    float *wz = nullptr;
    float *icomp2_a = nullptr, *icomp2_b = nullptr, *icomp2_z = nullptr;   // 1 / comp^2
    float2 *ph_a = nullptr, *ph_b = nullptr, *ph_z = nullptr;              // exp(i phase)
    double kmin_guess = 0.0, inv_dk_guess = 0.0;   // uniform-edge guess for the bin search
    // table-driven binning (default; APK_BIN_TABLE=0 disables): shell of every mode, and [ksum | - | - | nmodes] of the geometry pass
    bool use_table = false;
    unsigned short *bins = nullptr;
    double *geo = nullptr;
    // per-CTA private partial histograms (plan-lifetime allocation)
    double *partial = nullptr;
    int partial_ctas = 0;
    cudaEvent_t ev[3] = {};
    bool ev_ready = false, timed = false;
};
