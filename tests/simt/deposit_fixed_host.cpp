// Runs the SOURCE of astrild_b200/csrc/deposit_sorted.cu's kernels on the CPU (tests/simt/simt.h) with either launch
// sequence of partition_sorted() + run_sorted(), on buffers of exactly the size the library gives them (so that an
// AddressSanitizer build reports any access past them):
//   two-pass:   count -> segment sums -> scan -> scatter -> one tile kernel per mesh;
//   fixed-slot: scatter into `slots` records per brick -> segment sums -> scan -> two-pass scatter (runs only if a brick
//               overflowed) -> one tile kernel per mesh.
// Tests only.  deposit_sorted_kernels.inc is the device part of the .cu (tests/simt/build_simt.py), unchanged.
#include "simt.h"
#include "deposit_sorted_kernels.inc"

#include <algorithm>
#include <cmath>
#include <vector>

using namespace apk;

namespace {

DepositGeom make_geom(int N, double pos_scale, double shift, int resampler, int x0, int n0) {
    DepositGeom G;
    G.N = N; G.ldz = 2 * (N / 2 + 1); G.scale = pos_scale * (double)N; G.shift = shift;
    G.slab = n0 < N; G.plane0 = x0 - 1; G.nplanes = G.slab ? 1 + n0 + 2 : N;
    G.own0 = x0; G.nown = n0;
    G.s0 = (float)G.scale;
    G.s1 = (float)(G.scale - (double)G.s0);
    G.s2 = (float)(G.scale - (double)G.s0 - (double)G.s1);
    G.t32 = -1.f;
    if ((shift == 0.0 || shift == 0.5) && std::fabs(G.scale) < 1e30 && std::fabs(G.scale) > 1e-30)
        G.t32 = (float)shift + (resampler == APK_CIC ? 0.f : 0.5f);
    return G;
}

template <int S, typename PT, bool SOA, bool MASS, bool PAIR>
unsigned int run(const void *p0, const void *p1, const void *p2, const void *mass, int mass_f64, long long np,
                 const DepositGeom &G, float *mesh, float *mesh1, unsigned int slots) {
    using VT = typename std::conditional<MASS, P4, P3>::type;
    const BrickGrid B = make_brick_grid(G, S, PAIR);
    const size_t records = slots ? std::max((size_t)np, (size_t)B.nbricks * slots) : (size_t)np;
    std::vector<VT> vals(records);
    // counts[nbricks] is the fixed-slot partition's overflow word (zeroed with the counts), brick_start has nbricks + 1
    std::vector<unsigned int> counts(B.nbricks + 1, 0u), start(B.nbricks + 1, 0xdeadbeefu), cursor(B.nbricks, 0xdeadbeefu),
        filled(B.nbricks, 0xdeadbeefu);
    const int nseg = (B.nbricks + SCAN_SEG - 1) / SCAN_SEG;
    std::vector<unsigned int> seg_total(nseg, 0xdeadbeefu), seg_filled(nseg, 0xdeadbeefu);
    unsigned int nfilled = 0xdeadbeefu;
    unsigned int *overflow = counts.data() + B.nbricks;

    const long long tile = (long long)PART_THREADS * PART_ITEMS;
    const int pb = (int)std::min<long long>((np + tile - 1) / tile, 2LL * 8);
    if (slots)
        simt::launch(pb, PART_THREADS, [&] {
            brick_scatter_kernel<S, PT, SOA, MASS, VT>((const PT *)p0, (const PT *)p1, (const PT *)p2, mass, mass_f64, np, G,
                                                      B, counts.data(), vals.data(), slots);
        });
    else
        simt::launch(pb, PART_THREADS, [&] {
            brick_count_kernel<S, PT, SOA>((const PT *)p0, (const PT *)p1, (const PT *)p2, np, G, B, counts.data());
        });
    simt::launch(nseg, 1024, [&] { brick_segsum_kernel(counts.data(), B.nbricks, seg_total.data(), seg_filled.data()); });
    simt::launch(nseg, 1024, [&] {
        brick_scan_kernel(counts.data(), B.nbricks, seg_total.data(), seg_filled.data(), start.data(), cursor.data(),
                          filled.data(), &nfilled);
    });
    simt::launch(pb, PART_THREADS, [&] {
        brick_scatter_kernel<S, PT, SOA, MASS, VT>((const PT *)p0, (const PT *)p1, (const PT *)p2, mass, mass_f64, np, G,
                                                  B, cursor.data(), vals.data(), 0u, slots ? overflow : nullptr);
    });
    const unsigned int *fc = slots ? counts.data() : nullptr;
    simt::launch(B.nbricks, TILE_THREADS, [&] {
        brick_tile_kernel<S, MASS, PAIR, 0, VT>(vals.data(), start.data(), filled.data(), &nfilled, G, B, mesh, fc, slots);
    });
    if constexpr (PAIR)
        simt::launch(B.nbricks, TILE_THREADS, [&] {
            brick_tile_kernel<S, MASS, PAIR, 1, VT>(vals.data(), start.data(), filled.data(), &nfilled, G, B, mesh1, fc, slots);
        });
    return slots ? *overflow : 0u;
}

template <int S, typename PT, bool SOA>
unsigned int dispatch(const void *p0, const void *p1, const void *p2, const void *mass, int mass_f64, long long np,
                      const DepositGeom &G, float *mesh, float *mesh1, unsigned int slots) {
    if (mesh1)
        return mass ? run<S, PT, SOA, true, true>(p0, p1, p2, mass, mass_f64, np, G, mesh, mesh1, slots)
                    : run<S, PT, SOA, false, true>(p0, p1, p2, mass, mass_f64, np, G, mesh, mesh1, slots);
    return mass ? run<S, PT, SOA, true, false>(p0, p1, p2, mass, mass_f64, np, G, mesh, nullptr, slots)
                : run<S, PT, SOA, false, false>(p0, p1, p2, mass, mass_f64, np, G, mesh, nullptr, slots);
}

}  // namespace

// resampler: 2 = CIC, 3 = TSC; meshes as in deposit_host.cpp (slab plans: ghost planes 1 below / 2 above).
// slots != 0: the fixed-slot partition with that many records per brick.  Returns its overflow word (0 for the two-pass
// partition).
extern "C" unsigned int simt_deposit_partition(const void *p0, const void *p1, const void *p2, int soa, int pos_f64,
                                               const void *mass, int mass_f64, long long np, int N, double pos_scale,
                                               double shift, int resampler, int x0, int n0, float *mesh, float *mesh1,
                                               unsigned int slots) {
    if (np <= 0) return 0;
    const DepositGeom G = make_geom(N, pos_scale, shift, resampler, x0, n0);
#define APK_SIMT_GO(SS, PT, SOA) dispatch<SS, PT, SOA>(p0, p1, p2, mass, mass_f64, np, G, mesh, mesh1, slots)
    if (resampler == APK_CIC) {
        if (pos_f64) return soa ? APK_SIMT_GO(2, double, true) : APK_SIMT_GO(2, double, false);
        return soa ? APK_SIMT_GO(2, float, true) : APK_SIMT_GO(2, float, false);
    }
    if (pos_f64) return soa ? APK_SIMT_GO(3, double, true) : APK_SIMT_GO(3, double, false);
    return soa ? APK_SIMT_GO(3, float, true) : APK_SIMT_GO(3, float, false);
#undef APK_SIMT_GO
}
