// Runs the SOURCE of astrild_b200/csrc/tf.cu's kernels on the CPU (tests/simt/simt.h): the sorted deposit's NGP brick
// partition (count -> segment sums -> scan -> scatter, S = 1, from deposit_sorted.cu) followed by the moment tile kernel,
// and the combine kernel with the coefficient tables of apk_tf_create.  Tests only.
// deposit_sorted_kernels.inc and tf_kernels.inc are produced by tests/simt/build_simt_tf.py from the .cu files.
#include "simt.h"
#include "deposit_sorted_kernels.inc"
#include "tf_kernels.inc"

#include <algorithm>
#include <cmath>
#include <vector>

using namespace apk;

namespace {

template <int ORDER, typename PT, bool SOA, bool MASS>
void run(const void *p0, const void *p1, const void *p2, const void *mass, int mass_f64, long long np, int N,
         double pos_scale, int k0, int G, float *meshes, int num_sms) {
    using VT = typename std::conditional<MASS, P4, P3>::type;
    DepositGeom Gm;
    Gm.N = N; Gm.ldz = 2 * (N / 2 + 1); Gm.scale = pos_scale * (double)N; Gm.shift = 0.0;
    Gm.slab = 0; Gm.plane0 = 0; Gm.nplanes = N; Gm.own0 = 0; Gm.nown = N;
    Gm.s0 = (float)Gm.scale;
    Gm.s1 = (float)(Gm.scale - (double)Gm.s0);
    Gm.s2 = (float)(Gm.scale - (double)Gm.s0 - (double)Gm.s1);
    Gm.t32 = 0.5f;
    const BrickGrid B = make_brick_grid(Gm, 1, false);
    std::vector<VT> vals((size_t)np + 1);
    std::vector<unsigned int> counts(B.nbricks + 2, 0u), start(B.nbricks + 2, 0xdeadbeefu), cursor(B.nbricks + 2, 0xdeadbeefu),
        filled(B.nbricks + 2, 0xdeadbeefu);
    const int nseg = (B.nbricks + SCAN_SEG - 1) / SCAN_SEG;
    std::vector<unsigned int> seg_total(nseg + 1, 0xdeadbeefu), seg_filled(nseg + 1, 0xdeadbeefu);
    unsigned int counter[2] = {0u, 0xdeadbeefu};
    const long long tile = (long long)PART_THREADS * PART_ITEMS;
    const int pb = (int)std::min<long long>((np + tile - 1) / tile, (long long)num_sms * 8);
    simt::launch(pb, PART_THREADS, [&] {
        brick_count_kernel<1, PT, SOA>((const PT *)p0, (const PT *)p1, (const PT *)p2, np, Gm, B, counts.data());
    });
    simt::launch(nseg, 1024, [&] { brick_segsum_kernel(counts.data(), B.nbricks, seg_total.data(), seg_filled.data()); });
    simt::launch(nseg, 1024, [&] {
        brick_scan_kernel(counts.data(), B.nbricks, seg_total.data(), seg_filled.data(), start.data(), cursor.data(),
                          filled.data(), counter + 1);
    });
    simt::launch(pb, PART_THREADS, [&] {
        brick_scatter_kernel<1, PT, SOA, MASS, VT>((const PT *)p0, (const PT *)p1, (const PT *)p2, mass, mass_f64, np, Gm,
                                                   B, cursor.data(), vals.data());
    });
    const long long mstride = (long long)N * N * Gm.ldz;
    for (int sub = 0; sub < G; sub += TF_TILE_G) {
        TfTileArgs A;
        A.N = N; A.ldz = Gm.ldz; A.B = B;
        A.k0 = k0 + sub; A.G = std::min(TF_TILE_G, G - sub);
        A.degs = 0u;
        for (int j = 0; j < A.G; ++j)
            A.degs |= (unsigned int)(tf_exp(A.k0 + j, 0) + tf_exp(A.k0 + j, 1) + tf_exp(A.k0 + j, 2)) << (3 * j);
        A.mesh = meshes + sub * mstride; A.mstride = mstride;
        // a few CTAs walk all bricks (the persistent loop), as when the grid is smaller than the number of bricks
        simt::launch(std::min(B.nbricks, 3), TF_TILE_THREADS, [&] {
            tf_moment_tile_kernel<ORDER, MASS, VT>(vals.data(), start.data(), filled.data(), counter + 1, A);
        });
    }
}

template <int ORDER, typename PT, bool SOA>
void dispatch_mass(const void *p0, const void *p1, const void *p2, const void *mass, int mass_f64, long long np, int N,
                   double pos_scale, int k0, int G, float *meshes, int num_sms) {
    if (mass) run<ORDER, PT, SOA, true>(p0, p1, p2, mass, mass_f64, np, N, pos_scale, k0, G, meshes, num_sms);
    else run<ORDER, PT, SOA, false>(p0, p1, p2, mass, mass_f64, np, N, pos_scale, k0, G, meshes, num_sms);
}

template <int ORDER>
void dispatch(const void *p0, const void *p1, const void *p2, int soa, int pos_f64, const void *mass, int mass_f64,
              long long np, int N, double pos_scale, int k0, int G, float *meshes, int num_sms) {
    if (pos_f64) soa ? dispatch_mass<ORDER, double, true>(p0, p1, p2, mass, mass_f64, np, N, pos_scale, k0, G, meshes, num_sms)
                     : dispatch_mass<ORDER, double, false>(p0, p1, p2, mass, mass_f64, np, N, pos_scale, k0, G, meshes, num_sms);
    else soa ? dispatch_mass<ORDER, float, true>(p0, p1, p2, mass, mass_f64, np, N, pos_scale, k0, G, meshes, num_sms)
             : dispatch_mass<ORDER, float, false>(p0, p1, p2, mass, mass_f64, np, N, pos_scale, k0, G, meshes, num_sms);
}

}  // namespace

// moment grids k0 .. k0 + G - 1 of order `order` into G padded meshes float32 [G][N][N][2 (N/2+1)] (accumulated into)
extern "C" int simt_tf_moments(const void *p0, const void *p1, const void *p2, int soa, int pos_f64, const void *mass,
                               int mass_f64, long long np, int N, double pos_scale, int order, int k0, int G,
                               float *meshes, int num_sms) {
    if (np <= 0) return 0;
    switch (order) {
        case 0: dispatch<0>(p0, p1, p2, soa, pos_f64, mass, mass_f64, np, N, pos_scale, k0, G, meshes, num_sms); break;
        case 1: dispatch<1>(p0, p1, p2, soa, pos_f64, mass, mass_f64, np, N, pos_scale, k0, G, meshes, num_sms); break;
        case 2: dispatch<2>(p0, p1, p2, soa, pos_f64, mass, mass_f64, np, N, pos_scale, k0, G, meshes, num_sms); break;
        case 3: dispatch<3>(p0, p1, p2, soa, pos_f64, mass, mass_f64, np, N, pos_scale, k0, G, meshes, num_sms); break;
        default: dispatch<4>(p0, p1, p2, soa, pos_f64, mass, mass_f64, np, N, pos_scale, k0, G, meshes, num_sms); break;
    }
    return 0;
}

// combine of G transformed moments k0 .. k0 + G - 1 (complex64 [G][N][N][N/2+1], padded-mesh stride) into out
extern "C" int simt_tf_combine(const void *mom, int N, int k0, int G, int accumulate, int ctas, void *out) {
    std::vector<float> tw((size_t)(TF_MAX_ORDER + 1) * N);   // as apk_tf_create
    for (int i = 0; i < N; ++i) {
        const int n = 2 * i < N ? i : i - N;
        const double w = (double)n * (2.0 * M_PI / (double)N);
        double v = 1.0;
        for (int a = 0; a <= TF_MAX_ORDER; ++a) { tw[(size_t)a * N + i] = (float)v; v = v * w / (double)(a + 1); }
    }
    TfCombineArgs C;
    C.mom = (const float2 *)mom; C.mstride = (long long)N * N * (N / 2 + 1); C.tw = tw.data();
    C.N = N; C.Nk = N / 2 + 1; C.G = G; C.accumulate = accumulate;
    for (int j = 0; j < G; ++j) { C.ea[j] = tf_exp(k0 + j, 0); C.eb[j] = tf_exp(k0 + j, 1); C.ec[j] = tf_exp(k0 + j, 2); }
    C.out = (float2 *)out;
    simt::launch(ctas, TF_COMBINE_THREADS, [&] { tf_combine_kernel(C); });
    return 0;
}
