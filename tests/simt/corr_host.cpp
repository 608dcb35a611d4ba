// Runs the SOURCE of astrild_b200/csrc/corr.cu's kernels on the CPU (tests/simt/simt.h): the fill with the tables of
// apk_xi_create, and the real-space binning + fold (geometry or data pass, 1-D or (r, mu)).  Tests only.
// corr_kernels.inc is produced by tests/simt/build_simt_corr.py from the .cu (device part).
#include "simt.h"
#include "corr_kernels.inc"

#include <algorithm>
#include <cmath>
#include <vector>

using namespace apk;

// c*: complex64 [N][N][N/2+1] (c1s / c2 / c2s may be NULL); comp, phase: per-axis tables [N] or NULL; out: [N][N][N/2+1]
extern "C" int simt_xi_fill(const void *c1, const void *c1s, const void *c2, const void *c2s, int N, const double *comp,
                            const double *phase, float fac, int ctas, void *out) {
    const int Nk = N / 2 + 1;
    std::vector<float> ic;
    std::vector<float2> ph;
    if (comp) for (int i = 0; i < N; ++i) ic.push_back((float)(1.0 / (comp[i] * comp[i])));
    if (phase) for (int i = 0; i < N; ++i) ph.push_back(make_float2((float)std::cos(phase[i]), (float)std::sin(phase[i])));
    XiFillArgs F;
    F.c1 = (const float2 *)c1; F.c1s = (const float2 *)c1s; F.c2 = (const float2 *)c2; F.c2s = (const float2 *)c2s;
    F.ic_a = F.ic_b = F.ic_z = comp ? ic.data() : nullptr;
    F.ph_a = F.ph_b = F.ph_z = phase ? ph.data() : nullptr;
    F.N = N; F.Nk = Nk; F.fac = fac;
    F.out = (float2 *)out;
    const bool I = c1s != nullptr, C = c2 != nullptr, M = comp != nullptr;
#define GO(a, b, c) simt::launch(ctas, XI_FILL_THREADS, [&] { xi_fill_kernel<a, b, c>(F); })
    if (I) { if (C) { if (M) GO(true, true, true); else GO(true, true, false); }
             else { if (M) GO(true, false, true); else GO(true, false, false); } }
    else { if (C) { if (M) GO(false, true, true); else GO(false, true, false); }
           else { if (M) GO(false, false, true); else GO(false, false, false); } }
#undef GO
    return 0;
}

// grid: float [N][N][2 (N/2+1)]; out: [3][nbins] (geo != 0: rsum, musum, count as u64) or [nell][nbins] (data, times
// 1 / fac); nbins = (nedges + 1) (nmu + 2)
extern "C" int simt_xi_bin(const float *grid, int N, const double *r, const double *edges, int nedges, int nmu,
                           const int *ells, int nell, const double *los, double fac, int geo, int ctas, double *out) {
    const bool mu_path = !(nmu == 1 && nell == 1);
    std::vector<double> r2(N), e2(nedges), mue(nmu + 1);
    for (int i = 0; i < N; ++i) r2[i] = r[i] * r[i];
    for (int i = 0; i < nedges; ++i) e2[i] = edges[i] * edges[i];
    for (int i = 0; i <= nmu; ++i) mue[i] = i == nmu ? 1.0 : (double)i * (1.0 / (double)nmu);
    XiBinArgs A;
    A.grid = grid; A.r = r; A.r2 = r2.data(); A.edges2 = e2.data(); A.muedges = mue.data();
    A.N = N; A.ldz = 2 * (N / 2 + 1); A.nedges = nedges; A.nmu = nmu; A.nell = mu_path ? nell : 1;
    A.lmax = 0;
    for (int i = 0; i < XI_MAXL; ++i) { A.ells[i] = i < nell ? ells[i] : 0; if (i < nell) A.lmax = std::max(A.lmax, ells[i]); }
    for (int n = 0; n < 17; ++n) A.inv_n1[n] = 1.0 / (n + 1);
    for (int d = 0; d < 3; ++d) A.los[d] = los[d];
    A.rmin_f = (float)edges[0]; A.inv_dr_f = (float)(1.0 / (edges[1] - edges[0]));
    A.nbins = (long long)(nedges + 1) * (nmu + 2);
    const int narr = geo ? 3 : A.nell;
    if (!geo && (size_t)A.nell * A.nbins * sizeof(double) > simt::kDynSmem) return 5;
    std::vector<double> copies((size_t)XI_NCOPY * narr * A.nbins, 0.0);
    A.copies = copies.data();
    auto go = [&](auto kern) { simt::launch(ctas, XI_BIN_THREADS, [&] { kern(A); }); };
    if (geo) { if (mu_path) go(xi_bin_kernel<true, true>); else go(xi_bin_kernel<false, true>); }
    else { if (mu_path) go(xi_bin_kernel<true, false>); else go(xi_bin_kernel<false, false>); }
    simt::launch((unsigned)((A.nbins + 255) / 256), 256, [&] {
        xi_fold_kernel(copies.data(), narr, A.nbins, nmu, geo ? 2 : -1, geo ? 1.0 : 1.0 / fac, out);
    });
    return 0;
}
