// Runs the SOURCE of astrild_b200/csrc/bispec.cu's kernels on the CPU (tests/simt/simt.h): the shell fill with the tables
// of apk_bispec_create, and the triple-product reduction + fold over a tiling built as bk_make_tiling builds it (one tile
// group).  Tests only.  bispec_kernels.inc is produced by tests/simt/build_simt_bispec.py from the .cu (device part).
#include "simt.h"
#include "bispec_kernels.inc"

#include <cmath>
#include <vector>

using namespace apk;

// fields: float2 [nbins][N][N][N/2+1] (ind == 0) or double2 (ind != 0), zeroed by the caller
extern "C" int simt_bk_fill(const void *c1, const void *c1s, int N, const double *k, const double *edges, int nedges,
                            const double *comp, const double *phase, int ind, int ctas, void *fields) {
    const int Nk = N / 2 + 1;
    std::vector<double> ka2(N), kz2(Nk), e2(nedges);
    for (int i = 0; i < N; ++i) ka2[i] = k[i] * k[i];
    for (int i = 0; i < Nk; ++i) kz2[i] = k[i] * k[i];
    for (int i = 0; i < nedges; ++i) e2[i] = edges[i] * edges[i];
    std::vector<float> ic;
    std::vector<float2> ph;
    if (comp) for (int i = 0; i < N; ++i) ic.push_back((float)(1.0 / comp[i]));
    if (phase) for (int i = 0; i < N; ++i) ph.push_back(make_float2((float)std::cos(phase[i]), (float)std::sin(phase[i])));
    BkFillArgs F;
    F.c1 = (const float2 *)c1; F.c1s = (const float2 *)c1s;
    F.ka2 = ka2.data(); F.kb2 = ka2.data(); F.kz2 = kz2.data(); F.edges2 = e2.data();
    F.ic_a = F.ic_b = F.ic_z = comp ? ic.data() : nullptr;
    F.ph_a = F.ph_b = F.ph_z = phase ? ph.data() : nullptr;
    F.N = N; F.Nk = Nk; F.nedges = nedges;
    F.field_cplx = (long long)N * N * Nk;
    F.kmin_f = (float)edges[0]; F.inv_dk_f = (float)(1.0 / (edges[1] - edges[0]));
    F.fields = fields;
    const bool inter = c1s != nullptr, cm = comp != nullptr;
#define GO(I, P, C) simt::launch(ctas, BK_FILL_THREADS, [&] { bk_fill_kernel<I, P, C>(F); })
    if (ind) GO(true, false, false);
    else if (inter && cm) GO(false, true, true);
    else if (inter) GO(false, true, false);
    else if (cm) GO(false, false, true);
    else GO(false, false, false);
#undef GO
    return 0;
}

template <typename T>
static int reduce(const T *fields, int N, int nbins, const int *triples, int ntriples, int ctas, double *out) {
    constexpr int TJ = BkTile<T>::TJ, TD = BkTile<T>::TD;
    const int nb = nbins;
    std::vector<int> index((size_t)nb * nb * nb, -1);
    for (int t = 0; t < ntriples; ++t) index[((size_t)triples[3 * t] * nb + triples[3 * t + 1]) * nb + triples[3 * t + 2]] = t;
    std::vector<int4> tiles;
    std::vector<int> slot_of(ntriples, -1);
    for (int i = 0; i < nb; ++i)
        for (int j0 = (i / TJ) * TJ; j0 < nb; j0 += TJ)
            for (int d0 = 0; j0 + d0 < nb; d0 += TD) {
                bool any = false;
                for (int a = 0; a < TJ; ++a)
                    for (int d = 0; d < TD; ++d) {
                        const int j = j0 + a, l = j0 + a + d0 + d;
                        if (j < i || j >= nb || l >= nb) continue;
                        const int t = index[((size_t)i * nb + j) * nb + l];
                        if (t >= 0) { slot_of[t] = (int)tiles.size() * (TJ * TD) + a * TD + d; any = true; }
                    }
                if (any) tiles.push_back(make_int4(i, j0, d0, 0));
            }
    if (tiles.size() > (size_t)BK_MAX_THREADS) return 3;
    for (int s : slot_of) if (s < 0) return 4;
    const int threads = (int)((tiles.size() + 31) / 32 * 32);
    BkReduceArgs A;
    A.fields = fields;
    A.field_elems = (long long)N * N * (2 * (N / 2 + 1));
    A.N = N; A.ldz = 2 * (N / 2 + 1); A.nbins = nb;
    A.row = (nb + TJ + TD + 3) & ~3;
    A.npoints = (long long)N * N * N;
    A.nchunks = (A.npoints + BK_P - 1) / BK_P;
    tiles.resize(BK_MAX_THREADS, make_int4(0, 0, 0, 0));
    A.tiles = tiles.data(); A.ntiles = BK_MAX_THREADS;
    std::vector<double> slots((size_t)ctas * A.ntiles * TJ * TD, std::nan(""));
    A.slots = slots.data();
    if ((size_t)2 * BK_P * A.row * sizeof(T) > simt::kDynSmem) return 5;
    simt::launch(ctas, threads, [&] { bk_reduce_kernel<T>(A); });
    simt::launch((ntriples + 255) / 256, 256, [&] {
        bk_fold_kernel(slots.data(), slot_of.data(), ntriples, ctas, (long long)A.ntiles * (TJ * TD), out);
    });
    return 0;
}

// fields in the padded real layout [nbins][N][N][2 (N/2+1)]; out[t] = sum_x F_i F_j F_l of triples[t]
extern "C" int simt_bk_reduce_f32(const float *fields, int N, int nbins, const int *triples, int ntriples, int ctas, double *out) {
    return reduce<float>(fields, N, nbins, triples, ntriples, ctas, out);
}
extern "C" int simt_bk_reduce_f64(const double *fields, int N, int nbins, const int *triples, int ntriples, int ctas, double *out) {
    return reduce<double>(fields, N, nbins, triples, ntriples, ctas, out);
}
