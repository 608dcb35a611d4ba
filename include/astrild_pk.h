/* astrild_pk.h -- C ABI of libastrild_pk.so: the B200 (sm_100a) implementation of astrild's
 * matter/halo power-spectrum hot path (particle->mesh deposit, r2c 3-D FFT, |delta(k)|^2 shell
 * binning with mode counts).
 *
 * astrild has no FFI for this path: it calls pmesh / nbodykit from Python.  Each entry point
 * below names the reference call it replaces (paths relative to /root/reference):
 *
 *   apk_deposit        pm.paint(pos, mass=, resampler=)           src/astrild/particles/hutils/stats_subfind.py:130-131
 *   apk_load_mesh      ArrayMesh(value_map, BoxSize=, ...)         src/astrild/power_spectra/power_spectrum_3d.py:183-188, 197-212
 *   apk_fft_r2c        FFTPower -> mesh.compute('complex') (r2c)  src/astrild/power_spectra/power_spectrum_3d.py:189-195
 *   apk_power_from_particles / apk_power_from_mesh   the two call sites' numerical bodies in one call (see below)
 *   apk_bin_power      FFTPower(mode="1d", kmin=) binning         src/astrild/power_spectra/power_spectrum_3d.py:189-195, 216-222;
 *                                                                  src/astrild/particles/hutils/stats_subfind.py:142-148
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; apk_last_error() gives the
 *     message of the calling thread's last failure.  (The repo's only native precedent,
 *     src/astrild/rays/skys/sky_utils.py:402-435, has no error channel; this one does.)
 *   - all data pointers are DEVICE pointers unless the parameter name ends in _host.
 *   - the caller owns every buffer (particles, meshes, outputs, workspace); a plan owns only
 *     its cuFFT handle and small device tables.  A plan is bound to one device and must not
 *     be used from two host threads at once.
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream).
 *   - a "mesh" is the in-place r2c layout: float[n0][N][2*(N/2+1)], last axis padded; after
 *     apk_fft_r2c the same memory holds complex64[n0][N][N/2+1] (un-normalised cuFFT output;
 *     the 1/N^3 of pmesh's r2c is folded into the scale the host applies to the shell sums).
 *   - there is no CPU fallback anywhere in this library.
 */
#ifndef ASTRILD_PK_H
#define ASTRILD_PK_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define APK_VERSION 100

typedef struct apk_plan apk_plan;
typedef struct apk_binning apk_binning;
typedef struct apk_kmu apk_kmu;

enum { APK_F32 = 0, APK_F64 = 1 };
enum { APK_AOS = 0, APK_SOA = 1 };                     /* (Np,3) array or three (Np,) arrays   */
enum { APK_NGP = 1, APK_CIC = 2, APK_TSC = 3 };        /* = window support, pmesh resamplers   */
enum { APK_DEPOSIT_AUTO = 0, APK_DEPOSIT_ATOMIC = 1, APK_DEPOSIT_SORTED = 2 };

int apk_version(void);
const char *apk_last_error(void);

/* ---- plan: one mesh geometry on one device ------------------------------------------------ */
/* nmesh = N cells per side (pmesh Nmesh=[N]*3), boxsize = L.  n0/x0: this rank's slab of mesh
 * planes along axis 0 (single GPU: x0 = 0, n0 = N).                                           */
int apk_plan_create(apk_plan **plan, int nmesh, double boxsize, int x0, int n0, int device);
int apk_plan_destroy(apk_plan *plan);
/* floats in one local mesh: n0 * N * 2*(N/2+1)                                               */
int apk_plan_mesh_elems(const apk_plan *plan, int64_t *elems);
/* bytes of scratch apk_deposit (sorted path, max_particles; interlaced != 0: apk_deposit_interlaced)
 * and apk_fft_r2c need                                                                         */
int apk_plan_workspace_bytes(const apk_plan *plan, int64_t max_particles, int with_mass, int interlaced,
                             size_t *bytes);   /* deposit region + the cuFFT work areas of the plans made so far */
int apk_plan_set_workspace(apk_plan *plan, void *workspace, size_t bytes);
/* slab plans deposit into n_lo + n0 + n_hi planes (ghosts below/above the owned slab, to be
 * sent to and added by the ring neighbours); single-GPU plans report 0, 0.                    */
int apk_plan_ghost_planes(const apk_plan *plan, int *n_lo, int *n_hi);

/* ---- per-kernel timing (CUDA events recorded inside the library, on the caller's stream) ---- */
/* on != 0: apk_deposit / apk_bin_power bracket their kernels with events.                     */
int apk_plan_enable_timing(apk_plan *plan, int on);
/* last apk_deposit on this plan, ms: [0] brick count pass, [1] segment sums + scan of the counts, [2] brick scatter
 * pass, [3] tile kernel(s) (sorted path; both meshes of an interlaced pair) or the atomic kernel(s).  Synchronises on
 * the last event. */
int apk_plan_last_deposit_ms(apk_plan *plan, float ms[4]);
/* last apk_bin_power on this binning, ms: [0] fused binning kernel, [1] fold of per-CTA copies  */
int apk_binning_last_ms(apk_binning *binning, float ms[2]);

/* ---- deposit (pm.paint) ------------------------------------------------------------------- */
/* Adds mass * W(cell - g) to `mesh` for every particle, g = pos * pos_scale * N + shift (grid
 * units; cell i is centred on g = i), periodic.  pos_scale = 1/L for positions in box-length
 * units of L, 1 for Ramses-style [0,1) coordinates.  layout APK_AOS: p0 -> (Np,3), p1 = p2 = 0;
 * APK_SOA: p0,p1,p2 -> x,y,z.  mass may be NULL (unit mass).  shift = 0.5 paints the
 * interlaced twin.  zero_first != 0 clears the mesh before accumulating.
 * Slab plans (n0 < N): `mesh` has n_lo + n0 + n_hi planes (apk_plan_ghost_planes), plane 0 is
 * global plane x0 - n_lo; particles whose floor(g_x - shift) is outside [x0, x0+n0) are IGNORED
 * (their owner deposits them, see apk_route_particles).
 * Single-GPU plans wrap periodically.                                                        */
int apk_deposit(apk_plan *plan, const void *p0, const void *p1, const void *p2, int layout,
                int pos_dtype, double pos_scale, const void *mass, int mass_dtype, int64_t np,
                int resampler, double shift, int method, int zero_first, float *mesh, void *stream);

/* Both meshes of nbodykit's interlacing (CatalogMesh interlaced=True: a second paint with the
 * particles shifted by half a cell, src/astrild/power_spectra/power_spectrum_3d.py:201,209 ask for
 * it) in one call: `mesh` gets shift 0, `mesh_shifted` shift 0.5.  The sorted path builds ONE brick
 * partition for both (boundary particles are filed twice).  Same arguments as apk_deposit.       */
int apk_deposit_interlaced(apk_plan *plan, const void *p0, const void *p1, const void *p2, int layout,
                           int pos_dtype, double pos_scale, const void *mass, int mass_dtype, int64_t np,
                           int resampler, int method, int zero_first, float *mesh, float *mesh_shifted,
                           void *stream);

/* `event` is a cudaEvent_t (NULL clears it).  While set, apk_deposit_interlaced records it on its stream as soon
 * as the first mesh (shift 0) is complete, so that the caller can start that mesh's ghost exchange and FFT on
 * another stream while the twin is still being deposited.  The cuFFT work areas live at the end of the
 * workspace, disjoint from the deposit's region, for that reason.                                          */
int apk_plan_set_first_mesh_event(apk_plan *plan, void *event);

/* ---- slab routing (multi-GPU) ---------------------------------------------------------------- */
/* Extracts the particles that must LEAVE this rank: destination = owner of the x-slab holding
 * floor(pos_x*pos_scale*N) (N/nranks planes per rank).  Particles that stay are not touched -- a
 * slab plan's apk_deposit ignores particles it does not own, so the caller deposits its original
 * arrays plus whatever it receives.  Leavers are written as AoS (n,3) of the input dtype into
 * out_pos (masses, same dtype, into out_mass when mass != NULL), grouped by destination rank;
 * counts_dev[0..nranks) receives the per-destination counts (uint64, own rank = 0; the array must
 * hold 2*nranks entries, the second half is scratch).  At most `capacity` particles are written:
 * the host compares sum(counts) with capacity and retries with a larger buffer if needed.  One pass
 * over the particles (x only); the leavers are staged in the plan workspace, which must hold
 * capacity * (3 + [mass]) * sizeof(dtype) + 64 bytes.
 * pmesh equivalent: ParticleMesh.decompose + layout.exchange (unused by astrild).               */
int apk_route_particles(apk_plan *plan, const void *p0, const void *p1, const void *p2, int layout,
                        int pos_dtype, double pos_scale, const void *mass, int mass_dtype, int64_t np,
                        int nranks, uint64_t *counts_dev, int64_t capacity, void *out_pos, void *out_mass,
                        void *stream);
/* Fused pack + peer store of the x<->y slab transpose (step 5 of the distributed r2c) over NVLink peer
 * memory: the block (x_local, y in rank s's range) of `grid` (complex64 [n0][N][N/2+1], output of
 * apk_fft_r2c_2d) is written straight into rank s's receive buffer [N][N/nranks][N/2+1] at
 * [x0 + x_local][y_local][z].  peer_recv_dev: DEVICE array of nranks base addresses (uint64) of the ranks'
 * peer-mapped receive buffers (cuMem/IPC-mapped symmetric allocations); peer_offset_bytes is added to
 * each (field offset).  The caller brackets the call with cross-rank barriers.  Replaces pfft's MPI
 * transpose (PFFT_TRANSPOSED_OUT), which astrild never reaches on more than one rank.                */
int apk_slab_transpose_p2p(apk_plan *plan, const void *grid, const uint64_t *peer_recv_dev,
                           int64_t peer_offset_bytes, int nranks, void *stream);
/* dst[i] += src[i], i < n: adds received ghost planes into the owned slab                       */
int apk_mesh_accumulate(apk_plan *plan, float *dst, const float *src, int64_t n, void *stream);

/* ---- ArrayMesh: gridded field -> mesh ------------------------------------------------------ */
/* value_map: contiguous [n0][N][N] of dtype; writes (value - mean_subtract) as f32 into the
 * padded mesh.  apk_mesh_sum gives the f64 sum of a value_map (for the mean).                 */
int apk_mesh_sum(apk_plan *plan, const void *value_map, int dtype, double *sum_dev, void *stream);
int apk_load_mesh(apk_plan *plan, const void *value_map, int dtype, double mean_subtract,
                  float *mesh, void *stream);
/* the reverse: padded f32 mesh -> contiguous [n0][N][N] doubles, times scale (paint().value)  */
int apk_store_mesh(apk_plan *plan, const float *mesh, double scale, double *value_map, void *stream);
/* f64 sum over the N^3 real cells of a padded mesh (Sum mass; nbar for normalisation)         */
int apk_padded_mesh_sum(apk_plan *plan, const float *mesh, double *sum_dev, void *stream);

/* ---- r2c ----------------------------------------------------------------------------------- */
/* in-place, un-normalised, single precision; single-GPU plans only (slab plans run the
 * 2-D + transpose + 1-D stages from the host side, see astrild_b200/distributed.py).          */
int apk_fft_r2c(apk_plan *plan, float *mesh, void *stream);
/* slab stages: batched 2-D r2c over (y,z) of n0 local planes, and batched 1-D c2c along the
 * leading axis of a [N][ny_local][N/2+1] array.                                              */
int apk_fft_r2c_2d(apk_plan *plan, float *mesh, void *stream);
/* creates the 1-D plan for ny_local ahead of time so apk_plan_workspace_bytes accounts for it  */
int apk_plan_prepare_fft1d(apk_plan *plan, int ny_local);
int apk_plan_prepare_fft2d(apk_plan *plan);
int apk_fft_c2c_1d(apk_plan *plan, void *grid, int ny_local, void *stream);

/* ---- binning (FFTPower mode="1d") ---------------------------------------------------------- */
/* The k-grid is complex64 [n_a][n_b][nz] (nz = N/2+1).  k2 = (ka2[ia] + kb2[ib]) + kz2[iz] in
 * float64, tables = squares of the HOST-built per-axis k tables (so the host decides their
 * dtype/expression, SURVEY.md section 0 item 5); bin = numpy.digitize(k2, kedges2).
 * wz[iz] is the Hermitian weight (2 where k_z > 0 else 1).  Optional per-axis tables:
 * comp_* = factor the complex field is DIVIDED by (window compensation), phase_* = radians of
 * the interlacing phase 0.5*k_i*H.  dc_a/dc_b = local indices of the k=0 row (or -1).         */
int apk_binning_create(apk_binning **binning, apk_plan *plan, int n_a, int n_b, int nz,
                       const double *ka_host, const double *kb_host, const double *kz_host,
                       const double *wz_host, const double *kedges_host, int nedges,
                       const double *comp_a_host, const double *comp_b_host, const double *comp_z_host,
                       const double *phase_a_host, const double *phase_b_host, const double *phase_z_host,
                       int dc_a, int dc_b);
int apk_binning_destroy(apk_binning *binning);
/* c1: field 1; c1s: its interlaced twin or NULL; c2/c2s: second field for a cross spectrum or
 * NULL.  Outputs have nedges+1 entries (numpy.digitize indices 0..nedges: under/overflow
 * included) and are OVERWRITTEN: ksum = sum w*sqrt(k2), psum_re = sum w*Re(c1 conj c2),
 * psum_im = sum Im(c1 conj c2) over singular planes only, nmodes = sum w.                     */
int apk_bin_power(apk_binning *binning, const void *c1, const void *c1s, const void *c2,
                  const void *c2s, double *ksum, double *psum_re, double *psum_im,
                  int64_t *nmodes, void *stream);

/* ---- (k, mu) binning and multipoles (SURVEY.md section 8f, N4) ----------------------------------------------- */
/* nbodykit FFTPower(mode="2d", Nmu=, poles=, los=) -> project_to_basis (astrild hints at redshift-space use:
 * README.md:11, src/astrild/particles/hutils/tpcf.py:12-60).  Grid and optional tables as in apk_binning_create, but
 * ka / kb / kz are the SIGNED per-axis wavenumbers (host).  mu = (k . los) / |k|, binned by
 * numpy.digitize(|mu|, linspace(0, 1, nmu + 1)); ells[0] must be 0 (the (k, mu) spectrum is the monopole-weighted sum),
 * further entries are the requested multipoles.                                                                       */
int apk_kmu_create(apk_kmu **kmu, apk_plan *plan, int n_a, int n_b, int nz,
                   const double *ka_host, const double *kb_host, const double *kz_host, const double *wz_host,
                   const double *kedges_host, int nedges, int nmu, const int *ells_host, int nell,
                   const double *los_host /* [3] */,
                   const double *comp_a_host, const double *comp_b_host, const double *comp_z_host,
                   const double *phase_a_host, const double *phase_b_host, const double *phase_z_host,
                   int dc_a, int dc_b);
int apk_kmu_destroy(apk_kmu *kmu);
/* DEVICE outputs, OVERWRITTEN, laid out [nedges + 1][nmu + 2] (numpy.digitize indices; the k under/overflow rows 0 and
 * nedges, which nbodykit slices away, are NOT accumulated and stay zero; mu column 0 is unused, column nmu + 1 = |mu| == 1
 * is ALSO added to column nmu as nbodykit does): xsum = sum w |k|,
 * musum = sum w |mu|, nsum = sum w; ysum_re / ysum_im [nell][nedges + 1][nmu + 2] = sum (2 ell + 1) L_ell(mu) P with the
 * Hermitian doubling rules of project_to_basis.                                                                       */
int apk_kmu_bin(apk_kmu *kmu, const void *c1, const void *c1s, const void *c2, const void *c2s,
                double *xsum, double *musum, double *ysum_re, double *ysum_im, int64_t *nsum, void *stream);

/* ---- bispectrum B(k1, k2, k3) of one field (FFT estimator, exact triangle counts) ------------------------------ */
/* Shells b = 0 .. Nb-1 are the bins of the 1-D binning of the same edges (apk_tables_k_edges(N, L, kmin, dk, kmax);
 * dk <= 0: 2 pi / L; kmax <= 0: (2/3) pi N / L, which keeps every triangle free of aliasing; kmax above pi N / L is
 * refused); the k = 0 mode is in no shell.  Nb is at most 128.  F_b(x) = un-normalised c2r of the k-grid masked to shell
 * b; the triples are i <= j <= l minus those that provably hold no triangle (lo_l >= hi_i + hi_j and
 * hi_i + hi_j + hi_l <= 2 k_Nyquist).  tsum = sum_x F_i F_j F_l, N_tri = (sum_x D_i D_j D_l) / N^3 with D_b the same for
 * c == 1 (ordered (q1, q2, q3), q1 + q2 + q3 = 0 modulo the grid), and B = L^6 s^3 / N^9 * tsum / (N^3 N_tri) for a field
 * scale s as in FFTPower.  resampler (APK_CIC / APK_TSC, 0 = no compensation) and interlaced select the window
 * deconvolution and interlace-combine of apk_bin_power.  Single-GPU plans only.                                      */
typedef struct apk_bispec apk_bispec;
int apk_bispec_create(apk_bispec **bk, apk_plan *plan, double kmin, double dk, double kmax, int k_dtype,
                      int resampler /* 0 = no compensation */, int interlaced);
int apk_bispec_destroy(apk_bispec *bk);
/* the kept triples (i, j, l) as ijl_host[3 t + 0..2]; ijl_host may be NULL to query the number                     */
int apk_bispec_triples(const apk_bispec *bk, int *ijl_host, int capacity, int *ntriples); /* after the skip rule */
int apk_bispec_scratch_bytes(const apk_bispec *bk, size_t *bytes);   /* max(f64 indicator fields, f32 fields) + cuFFT */
/* N_tri per kept triple (DEVICE int64); computed once per object in float64 and cached.  Fails if a count is further
 * than 0.1 from an integer (precision lost); residual_host (may be NULL) receives the largest |T_D / N^3 - N_tri|.
 * Synchronises `stream`.                                                                                            */
int apk_bispec_count(apk_bispec *bk, void *scratch, size_t bytes, int64_t *ntri_dev, double *residual_host, void *stream);
/* tsum_dev (DEVICE float64 per kept triple) = sum_x F_i F_j F_l of the field c1 (complex64 k-grid after apk_fft_r2c) and
 * its interlaced twin c1s (NULL unless created with interlaced != 0)                                                */
int apk_bispec_measure(apk_bispec *bk, const void *c1, const void *c1s, void *scratch, size_t bytes,
                       double *tsum_dev, void *stream);     /* c1 / c1s are read, never modified */
int apk_bispec_last_ms(apk_bispec *bk, float ms[4]);       /* fill, c2r, reduction, fold (plan timing on) */

/* ---- ingest (SURVEY.md section 8f, N1) ------------------------------------------------------------------- */
/* PowerSpectrum3D._read_data's gridder (src/astrild/power_spectra/power_spectrum_3d.py:142-148):
 *   value_map = zeros((N, N, N)); value_map[((N*x).astype(int), (N*y).astype(int), (N*z).astype(int))] = values
 * One value per cell (assignment, not accumulation); the product is formed in the dtype of the coordinate columns and
 * truncated toward zero; a negative index wraps once like NumPy's; a cell hit by several samples keeps the value of the
 * LAST one (highest index).  x, y, z, values: DEVICE arrays of n entries; value_map: DEVICE float64 [N][N][N], cleared by
 * the call; winner_scratch: DEVICE uint32 [N^3]; bad_count_dev: DEVICE uint64 that receives the number of samples whose
 * index lies outside [-N, N) (NumPy raises IndexError for those: the host side does the same).                      */
int apk_assign_grid(apk_plan *plan, const void *x, const void *y, const void *z, int pos_dtype, const void *values,
                    int val_dtype, int64_t n, double *value_map, uint32_t *winner_scratch, uint64_t *bad_count_dev,
                    void *stream);
/* Ecosmog.compress_snapshot's record reader (src/astrild/particles/ecosmog.py:184-230) on the device: raw_dev is the
 * image of an output_poisson file (Fortran unformatted records); pieces_dev is int64 [npieces][3] = (byte offset of a
 * block of float64 values in the image -- 4-byte aligned, record markers are 4 bytes --, first destination element,
 * number of values); every block is copied into out[dst .. dst + count).  The host walks the record headers
 * (astrild_b200/ingest.py) and this kernel moves the data: one CTA per piece.                                     */
int apk_gather_records(const void *raw_dev, const int64_t *pieces_dev, int64_t npieces, double *out, int device,
                       void *stream);

/* ---- binning tables (host side of FFTPower: who decides which float lands on which side of an edge) ---- */
/* The per-axis tables and edges apk_binning_create takes, computed INSIDE the library with the reference stack's
 * expression order (pmesh ParticleMesh k tables: w = n * (2 pi / N), k = w * N / L; nbodykit FFTPower:
 * dk = 2 pi / L, kmax = pi N / L + dk/2, numpy.arange(kmin, kmax, dk); Compensate{CIC,TSC}[Shotnoise]; the interlacing
 * phase 0.5 k H), so that a C / Fortran caller gets bit-identical bins without re-implementing them.
 * Call sites: src/astrild/power_spectra/power_spectrum_3d.py:181-195; src/astrild/particles/hutils/stats_subfind.py:142-148.
 * All outputs are HOST arrays.  k_dtype: APK_F64 (default reading) or APK_F32 (float32 index ramp).
 * dk <= 0: 2 pi / L;  kmax <= 0: pi N / L + dk / 2.                                                                  */
int apk_tables_k_axis(int nmesh, double boxsize, int k_dtype, double *k_host /* [nmesh] */);
int apk_tables_k_edges(int nmesh, double boxsize, double kmin, double dk, double kmax,
                       double *edges_host /* [capacity] or NULL */, int capacity, int *nedges);
int apk_tables_hermitian_weights(int nmesh, double *w_host /* [nmesh/2+1] */);
int apk_tables_compensation(int resampler, int interlaced, int nmesh, double *comp_host /* [nmesh] */);
int apk_tables_interlace_phase(int nmesh, double boxsize, double *phase_host /* [nmesh] */);

/* ---- one call: particles or gridded fields -> (k, P(k), Nmodes) ------------------------------------------- */
/* floats of scratch the two calls below need: mesh_elems * (interlaced ? 2 : 1) * nfields                       */
int apk_power_scratch_elems(const apk_plan *plan, int interlaced, int nfields, int64_t *elems);
/* SubFind.power_spectrum's numerical body (src/astrild/particles/hutils/stats_subfind.py:129-150: paint -> / dx^3 ->
 * ArrayMesh -> FFTPower(mode="1d", kmin=) -> power.real) with nbodykit's CatalogMesh options: deposit (interlaced twin
 * if asked), r2c, fused binning.  normalize = 0 keeps rho = mass / dx^3 (astrild as written), 1 gives 1 + delta.
 * Particle arguments as in apk_deposit (DEVICE pointers); scratch: DEVICE, apk_power_scratch_elems(plan, interlaced, 1)
 * floats; the plan's workspace must be set (apk_plan_workspace_bytes).  k_host / power_host / modes_host: HOST arrays
 * of `capacity` >= nbins entries (nbins = nedges - 1; empty bins give NaN k and power, like nbodykit); total_mass
 * (may be NULL) receives sum(mass).  The shot noise astrild subtracts is 0 (ArrayMesh); V * sum(m^2) / sum(m)^2 is the
 * caller's to subtract if wanted.  Synchronises `stream`.  Single-GPU plans only.                                 */
int apk_power_from_particles(apk_plan *plan, const void *p0, const void *p1, const void *p2, int layout, int pos_dtype,
                             double pos_scale, const void *mass, int mass_dtype, int64_t np, int resampler,
                             int interlaced, int compensated, int normalize, double kmin, double dk, double kmax,
                             float *scratch, double *k_host, double *power_host, int64_t *modes_host, int capacity,
                             int *nbins, double *total_mass, void *stream);
/* PowerSpectrum3D._power_spectrum_3d (src/astrild/power_spectra/power_spectrum_3d.py:164-226): value_map1 (and
 * value_map2 for the cross spectrum Re(c1 conj c2), else NULL): DEVICE, contiguous [N][N][N] of dtype.  ArrayMesh
 * semantics: no window, no interlacing, no normalisation, shot noise 0.  scratch: apk_power_scratch_elems(plan, 0,
 * value_map2 ? 2 : 1) floats.                                                                                      */
int apk_power_from_mesh(apk_plan *plan, const void *value_map1, const void *value_map2, int dtype, double kmin,
                        double dk, double kmax, float *scratch, double *k_host, double *power_host,
                        int64_t *modes_host, int capacity, int *nbins, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* ASTRILD_PK_H */
