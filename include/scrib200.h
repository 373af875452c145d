/*
 * scrib200.h - C ABI of libscrib200.so, the sm_100a implementation of scri's data-parallel
 * waveform-transformation hot path (reference: moble/scri 2024.0.13).
 *
 * The reference is pure Python + numba and has no FFI of its own; the boundary below mirrors the
 * numba / third-party kernel signatures the reference crosses on this path (SURVEY.md 8b), one entry
 * point per kernel, so that a maintainer can bind them with ctypes in place of those calls
 * (see INTEGRATION.md for the stubs).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; caller owns all buffers
 *   - complex128 = interleaved double[2]; arrays are C-contiguous (row-major), 16-byte aligned
 *   - (ell,m) mode layout: index = ell(ell+1) - ell_min^2 + m        (scri/waveform_modes.py:455)
 *   - grid layout: index = j*n_phi + k, theta_j = pi j/(n_theta-1), phi_k = 2 pi k/n_phi
 *                                                                    (scri/waveform_grid.py:130-135,594)
 *   - `stream` is a cudaStream_t passed as void*; kernels are enqueued asynchronously on it
 *   - return value: 0 = ok, negative = error (message via scrib200_last_error()); no hidden
 *     allocation - scratch comes from the *_workspace_bytes queries
 */
#ifndef SCRIB200_H
#define SCRIB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SCRIB200_OK 0
#define SCRIB200_EINVAL (-1)
#define SCRIB200_ECUDA (-2)

int scrib200_version(void);
const char* scrib200_last_error(void);
/* number of kernels launched by this library since load (bench.py's gpu_launches) */
int64_t scrib200_launch_count(void);

/* ---------------------------------------------------------------------------------------------
 * Wigner-D rotation of modes, in place.
 * Replaces  scri/rotations.py:370-392 `_rotate_decomposition_basis_by_series(data, R_basis, ell_min,
 * ell_max, D)` (+ the per-step sf._Wigner_D_matrices call) and, with spinor_stride = 0,
 * rotations.py:346-367 `_rotate_decomposition_basis_by_constant`.
 *   data    [n_times, n_modes] complex128, n_modes = LM_total_size(ell_min, ell_max)
 *   spinors [n_times, 2] complex128 (Ra = w + i z, Rb = y + i x)  - or a single pair if stride 0
 *   seed    [(2L+1)^2], rec [L, 2L+1, 2L+1, 3]  recurrence tables for L = ell_max
 *           (scri_b200._sf.wigner_tables); uv [L, 2L+1, 2] the factored coefficients
 *           U[l][m] = sqrt((2l+1)(l+1)/((l+1)^2-m^2)), V[l][m] = sqrt((l+1)(l^2-m^2)/(l((l+1)^2-m^2)))
 *           (scri_b200._sf.wigner_factor_table).  ell_max <= 16 with `uv` non-NULL takes the lanes-along-time recurrence
 *           kernel (rec may be NULL; the kernel reads the multiplied-out coefficients a = U U, b, c = V V from a table the
 *           library builds itself from the same formulas, `uv` only selects it); larger ell_max, or uv == NULL, uses `rec`.
 */
int scrib200_rotate_modes(double* data, int64_t n_times, int ell_min, int ell_max, const double* spinors,
                          int64_t spinor_stride, const double* seed, const double* rec, const double* uv, void* stream);

/* The same rotation on the FP64 tensor cores (ell_max <= 16): D^l(R) = phases * Delta^l * phases(beta) * Delta^l^T * phases
 * with the constant real matrices Delta^l = d^l(pi/2), so that the 16 time steps of a tile and one l are two small DMMA
 * products and three diagonal multiplications (scri_b200/csrc/rotate.cu).  Replaces the same reference loop as
 * scrib200_rotate_modes (scri/rotations.py:346-392, one sf.Wigner_D_matrices call per time step there).
 *   frags: DEVICE table of m8n8k4 A fragments from scri_b200/ops.py:wigner_delta_fragments - for every l = 0 .. ell_max the
 *          tiles [Kt][Mt][32] of Delta^l^T followed by those of Delta^l (Mt = ceil((2l+1)/8), Kt = ceil((2l+1)/4), zero padded);
 *   frag_offsets_host: HOST int[ell_max + 1], start of l's tiles in `frags` (in doubles).
 * A time step whose rotor is a pure z rotation (Rb == 0 exactly) is finished by its diagonal: the identity is bit-exact. */
int scrib200_rotate_modes_dmma(double* data, int64_t n_times, int ell_min, int ell_max, const double* spinors,
                               int64_t spinor_stride, const double* frags, const int* frag_offsets_host, void* stream);

/* ---------------------------------------------------------------------------------------------
 * SWSH synthesis with the BMS epilogue.
 * Replaces  scri/waveform_grid.py:475-484 (np.tensordot of the modes with sf.SWSH_grid), the constant
 * data-type correction :486-503 and the conformal factor :559:
 *     F[i, g] = (sum_lm a[i, lm] Y[g, lm] - c[g]) * k[g]^w
 * as one real FP64 tensor-core (DMMA) GEMM  [n_times, 2 n_modes] x [2 n_modes, 2 G].
 *   modes   [n_times, n_modes] complex128
 *   Bmat    [Kpad, Ncpad] real: packed table (scri_b200.plan.pack_synthesis_matrix);
 *           Kpad = roundup(2 n_modes, 16), Ncpad = roundup(2 G, 64)
 *   offset  [Ncpad] real (Re c, Im c interleaved), scale [Ncpad] real (k^w repeated twice)
 *   F       [n_times, G] complex128 (output)
 */
int scrib200_swsh_synthesize(const double* modes, int64_t n_times, int n_modes, const double* Bmat, int Kpad,
                             int Ncpad, const double* offset, const double* scale, int G, double* F, void* stream);

/* The same synthesis by the three-multiplication complex product (T1 = a_r Y_r, T2 = a_i Y_i, T3 = (a_r + a_i)(Y_r + Y_i);
 * Re = T1 - T2, Im = T3 - T1 - T2): 6 n G flops per time step instead of 8 n G on the FP64 tensor cores.
 *   scrib200_swsh_pack3m: packed table Bmat [Kpad, Ncpad] of scrib200_swsh_synthesize -> B3 [3, npad, Gpad] real planes
 *   Y_r, Y_i, Y_r + Y_i (npad multiple of 8 >= n_modes, Gpad multiple of 32 >= G, zero padded).
 *   scrib200_swsh_synthesize_3m: modes [n_times, n_modes] complex128, offset / scale [>= 2 G] as above, F [n_times, G].
 * Replaces the same reference lines (scri/waveform_grid.py:475-503,559). */
int scrib200_swsh_pack3m(const double* Bmat, int Kpad, int Ncpad, int n_modes, int G, double* B3, int npad, int Gpad, void* stream);
int scrib200_swsh_synthesize_3m(const double* modes, int64_t n_times, int n_modes, const double* B3, int npad, int Gpad,
                                const double* offset, const double* scale, int G, double* F, void* stream);

/* ---------------------------------------------------------------------------------------------
 * BMS retarded-time remap: batched not-a-knot cubic-spline construction + evaluation.
 * Replaces  scri/waveform_grid.py:564-588: the output time grid u' = (1/gamma)(t - time_translation) restricted
 * to [max_g k(t_0-alpha), min_g k(t_{N-1}-alpha)], and two scipy InterpolatedUnivariateSpline builds per grid point
 * evaluated at u':  for each g: knots x_i = k[g]*(t[i]-alpha[g]), values F[i,g] (Re and Im),
 * out[i', g] = spline_g(uprm[i']).
 *
 * scrib200_spline_prepare (once per time axis): the knots of all grid points are affine images of t, so the
 * tridiagonal moment system is factorised once, in t-units:
 *   tab  [n_times, 8]  allocation (16-byte aligned); the first 6 n_times doubles hold (P, Q, Phi, c', W, Psi) per row, rows
 *                      contiguous - consumed by scrib200_spline_remap / scrib200_spline_calculus (one bulk copy per tile)
 *   uprm [n_times]     u'_i = gamma_factor * (t_i - time_translation) (divide = 0, gamma_factor = 1/gamma: the
 *                      WaveformGrid arithmetic) or (t_i - time_translation) / gamma_factor (divide = 1, gamma_factor =
 *                      gamma: scri/asymptotic_bondi_data/transformations.py:393); may be NULL together with kconf/alpha
 *   info [8] (device)  [0] lo, [1] hi: the retained block is uprm[lo:hi];  [2], [3]: worst decay of the spline
 *                      recurrences over any 32 / 64 consecutive rows (choose halo = 32 if [2] <= 1e-15, else 64 if
 *                      [3] <= 1e-15, else 128);  [4], [5]: u'min, u'max;  [6]: the smallest sample spacing min(t[i+1] - t[i])
 *
 * scrib200_spline_remap: t [n_times], F [n_times, G] complex128, kconf [G], alpha [G], uprm [n_out] increasing,
 *   tile == 0: out [n_out, G] complex128 time-major;  tile = T (power of two >= 2): out written time-tiled,
 *   out[(i'/T)*(G*T) + g*T + i'%T], buffer of ceil(n_out/T)*G*T elements - the layout scrib200_map2salm_tiled reads
 *   (stores are contiguous runs of T samples, each analysis CTA reads one contiguous [G, T] tile).
 *   halo / body: rows of run-in on each side of a tile / intervals per tile, multiples of 16, body + 2 halo <= 384
 *   (0 = defaults 32 / 240).
 *   n_series >= 1: a batch of series sharing t, kconf, alpha and uprm: F is [n_series, n_times, G] and the outputs of
 *   series b are rows b*n_out .. (b+1)*n_out-1 of `out` (time-major) or of the time-tiled index space (tile = T).
 *   workspace: scrib200_spline_remap_workspace_bytes() - one int per (tile, grid point): the first output of each
 *   tile, and one flag per (tile, group of 8 grid points): tiles no output time falls in are skipped, so a call on a
 *   slice of u' costs its share of the sweep.  A CTA keeps its tile of F in shared memory; F is read once.
 */
size_t scrib200_spline_remap_workspace_bytes(int64_t n_times, int G, int halo, int body);
int scrib200_spline_prepare(const double* t, int64_t n_times, double gamma_factor, int divide, double time_translation,
                            const double* kconf, const double* alpha, int G, double* tab, double* uprm, double* info,
                            void* stream);
int scrib200_spline_remap(const double* t, int64_t n_times, const double* F, int G, const double* kconf,
                          const double* alpha, const double* tab, const double* uprm, int64_t n_out, double* out,
                          int tile, int halo, int body, int n_series, void* workspace, size_t workspace_bytes,
                          void* stream);
/* The same, for a caller that evaluates a slice of the output times and knows that no grid point needs input samples outside
 * rows [row_lo, row_hi) for it (a slab of the end-to-end pipeline): only the tiles holding those rows are launched. */
int scrib200_spline_remap_rows(const double* t, int64_t n_times, const double* F, int G, const double* kconf,
                               const double* alpha, const double* tab, const double* uprm, int64_t n_out, double* out,
                               int tile, int halo, int body, int n_series, int64_t row_lo, int64_t row_hi, void* workspace,
                               size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * SWSH analysis, batched over time steps.
 * Replaces  scri/waveform_grid.py:303-307 (spinsfast.map2salm per time step, first ell_min^2 modes
 * dropped): phi-DFT followed by the Clenshaw-Curtis theta quadrature that Huffenberger & Wandelt's
 * algorithm reduces to.
 *   grid [n_times, n_theta, n_phi] complex128
 *   E    [n_phi, 2 ell_max + 1] complex128, Wt [n_modes, n_theta] real (scri_b200._sf.analysis_tables)
 *   out  [n_times, n_modes] complex128, n_modes = LM_total_size(ell_min, ell_max)
 */
size_t scrib200_map2salm_workspace_bytes(int64_t n_times, int n_theta, int n_phi, int ell_max);
int scrib200_map2salm(const double* grid, int64_t n_times, int n_theta, int n_phi, const double* E,
                      const double* Wt, int ell_min, int ell_max, double* out, void* workspace,
                      size_t workspace_bytes, void* stream);

/* Same analysis on a time-tiled grid (output of scrib200_spline_remap with the same `tile`).
 *   trig [n_phi, ell_max+1] complex128 = (cos, sin)(m phi_k)/n_phi  (scri_b200.plan: from the E table)
 * scrib200_map2salm_tile_size returns the tile to use (8, 4 or 2) or 0 when the tables do not fit one CTA;
 * callers then use the time-major pair scrib200_spline_remap(tile=0) / scrib200_map2salm. */
int scrib200_map2salm_tile_size(int n_theta, int n_phi, int ell_min, int ell_max);
int scrib200_map2salm_tiled(const double* gridT, int tile, int64_t n_times, int n_theta, int n_phi, const double* trig,
                            const double* Wt, int ell_min, int ell_max, double* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Time calculus of every mode through the not-a-knot cubic spline.
 * Replaces  scri/waveform_base.py:689-703  CubicSpline(t, data).derivative(k)(t)  (data_dot, data_ddot; order = 1, 2)
 * and .antiderivative(k)(t) (data_int, data_iint; order = -1, -2: exact integrals of the piecewise cubic, zero at t[0]).
 *   data/out [n_times, ncol] complex128; tab from scrib200_spline_prepare(t); halo/body as in scrib200_spline_remap;
 *   aux [n_times, ncol] complex128: needed for order -2 only (receives the first antiderivative), else may be NULL.
 */
int scrib200_spline_calculus(const double* t, int64_t n_times, const double* data, int ncol, const double* tab,
                             int order, double* out, double* aux, int halo, int body, void* stream);

/* sum_modes |a|^2 per time step.  Replaces scri/waveform_base.py:19-35 complex_array_norm. */
int scrib200_norm(const double* data, int64_t n_times, int n_modes, double* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Time-domain inner products: spline definite integrals over time of products of mode series (scri_b200/csrc/inner.cu).
 * The not-a-knot spline integral of samples f_i is sum_i w_i f_i; the caller computes the weights w [n_times] on the host
 * once per (t, t1, t2) (scri_b200/ops.py:spline_integral_weights) and passes them as a DEVICE array.
 *
 * scrib200_inner_product replaces the integral of scri/mode_calculations.py:493-534 `inner_product` (quaternion.calculus.
 * spline_definite_integral of abar * b, conj(abar) * b with apply_conjugate) and of scri/waveform_modes.py:574-656
 * `WaveformModes.inner_product` (sum over modes of conj(a) b, then the same integral):
 *   a, b    complex128 rows of pitch lda / ldb complex elements; the operands are columns [a_col0, a_col0 + n_cols) and
 *           [b_col0, b_col0 + n_cols) of them (an ell-clipped view needs no copy)
 *   n_batch independent products, operand z at a + z a_batch_stride (complex elements; 0 broadcasts one operand)
 *   conjugate: f(a) = conj(a) (1) or a (0)
 *   per_column = 0: out [n_batch] complex128, out[z] = sum_i w_i sum_c f(a_ic) b_ic
 *   per_column = 1: out [n_batch, n_cols] complex128, out[z, c] = sum_i w_i f(a_ic) b_ic
 *   workspace: scrib200_inner_product_workspace_bytes(n_times, n_cols, n_batch).  Fixed-order reduction, no atomics.
 *
 * scrib200_inner_product_matrix: G[p, q] = sum_i w_i sum_m conj(A[p, i, m]) B[q, i, m], the WaveformModes.inner_product of
 * every pair of two waveform batches (no reference counterpart: the reference computes one pair per call).
 *   A [P, n_times, n_cols], B [Q, n_times, n_cols] complex128, waveform p at A + p a_stride (complex elements, rows
 *   contiguous); G [P, Q] complex128; workspace: scrib200_inner_product_matrix_workspace_bytes(P, Q, n_times, n_cols).
 *   P == 1 or Q == 1 runs the streaming kernel of scrib200_inner_product; otherwise the FP64 tensor-core (DMMA) GEMM with
 *   K = n_times n_cols split across CTAs and the splits summed in a fixed order.  n_times n_cols < 2^31. */
size_t scrib200_inner_product_workspace_bytes(int64_t n_times, int n_cols, int n_batch);
int scrib200_inner_product(const double* a, int64_t lda, int a_col0, int64_t a_batch_stride, const double* b, int64_t ldb,
                           int b_col0, int64_t b_batch_stride, int64_t n_times, int n_cols, int n_batch, const double* w,
                           int conjugate, int per_column, double* out, void* workspace, size_t workspace_bytes, void* stream);
size_t scrib200_inner_product_matrix_workspace_bytes(int P, int Q, int64_t n_times, int n_cols);
int scrib200_inner_product_matrix(const double* A, int P, int64_t a_stride, const double* B, int Q, int64_t b_stride,
                                  int64_t n_times, int n_cols, const double* w, double* G, void* workspace,
                                  size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * <LL> matrix and <L d/dt> vector in one pass over the modes.
 * Replaces  scri/mode_calculations.py:209-295 `_LLMatrix(data, lm, LL)` and :14-43
 * `_LdtVector(data, datadot, lm, Ldt)`.  datadot/Ldt may both be NULL (LL only).
 *   coef [n_modes, 5]: ladder-coefficient table (scri_b200.mode_calculations.ladder_table)
 *   LL [n_times, 3, 3], Ldt [n_times, 3] real
 */
int scrib200_ll_ldt(const double* data, const double* datadot, int64_t n_times, int n_modes, const double* coef,
                    double* LL, double* Ldt, void* stream);

/* <L> vector.  Replaces scri/mode_calculations.py:60-89 `_LVector(data1, data2, lm, Lvec)`; Lvec [n_times,3] complex */
int scrib200_l_vector(const double* data1, const double* data2, int64_t n_times, int n_modes, const double* coef,
                      double* Lvec, void* stream);

/* <LL>^{ab} between two waveforms, complex [n_times, 3, 3], not symmetrised.
 * Replaces  scri/mode_calculations.py:106-206 `_LLComparisonMatrix(data1, data2, lm, LL)` literally (the reference adds
 * its (y,z) term to element (y,y); so does this). coef as for scrib200_ll_ldt. */
int scrib200_ll_comparison(const double* data1, const double* data2, int64_t n_times, int n_modes, const double* coef,
                           double* LL, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Dominant principal axis of <LL>, made continuous in time.
 * Replaces  np.linalg.eigh(LL)[1][:, :, 2] + scri/mode_calculations.py:316-363
 * `_LLDominantEigenvector(dpa, dpa_i, i_index)`.
 *   LL [n_times,3,3]; rough_direction [3] (device); dpa [n_times,3] output
 */
size_t scrib200_dominant_eigenvector_workspace_bytes(int64_t n_times);
int scrib200_dominant_eigenvector(const double* LL, int64_t n_times, const double* rough_direction,
                                  int64_t rough_index, double* dpa, void* workspace, size_t workspace_bytes,
                                  void* stream);

/* x = scale * A^{-1} b for n 3x3 systems (LU with partial pivoting).
 * Replaces  np.linalg.solve at scri/mode_calculations.py:424 (scale = -1 gives omega). */
int scrib200_solve3(const double* A, const double* b, int64_t n, double scale, double* x, void* stream);

/* ---------------------------------------------------------------------------------------------
 * K sparse expectation values <a|M_k|b>(t) in one pass over the rows.
 * Replaces  scri/flux.py:40-78 `sparse_expectation_value(abar, rows, columns, values, b)` (called once per
 * matrix by the reference).  Elements of matrix k are [seg[k], seg[k+1]); `a` is NOT pre-conjugated.
 *   rows/cols int32 [nnz], vals complex128 [nnz], seg int32 [K+1] (seg_dev on device; seg_host may be NULL)
 *   out [n_times, K] complex128
 */
int scrib200_sparse_expectation(const double* a, const double* b, int64_t n_times, int n_modes, const int* rows,
                                const int* cols, const double* vals, const int* seg_host, const int* seg_dev, int K,
                                double* out, void* stream);
/* The same contraction with the K matrices in column-major ELL form (what scri_b200.ops.sparse_expectation builds from the COO
 * triples of scri/flux.py:182-441): entry w of column c of matrix k at [off_k + w n_modes + c], off_k = n_modes * (widths[0] +
 * ... + widths[k-1]); ell_rows int32 (row index, -1 = no entry), ell_vals double (real_values = 1) or complex128 (0) in the
 * same order; widths HOST int[K] (entries per column, <= 64), K <= 32.  3 loads per non-zero instead of 5. */
int scrib200_sparse_expectation_ell(const double* a, const double* b, int64_t n_times, int n_modes, const int* ell_rows,
                                    const double* ell_vals, const int* widths_host, int K, int real_values, double* out,
                                    void* stream);

/* Time-lane form of the same contraction (the default when the matrices are banded enough for shared memory): a CTA owns
 * 32 time steps (lanes along time), stages the mode rows it needs transposed in shared memory and walks the matrix columns
 * with warp-uniform table reads - scri/flux.py:40-78 (sparse_expectation_value) as called by the flux functions
 * (scri/flux.py:301-441).
 *   entries: DEVICE table [n_modes][K][width] of 16-byte {int32 row, int32 0, double value} (real values) or 32-byte
 *            {int32 row, int32 0, double re, double im, double 0} entries: matrix k's entries of column c, padded to `width`
 *            (1..4) slots by entries of value 0 on a row the column touches anyway; a column without entries in any matrix
 *            has row -1 in all its slots (scri_b200/ops.py:_time_tables);
 *   blocks_host: HOST int[4 * n_blocks] = (c0, c1, rlo, rhi) per column block: columns [c0, c1) touch rows [rlo, rhi) of `a`
 *            only; when a == b the columns of a block must lie inside its row window.  Tiles over 110 KB are refused. */
int scrib200_sparse_expectation_time(const double* a, const double* b, int64_t n_times, int n_modes, const void* entries,
                                     int width, int K, int complex_values, const int* blocks_host, int n_blocks,
                                     double* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Weyl-scalar mixing under a BMS transformation, elementwise over synthesized grids.
 * Replaces  scri/waveform_grid.py:504-550,559 (psi0..psi3 <- higher Weyl scalars times powers of eth u'/k) and the
 * Horner ladders of scri/asymptotic_bondi_data/transformations.py:340-390:
 *   out[i,g] = scale[g] * ( sum_q coef[q] fields[q][i,g] z^q - offset[g] ),   z = (t[i] - alpha[g]) A[g] - C[g]
 *   fields: host array of n_fields (1..5) device pointers, each [n_times, G] complex128 (fields[0] may alias out);
 *   coef [n_fields] (host), alpha/scale [G] real, A/C/offset [G] complex128 (offset may be NULL).
 */
int scrib200_weyl_mix(const double* const* fields, const double* coef, int n_fields, const double* t, int64_t n_times,
                      int G, const double* alpha, const double* A, const double* C, const double* scale,
                      const double* offset, double* out, void* stream);

/* The same mix over a batch of n_series series that share the time axis and the transformation (TransformPlan.run_batch
 * for psi0..psi3, whose companion fields come per waveform): fields[q] and out are [n_series * n_times, G] complex128,
 * the series stacked along time, and row r takes t[r mod n_times].  Every element takes the operations of
 * scrib200_weyl_mix in the same order, so a batch equals its series mixed one at a time, bit for bit.  Any row count
 * launches (64-bit indices; series and slabs of rows stride over the grid); fields[0] may alias out. */
int scrib200_weyl_mix_series(const double* const* fields, const double* coef, int n_fields, const double* t,
                             int64_t n_times, int64_t n_series, int G, const double* alpha, const double* A,
                             const double* C, const double* scale, const double* offset, double* out, void* stream);

/* The packed real operand `Bmat` of scrib200_swsh_synthesize built on the device from the rotor grid:
 * Y[g, (l,m)] = (-1)^s sqrt((2l+1)/4pi) D^l_{m,-s}(R_g) - replaces sf.SWSH_grid(R_j_k, s, ell_max)
 * (scri/waveform_grid.py:470-471) and the host-side packing.
 *   rotors [G, 4] (w, x, y, z) unit quaternions; seed [(2Lt+1)^2], uv [Lt, 2Lt+1, 2]: scri_b200._sf.wigner_tables /
 *   wigner_factor_table for Lt = table_ell_max >= max(ell_max, |spin|); Bmat [Kpad, Ncpad] is zero-filled first. */
int scrib200_swsh_pack(const double* rotors, int G, int spin, int ell_min, int ell_max, const double* seed,
                       const double* uv, int table_ell_max, double* Bmat, int Kpad, int Ncpad, void* stream);

/* out[e] = a[e] * b[e] for n complex128 elements: the pointwise product of ModesTimeSeries.grid_multiply
 * (scri/modes_time_series.py:190). */
int scrib200_grid_product(const double* a, const double* b, double* out, int64_t n, void* stream);

/* Modes of the pointwise product of two spin-weighted mode series on spinsfast's regular grid, fused and separable
 * (the grids are never formed): replaces spinsfast.salm2map x 2, the product and spinsfast.map2salm of
 * ModesTimeSeries.grid_multiply (scri/modes_time_series.py:177-193), and sf.Modes.multiply as bms_charges.py:40-187
 * calls it (the quadrature is exact once the working band limit reaches ell1 + ell2).
 *   a1 [n_times, n1], a2 [n_times, n2] complex128 mode series; out [n_times, (L_out+1)^2] (modes from ell = 0);
 *   perm1/perm2, ctl [n_steps], lamfrag [n_chunks, lam_stride], tiles [n_tiles, 2], wtfrag [n_chunks, wt_stride]:
 *   device tables from scri_b200._product.product_tables (Wigner-d values and quadrature weights per ring, laid out as
 *   DMMA fragments); cfg: HOST int[15] = (ell1, ell2, L_out, n_phi, n_chunks, qmax, szA, offF1, offF2, smem doubles,
 *   warps, max k-steps, M per convolution warp, tiles per warp, 0).  n_ctas <= 0 selects one persistent CTA per SM.  Fails (SCRIB200_EINVAL) when the tables do
 *   not fit one CTA (ell beyond ~35): callers then use scrib200_swsh_synthesize / scrib200_grid_product / scrib200_map2salm. */
size_t scrib200_modes_product_max_shared_bytes(void);
int scrib200_modes_product(const double* a1, int n1, const double* a2, int n2, int64_t n_times, const int* perm1,
                           const int* perm2, const int* ctl, int n_steps, const double* lamfrag, int64_t lam_stride,
                           const int* tiles, int n_tiles, const double* wtfrag, int64_t wt_stride, const int* cfg,
                           double* out, int n_ctas, void* stream);

/* Separable synthesis on spinsfast's regular grid (theta_j = pi j/(n_theta-1), phi_k = 2 pi k/n_phi), theta stage:
 * out[t, j, m + l_max] = sum_l sY_lm(theta_j, 0) modes[t, (l, m)] - the Wigner-d contraction over l with time as the batch
 * dimension (FP64 DMMA).  The phi stage is scrib200_swsh_synthesize over the rows (t, j) with the packed table
 * e^{i m phi_k}: together they replace spinsfast.salm2map(salm, s, lmax, Ntheta, Nphi) (scri/modes_time_series.py:177-182)
 * at ~(l_max+1)/2 times fewer flops than the dense synthesis.
 *   modes [n_times, n_modes]; out [n_times, n_theta, 2 l_max + 1]; perm / ctl / lamfrag / cfg (HOST int[5] = n_theta, 2 l_max+1,
 *   ring chunks, mode-tile doubles, shared-memory doubles) from scri_b200/_product.py:theta_tables. */
int scrib200_theta_synth(const double* modes, int n_modes, int64_t n_times, const int* perm, const int* ctl, int n_ctl,
                         const double* lamfrag, int64_t lam_stride, const int* cfg, double* out, void* stream);

/* Separable analysis on the regular grid, theta stage: out[t, (l, M)] = sum_j W_lM(theta_j) P[t, j, M + l_max], W = 2 pi q_j
 * sY_lM(theta_j, 0) with the Clenshaw-Curtis weights q_j (FP64 DMMA, accumulators in registers over all rings).  P is the
 * phi-DFT of the map, (1/n_phi) sum_k f(theta_j, phi_k) e^{-i M phi_k}, produced by scrib200_swsh_synthesize over the rows
 * (t, j) with the packed table e^{-i M phi_k}/n_phi: together they replace spinsfast.map2salm(map, s, lmax)[ell_min^2:]
 * (scri/waveform_grid.py:303-307, scri/modes_time_series.py:188) for grids beyond the shared-memory tile kernels.
 *   P [n_times, n_theta, 2 l_max + 1]; out [n_times, (l_max+1)^2 - ell_min^2]; tiles [8*21, 2], wtfrag [ring chunks, 8*21*64],
 *   cfg (HOST int[6] = n_theta, 2 l_max+1, ring chunks, n_out, ell_min^2, l_max) from scri_b200/_product.py:quad_tables. */
int scrib200_theta_quad(const double* P, int64_t n_times, const int* tiles, int n_tiles, const double* wtfrag,
                        int64_t wt_stride, const int* cfg, double* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Host -> device copy of a pageable host array through the library's pinned staging ring (worker threads fill
 * chunk i+1 while the copy engine drains chunk i; the number of threads is this process's share of the cores in its CPU
 * affinity mask, divided by LOCAL_WORLD_SIZE, override: SCRIB200_COPY_THREADS).  For a pageable source all of `src_host`
 * has been read on return and the DMAs are ordered on `stream`.  A page-locked source (cudaHostAlloc, or
 * scrib200_host_register) goes up in one asynchronous DMA: it must stay unchanged until `stream` reaches that point.
 * scrib200_host_register / _unregister page-lock and release a caller's array in place (cudaHostRegister): worth it
 * for arrays that are transferred more than once - replaces the reference's host-resident `w.data` as the operand of
 * every transform (scri/waveform_grid.py:475).  scrib200_host_register returns 0 when it page-locked the array (the
 * caller owes a scrib200_host_unregister), 1 when the memory was page-locked already (nothing to undo), < 0 on failure.
 */
int scrib200_h2d(void* dst_device, const void* src_host, size_t nbytes, void* stream);
int scrib200_host_register(const void* host, size_t nbytes);
int scrib200_host_unregister(const void* host);

/* Integer stages of the RPXMB waveform codec (scri/utilities.py:194-407, called from scri/SpEC/file_io/corotating_paired_xor.py and
 * rotating_paired_xor_multishuffle_bzip2.py), bit-exact:
 *   scrib200_xor_timeseries: [n_rows, n_cols] 64-bit words, time along rows.  reverse = 0: out[i] = in[i] ^ in[i-1], row 0 kept
 *   (xor_timeseries; out of place); reverse = 1: the prefix XOR that undoes it (xor_timeseries_reverse; in place allowed), workspace
 *   of scrib200_xor_timeseries_workspace_bytes().
 *   scrib200_fletcher32: acc2 (device, 2 x uint64) receives (c0, c1) of the Fletcher-32 checksum over n_words16 16-bit words, both
 *   already reduced modulo 65535; the checksum is c1 << 16 | c0.
 *   scrib200_multishuffle: `widths` (HOST int[n_widths], bits per piece from the highest significance down, summing to bit_width =
 *   8 / 16 / 32 / 64); forward = 1 shuffles n elements into the bit stream "lowest piece of every element, next piece of every
 *   element, ...", forward = 0 undoes it.  Out of place. */
int scrib200_xor_timeseries(const void* in, void* out, int64_t n_rows, int64_t n_cols, int reverse, void* workspace,
                            size_t workspace_bytes, void* stream);
size_t scrib200_xor_timeseries_workspace_bytes(int64_t n_rows, int64_t n_cols);
int scrib200_fletcher32(const void* data, int64_t n_words16, void* acc2, void* stream);
int scrib200_multishuffle(const void* in, void* out, int64_t n, int bit_width, const int* widths, int n_widths, int forward,
                          void* stream);

/* Floating-point stages of the same codec (scri/waveform_modes.py:457-476, 658-703), in place on modes [n_times, n_modes]
 * complex128, n_modes = (ell_max+1)^2 - ell_min^2:
 *   scrib200_conjugate_pairs: inverse = 0: convert_to_conjugate_pairs, f[l,m] <- (f[l,m] + conj f[l,-m]) / sqrt 2 and
 *   f[l,-m] <- (f[l,m] - conj f[l,-m]) / sqrt 2 for m > 0; inverse = 1: convert_from_conjugate_pairs.  Bit-identical to numpy's
 *   arithmetic (complex division by the real sqrt 2).
 *   scrib200_truncate: WaveformModes.truncate with tol_per_mode = tol / sqrt(n_modes): each row is rounded to a multiple of
 *   2^-floor(-log2(|row| tol_per_mode)) (round half to even).  n_complex = complex numbers per row. */
int scrib200_conjugate_pairs(void* data, int64_t n_times, int ell_min, int ell_max, int inverse, void* stream);
int scrib200_truncate(void* data, int64_t n_times, int n_complex, double tol_per_mode, void* stream);

/* HOST function (no device work, all pointers are host memory): rotor series with dR/dt = omega(t) R / 2, R(t[0]) = R0, on
 * the samples t - replaces quaternion.integrate_angular_velocity((t, omega), t0, t1, R0, tolerance) as
 * scri/mode_calculations.py:467 calls it.  Dormand-Prince 8(5,3) with the standard step controller (error norm < 1 against
 * atol + rtol |y|), steps clipped to the samples; omega is the cubic spline whose piecewise-polynomial coefficients
 * coef[4][n-1][3] (scipy PPoly layout) the caller provides.  out [n, 4] (w, x, y, z), not normalised; n_rhs (may be NULL)
 * receives the number of right-hand-side evaluations. */
int scrib200_integrate_angular_velocity(const double* t, int64_t n, const double* coef, const double* R0, double atol,
                                        double rtol, double* out, int64_t* n_rhs);

#ifdef __cplusplus
}
#endif
#endif /* SCRIB200_H */
