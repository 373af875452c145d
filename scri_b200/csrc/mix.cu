// K10: Weyl-scalar mixing under a BMS transformation (elementwise over the synthesized grid).
//
// Replaces scri/waveform_grid.py:504-550, 559 (psi0..psi3 pick up the higher Weyl scalars multiplied by powers of the
// time-dependent factor  z = eth u' / k = (t - alpha) gamma k eth(v.r) - eth alpha) and the Horner ladders of
// scri/asymptotic_bondi_data/transformations.py:340-390 (z = (eth k / k)(u - alpha) - eth alpha).  Both are
//     out[i, g] = scale[g] * ( c_0 F_0[i,g] + c_1 F_1[i,g] z + ... + c_Q F_Q[i,g] z^Q - offset[g] ),
//     z[i, g]   = (t[i] - alpha[g]) * A[g] - C[g]                                    (complex A, C; Q <= 4)
// evaluated by Horner's rule from the highest field.  HBM-bound: (Q+1) reads + 1 write of 16 bytes per element; one
// thread owns one grid point (its constants stay in registers) and walks a slab of time steps, lanes along g.
// weyl_mix_series_kernel (scrib200_weyl_mix_series) does the same over a batch of series that share the time axis, row r
// taking t[r mod n_times]: the batched, graph-captured and time-sharded transforms of psi0..psi3 (TransformPlan.run_batch,
// capture, parallel.sharded_transform) mix through it, and so does TransformPlan.run with n_series = 1.
#include "common.cuh"

namespace scrib200 {

struct MixFields {
    const double2* F[5];
    double c[5];
};

// One element of the mix, called by both kernels.  Every rounding is spelled out (fma, __dmul_rn, __dsub_rn), so that
// neither nvcc nor ptxas is free to contract a product into an FMA differently in the two kernels: a batch mixed by
// weyl_mix_series_kernel equals its series mixed one at a time by weyl_mix_kernel, bit for bit.  (The same expression
// written as `dt * a.x - c.x` and `cmul(acc, z)` was contracted one way inline in weyl_mix_kernel and another way once
// moved into a shared function.)  The contractions are those nvcc chose for the original inline body of weyl_mix_kernel:
//     z = fma(a, dt, -c),   acc z = (fma(z.x, acc.x, -(z.y acc.y)), fma(z.x, acc.y, z.y acc.x)),
// and, for a single field, out = scale fma(c_0, F_0, -offset).
__device__ __forceinline__ double2 weyl_mix_element(const MixFields& f, int nq, int64_t e, double ti, double al, double2 a,
                                                    double2 c, double sc, double2 off) {
    const double2 top = f.F[nq - 1][e];
    if (nq == 1) return make_double2(__dmul_rn(sc, fma(f.c[0], top.x, -off.x)), __dmul_rn(sc, fma(f.c[0], top.y, -off.y)));
    const double dt = __dsub_rn(ti, al);
    const double2 z = make_double2(fma(a.x, dt, -c.x), fma(a.y, dt, -c.y));
    double2 acc = make_double2(__dmul_rn(f.c[nq - 1], top.x), __dmul_rn(f.c[nq - 1], top.y));
    for (int q = nq - 2; q >= 0; --q) {
        acc = make_double2(fma(z.x, acc.x, -__dmul_rn(z.y, acc.y)), fma(z.x, acc.y, __dmul_rn(z.y, acc.x)));
        const double2 v = f.F[q][e];
        acc.x = fma(f.c[q], v.x, acc.x);
        acc.y = fma(f.c[q], v.y, acc.y);
    }
    return make_double2(__dmul_rn(sc, __dsub_rn(acc.x, off.x)), __dmul_rn(sc, __dsub_rn(acc.y, off.y)));
}

__global__ void __launch_bounds__(128)
weyl_mix_kernel(MixFields f, int nq, const double* __restrict__ t, int64_t N, int G, const double* __restrict__ alpha,
                const double2* __restrict__ A, const double2* __restrict__ C, const double* __restrict__ scale,
                const double2* __restrict__ offset, double2* __restrict__ out, int rows_per_cta) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    const double al = alpha[g], sc = scale[g];
    const double2 a = A[g], c = C[g];
    const double2 off = offset ? offset[g] : make_double2(0.0, 0.0);
    const int64_t i0 = (int64_t)blockIdx.y * rows_per_cta;
    const int64_t i1 = (i0 + rows_per_cta < N) ? i0 + rows_per_cta : N;
    for (int64_t i = i0; i < i1; ++i) {
        const int64_t e = i * G + g;
        out[e] = weyl_mix_element(f, nq, e, t[i], al, a, c, sc, off);
    }
}

// Slab k of series s covers rows s * n_times + [k * rows_per_cta, (k + 1) * rows_per_cta) and reads t from row k * rows_per_cta
// on.  Slabs stride over gridDim.y and series over gridDim.z (each capped at 65535), so any row count launches.  `out` may
// alias field 0: every element is read and written by the same thread, reads first.
__global__ void __launch_bounds__(128)
weyl_mix_series_kernel(MixFields f, int nq, const double* __restrict__ t, int64_t n_times, int64_t n_series, int G,
                       const double* __restrict__ alpha, const double2* __restrict__ A, const double2* __restrict__ C,
                       const double* __restrict__ scale, const double2* __restrict__ offset, double2* out, int rows_per_cta) {
    const int g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= G) return;
    const double al = alpha[g], sc = scale[g];
    const double2 a = A[g], c = C[g];
    const double2 off = offset ? offset[g] : make_double2(0.0, 0.0);
    const int64_t n_slabs = (n_times + rows_per_cta - 1) / rows_per_cta;
    for (int64_t s = blockIdx.z; s < n_series; s += gridDim.z) {
        for (int64_t k = blockIdx.y; k < n_slabs; k += gridDim.y) {
            const int64_t i0 = k * rows_per_cta;
            const int64_t i1 = (i0 + rows_per_cta < n_times) ? i0 + rows_per_cta : n_times;
            for (int64_t i = i0; i < i1; ++i) {
                const int64_t e = (s * n_times + i) * G + g;
                out[e] = weyl_mix_element(f, nq, e, t[i], al, a, c, sc, off);
            }
        }
    }
}

// out[e] = a[e] * b[e] (complex), the pointwise product of ModesTimeSeries.grid_multiply (modes_time_series.py:190).
__global__ void __launch_bounds__(256)
grid_product_kernel(const double2* __restrict__ a, const double2* __restrict__ b, double2* __restrict__ out, int64_t n) {
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x)
        out[e] = cmul(a[e], b[e]);
}

}  // namespace scrib200

extern "C" int scrib200_grid_product(const double* a, const double* b, double* out, int64_t n, void* stream) {
    using namespace scrib200;
    SCRIB200_REQUIRE(a && b && out, "grid_product: null pointer");
    SCRIB200_REQUIRE(aligned16(a) && aligned16(b) && aligned16(out), "grid_product: pointers must be 16-byte aligned");
    if (n <= 0) return SCRIB200_OK;
    int64_t blocks = (n + 255) / 256;
    if (blocks > 148 * 16) blocks = 148 * 16;
    grid_product_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        reinterpret_cast<const double2*>(a), reinterpret_cast<const double2*>(b), reinterpret_cast<double2*>(out), n);
    SCRIB200_CHECK_LAUNCH("grid_product");
    return SCRIB200_OK;
}

extern "C" int scrib200_weyl_mix(const double* const* fields, const double* coef, int n_fields, const double* t,
                                 int64_t n_times, int G, const double* alpha, const double* A, const double* C,
                                 const double* scale, const double* offset, double* out, void* stream) {
    using namespace scrib200;
    SCRIB200_REQUIRE(fields && coef && t && alpha && A && C && scale && out, "weyl_mix: null pointer");
    SCRIB200_REQUIRE(n_fields >= 1 && n_fields <= 5, "weyl_mix: n_fields=%d must be 1..5", n_fields);
    SCRIB200_REQUIRE(G > 0, "weyl_mix: G=%d", G);
    if (n_times <= 0) return SCRIB200_OK;
    MixFields f;
    for (int q = 0; q < 5; ++q) {
        f.F[q] = (q < n_fields) ? reinterpret_cast<const double2*>(fields[q]) : nullptr;
        f.c[q] = (q < n_fields) ? coef[q] : 0.0;
        SCRIB200_REQUIRE(q >= n_fields || (fields[q] && aligned16(fields[q])), "weyl_mix: field %d is null or misaligned", q);
    }
    SCRIB200_REQUIRE(aligned16(A) && aligned16(C) && aligned16(out) && aligned16(offset), "weyl_mix: pointers must be 16-byte aligned");
    const int rows = 64;
    dim3 grid((G + 127) / 128, (unsigned)((n_times + rows - 1) / rows));
    SCRIB200_REQUIRE(grid.y <= 65535u * 16u, "weyl_mix: series too long");
    weyl_mix_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(
        f, n_fields, t, n_times, G, alpha, reinterpret_cast<const double2*>(A), reinterpret_cast<const double2*>(C), scale,
        reinterpret_cast<const double2*>(offset), reinterpret_cast<double2*>(out), rows);
    SCRIB200_CHECK_LAUNCH("weyl_mix");
    return SCRIB200_OK;
}

extern "C" int scrib200_weyl_mix_series(const double* const* fields, const double* coef, int n_fields, const double* t,
                                        int64_t n_times, int64_t n_series, int G, const double* alpha, const double* A,
                                        const double* C, const double* scale, const double* offset, double* out, void* stream) {
    using namespace scrib200;
    SCRIB200_REQUIRE(fields && coef && t && alpha && A && C && scale && out, "weyl_mix_series: null pointer");
    SCRIB200_REQUIRE(n_fields >= 1 && n_fields <= 5, "weyl_mix_series: n_fields=%d must be 1..5", n_fields);
    SCRIB200_REQUIRE(G > 0, "weyl_mix_series: G=%d", G);
    SCRIB200_REQUIRE(n_times >= 0 && n_series >= 0, "weyl_mix_series: n_times=%lld n_series=%lld", (long long)n_times,
                     (long long)n_series);
    if (n_times == 0 || n_series == 0) return SCRIB200_OK;
    SCRIB200_REQUIRE(n_times <= INT64_MAX / n_series / G, "weyl_mix_series: %lld x %lld rows of %d points overflow 64-bit indices",
                     (long long)n_series, (long long)n_times, G);
    MixFields f;
    for (int q = 0; q < 5; ++q) {
        f.F[q] = (q < n_fields) ? reinterpret_cast<const double2*>(fields[q]) : nullptr;
        f.c[q] = (q < n_fields) ? coef[q] : 0.0;
        SCRIB200_REQUIRE(q >= n_fields || (fields[q] && aligned16(fields[q])), "weyl_mix_series: field %d is null or misaligned", q);
    }
    SCRIB200_REQUIRE(aligned16(A) && aligned16(C) && aligned16(out) && aligned16(offset),
                     "weyl_mix_series: pointers must be 16-byte aligned");
    const int rows = 64;
    const int64_t slabs = (n_times + rows - 1) / rows;
    dim3 grid((G + 127) / 128, (unsigned)(slabs < 65535 ? slabs : 65535), (unsigned)(n_series < 65535 ? n_series : 65535));
    weyl_mix_series_kernel<<<grid, 128, 0, (cudaStream_t)stream>>>(
        f, n_fields, t, n_times, n_series, G, alpha, reinterpret_cast<const double2*>(A), reinterpret_cast<const double2*>(C),
        scale, reinterpret_cast<const double2*>(offset), reinterpret_cast<double2*>(out), rows);
    SCRIB200_CHECK_LAUNCH("weyl_mix_series");
    return SCRIB200_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// The packed synthesis operand of scrib200_swsh_synthesize, built on the device from the rotor grid:
//   Y[g, (l, m)] = (-1)^s sqrt((2l+1)/4pi) D^l_{m,-s}(R_g)      (sf.SWSH_grid, scri/waveform_grid.py:470-471)
//   B[2lm, 2g] = Re Y, B[2lm+1, 2g] = -Im Y, B[2lm, 2g+1] = Im Y, B[2lm+1, 2g+1] = Re Y   (lm counted from ell_min).
// One thread per (grid point, m): phases from powers of the spinor components, the real factor advanced in l by the
// three-term recurrence (seed / factored coefficient tables of scri_b200._sf, the same as the rotation kernel's).
namespace scrib200 {

__global__ void __launch_bounds__(128)
swsh_pack_kernel(const double* __restrict__ R, int G, int s, int ell_min, int ell_max, const double* __restrict__ seed,
                 const double2* __restrict__ uv, int Lt, double* __restrict__ B, int Ncpad) {
    const int nm_out = 2 * ell_max + 1;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= G * nm_out) return;
    const int g = idx / nm_out, mp = idx - g * nm_out - ell_max;
    const int m = -s;                                  // column of D
    const int nmt = 2 * Lt + 1;
    const double w = R[4 * g], x = R[4 * g + 1], y = R[4 * g + 2], z = R[4 * g + 3];
    const double2 Ra = make_double2(w, z), Rb = make_double2(y, x);
    const double cosb = (Ra.x * Ra.x + Ra.y * Ra.y) - (Rb.x * Rb.x + Rb.y * Rb.y);
    const int amp = mp < 0 ? -mp : mp, am = m < 0 ? -m : m;
    const int l0 = amp > am ? amp : am;
    if (l0 > ell_max) return;
    auto cpow = [](double2 zz, int k) {               // zz^k for k >= 0, conj(zz)^|k| for k < 0
        if (k < 0) { zz = cconj(zz); k = -k; }
        double2 acc = make_double2(1.0, 0.0);
        for (int i = 0; i < k; ++i) acc = cmul(acc, zz);
        return acc;
    };
    const double2 ph = cmul(cpow(Ra, mp + m), cpow(Rb, m - mp));
    double P = seed[(mp + Lt) * nmt + (m + Lt)], Pm1 = 0.0;
    const double sgn = (s & 1) ? -1.0 : 1.0;
    const double mmp = (double)(m * mp);
    for (int l = l0; l <= ell_max; ++l) {
        if (l >= ell_min) {
            const double f = sgn * sqrt((2.0 * l + 1.0) / (4.0 * 3.14159265358979323846)) * P;
            const double re = f * ph.x, im = f * ph.y;
            const size_t lm = (size_t)(l * (l + 1) - ell_min * ell_min + mp);
            double* b0 = B + (2 * lm) * Ncpad + 2 * g;
            double* b1 = b0 + Ncpad;
            b0[0] = re;
            b0[1] = im;
            b1[0] = -im;
            b1[1] = re;
        }
        if (l < ell_max) {
            const double2 f1 = uv[l * nmt + mp + Lt], f2 = uv[l * nmt + m + Lt];
            const double rl = (l > 0) ? 1.0 / (double)(l * (l + 1)) : 0.0;
            const double Pn = (f1.x * f2.x) * (cosb - mmp * rl) * P - (f1.y * f2.y) * Pm1;
            Pm1 = P;
            P = Pn;
        }
    }
}

}  // namespace scrib200

extern "C" int scrib200_swsh_pack(const double* rotors, int G, int spin, int ell_min, int ell_max, const double* seed,
                                  const double* uv, int table_ell_max, double* Bmat, int Kpad, int Ncpad, void* stream) {
    using namespace scrib200;
    SCRIB200_REQUIRE(rotors && seed && uv && Bmat, "swsh_pack: null pointer");
    SCRIB200_REQUIRE(G > 0 && ell_min >= 0 && ell_max >= ell_min, "swsh_pack: bad sizes G=%d ell=[%d, %d]", G, ell_min, ell_max);
    const int as = spin < 0 ? -spin : spin;
    SCRIB200_REQUIRE(table_ell_max >= ell_max && table_ell_max >= as, "swsh_pack: tables for ell <= %d cannot serve ell_max=%d, |s|=%d",
                     table_ell_max, ell_max, as);
    const int n = ell_max * (ell_max + 2) - ell_min * ell_min + 1;
    SCRIB200_REQUIRE(Kpad >= 2 * n && Ncpad >= 2 * G, "swsh_pack: Bmat [%d, %d] too small for %d modes x %d points", Kpad, Ncpad, n, G);
    SCRIB200_REQUIRE(aligned16(uv), "swsh_pack: uv must be 16-byte aligned");
    cudaError_t e = cudaMemsetAsync(Bmat, 0, (size_t)Kpad * Ncpad * sizeof(double), (cudaStream_t)stream);
    SCRIB200_REQUIRE(e == cudaSuccess, "swsh_pack: %s", cudaGetErrorString(e));
    const int total = G * (2 * ell_max + 1);
    swsh_pack_kernel<<<(total + 127) / 128, 128, 0, (cudaStream_t)stream>>>(rotors, G, spin, ell_min, ell_max, seed,
                                                                             reinterpret_cast<const double2*>(uv), table_ell_max,
                                                                             Bmat, Ncpad);
    SCRIB200_CHECK_LAUNCH("swsh_pack");
    return SCRIB200_OK;
}
