// K12: time-domain inner products of mode series.
//
// Replaces scri/mode_calculations.py:493-534 `inner_product(t, abar, b, axis, apply_conjugate)` and the integral of
// scri/waveform_modes.py:574-656 `WaveformModes.inner_product`: a spline definite integral over time of a product of two
// mode series.  The not-a-knot spline integral is linear in the samples, so the caller supplies the weights w [N]
// (scri_b200/ops.py:spline_integral_weights, computed once per (t, t1, t2)) and every integral is a weighted sum:
//
//   scrib200_inner_product          out = sum_i w_i sum_c f(a_ic) b_ic   (per_column = 0), or
//                                   out[c] = sum_i w_i f(a_ic) b_ic      (per_column = 1),  f = conj or identity;
//                                   one streaming pass, 32 bytes read per complex term: HBM-bound.
//   scrib200_inner_product_matrix   G[p,q] = sum_i w_i sum_m conj(A[p,i,m]) B[q,i,m] for waveform batches: a complex GEMM
//                                   with K = N n on the FP64 tensor cores (mma.sync.m8n8k4.f64, SASS DMMA).
//
// Both reduce in fixed order through a workspace (no atomics), so two runs on the same input agree bit for bit.
#include "common.cuh"

namespace scrib200 {

// ------------------------------------------------------------------------------------------------ streaming kernel
// CTA = 8 warps; lane = one complex column of a 32-column tile, warp = one of 8 interleaved row lanes of the CTA's
// contiguous row chunk.  Stage 1 writes one partial sum per (batch, row chunk, column); stage 2 adds the chunks (and,
// for the scalar form, the columns) in a fixed order.
constexpr int IP_COLS = 32;
constexpr int IP_ROWS = 8;
constexpr int IP_THREADS = IP_COLS * IP_ROWS;
constexpr int IP_UNROLL = 4;

struct IpGeom {
    int64_t rows_per_cta;
    int row_ctas, col_tiles;
};

static IpGeom ip_geometry(int64_t N, int n, int n_batch) {
    IpGeom g;
    g.col_tiles = (n + IP_COLS - 1) / IP_COLS;
    const int64_t target = 148 * 8;                                 // ~8 resident CTAs per SM
    const int64_t per = (int64_t)g.col_tiles * n_batch;
    int64_t rc = (target + per - 1) / per;
    const int64_t max_rc = (N + 255) / 256;                          // at least 256 rows (32 per row lane) per CTA
    if (rc > max_rc) rc = max_rc;
    if (rc < 1) rc = 1;
    int64_t rows = (N + rc - 1) / rc;
    rows = (rows + IP_ROWS - 1) / IP_ROWS * IP_ROWS;
    g.rows_per_cta = rows;
    g.row_ctas = (int)((N + rows - 1) / rows);
    return g;
}

template <bool CONJ>
__device__ __forceinline__ void ip_acc(double2& acc, double wi, double2 x, double2 y) {
    double pr, pi;
    if (CONJ) {
        pr = fma(x.x, y.x, x.y * y.y);
        pi = fma(x.x, y.y, -(x.y * y.x));
    } else {
        pr = fma(x.x, y.x, -(x.y * y.y));
        pi = fma(x.x, y.y, x.y * y.x);
    }
    acc.x = fma(wi, pr, acc.x);
    acc.y = fma(wi, pi, acc.y);
}

template <bool CONJ>
__global__ void __launch_bounds__(IP_THREADS)
inner_product_kernel(const double2* __restrict__ a, int64_t lda, int64_t a_bstride, const double2* __restrict__ b,
                     int64_t ldb, int64_t b_bstride, int64_t N, int n, const double* __restrict__ w, int64_t rows_per_cta,
                     double2* __restrict__ partial) {
    __shared__ double2 red[IP_ROWS][IP_COLS];
    const int lane = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int c = blockIdx.y * IP_COLS + lane;
    const int64_t z = blockIdx.z;
    const int64_t i0 = (int64_t)blockIdx.x * rows_per_cta;
    const int64_t i1 = (i0 + rows_per_cta < N) ? i0 + rows_per_cta : N;
    double2 acc = make_double2(0.0, 0.0);
    if (c < n) {
        const double2* pa = a + z * a_bstride + c;
        const double2* pb = b + z * b_bstride + c;
        int64_t i = i0 + ry;
        for (; i + (IP_UNROLL - 1) * IP_ROWS < i1; i += IP_UNROLL * IP_ROWS) {
            double2 x[IP_UNROLL], y[IP_UNROLL];
            double wi[IP_UNROLL];
#pragma unroll
            for (int u = 0; u < IP_UNROLL; ++u) {
                const int64_t r = i + u * IP_ROWS;
                x[u] = __ldcs(pa + r * lda);
                y[u] = __ldcs(pb + r * ldb);
                wi[u] = __ldg(w + r);
            }
#pragma unroll
            for (int u = 0; u < IP_UNROLL; ++u) ip_acc<CONJ>(acc, wi[u], x[u], y[u]);
        }
        for (; i < i1; i += IP_ROWS) ip_acc<CONJ>(acc, __ldg(w + i), __ldcs(pa + i * lda), __ldcs(pb + i * ldb));
    }
    red[ry][lane] = acc;
    __syncthreads();
    if (ry == 0 && c < n) {
        double2 s = red[0][lane];
#pragma unroll
        for (int r = 1; r < IP_ROWS; ++r) s = cadd(s, red[r][lane]);
        partial[(z * gridDim.x + blockIdx.x) * n + c] = s;
    }
}

// out[z, c] = sum over row chunks: lane = column, warp w adds chunks w, w + 8, ...; the 8 warp sums are added in order.
__global__ void __launch_bounds__(IP_THREADS)
inner_product_columns_kernel(const double2* __restrict__ partial, int row_ctas, int n, double2* __restrict__ out) {
    __shared__ double2 red[IP_ROWS][IP_COLS];
    const int lane = threadIdx.x & 31, ry = threadIdx.x >> 5;
    const int c = blockIdx.x * IP_COLS + lane;
    const int64_t z = blockIdx.y;
    double2 s = make_double2(0.0, 0.0);
    if (c < n) {
        const double2* p = partial + z * row_ctas * (int64_t)n + c;
#pragma unroll 4
        for (int r = ry; r < row_ctas; r += IP_ROWS) s = cadd(s, p[(int64_t)r * n]);
    }
    red[ry][lane] = s;
    __syncthreads();
    if (ry == 0 && c < n) {
        double2 t = red[0][lane];
#pragma unroll
        for (int r = 1; r < IP_ROWS; ++r) t = cadd(t, red[r][lane]);
        out[z * n + c] = t;
    }
}

// out[z] = sum over row chunks and columns: thread t adds the partials t, t + 1024, ... of the flat [chunk, column] array,
// then a fixed tree.
constexpr int IP_RED = 1024;
__global__ void __launch_bounds__(IP_RED)
inner_product_scalar_kernel(const double2* __restrict__ partial, int row_ctas, int n, double2* __restrict__ out) {
    __shared__ double2 red[IP_RED];
    const int64_t z = blockIdx.x;
    const int64_t total = (int64_t)row_ctas * n;
    const double2* p = partial + z * total;
    double2 s = make_double2(0.0, 0.0);
#pragma unroll 8
    for (int64_t e = threadIdx.x; e < total; e += IP_RED) s = cadd(s, p[e]);
    red[threadIdx.x] = s;
    __syncthreads();
    for (int h = IP_RED / 2; h > 0; h >>= 1) {
        if ((int)threadIdx.x < h) red[threadIdx.x] = cadd(red[threadIdx.x], red[threadIdx.x + h]);
        __syncthreads();
    }
    if (threadIdx.x == 0) out[z] = red[0];
}

// --------------------------------------------------------------------------------------------------- matrix kernel
// C[p, 2q + {0,1}] = (Re, Im) G[p, q] as ONE real GEMM of length 2K ("four real products" form; the interleaved complex
// memory is the real operand as it stands):  A'[p, 2k + {0,1}] = w_i (Re, Im) A[p, k],  B~[2q] = (Re, Im) B[q, k],
// B~[2q+1] = (Im, -Re) B[q, k], so that  A'.B~[2q] = Re conj(A) B  and  A'.B~[2q+1] = Im conj(A) B.  8 K real flops per
// (p, q); the three-multiplication form would save a quarter of them but needs sums of the operands staged alongside.
// CTA tile 64 rows (p) x 64 real columns (32 q), 4 warps of 32 x 32 = 4 x 4 DMMA tiles; 8 complex k (16 real) per stage,
// register-staged double buffer (the weights are applied between the global load and the shared store).  K is split
// across gridDim.y; each split writes its own partial tile and a second pass adds the splits in order.
constexpr int MM_BM = 64;
constexpr int MM_BN = 64;              // real output columns per CTA
constexpr int MM_KC = 8;               // complex k per stage
constexpr int MM_LD = 2 * MM_KC + 4;   // shared-memory row stride (doubles): conflict-free fragment loads

__device__ __forceinline__ void ip_dmma(double& d0, double& d1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
                 : "+d"(d0), "+d"(d1)
                 : "d"(a), "d"(b));
}

__global__ void __launch_bounds__(128, 4)
inner_product_dmma_kernel(const double2* __restrict__ A, int P, int64_t sa, const double2* __restrict__ B, int Q, int64_t sb,
                          int n, int64_t K, const double* __restrict__ w, int64_t k_per_split, int tiles_m,
                          double* __restrict__ partial) {
    __shared__ __align__(16) double sA[2][MM_BM * MM_LD];
    __shared__ __align__(16) double sB[2][MM_BN * MM_LD];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int wm = warp >> 1, wn = warp & 1;
    const int tm = blockIdx.x % tiles_m, tn = blockIdx.x / tiles_m;
    const int p0 = tm * MM_BM, q0 = tn * (MM_BN / 2);
    const int64_t kb = (int64_t)blockIdx.y * k_per_split;
    const int64_t ke = (kb + k_per_split < K) ? kb + k_per_split : K;
    const int kc = tid & (MM_KC - 1);                 // this thread's k within a stage, the same for all its loads
    const int r0 = tid >> 3;                           // first row it loads; rows r0 + 16 s

    double2 ra[4], rb[2];
    auto load = [&](int64_t k0) {
        const int64_t k = k0 + kc;
        const bool kin = k < ke;
        const double wk = kin ? __ldg(w + (unsigned)k / (unsigned)n) : 0.0;
#pragma unroll
        for (int s = 0; s < 4; ++s) {
            const int p = p0 + r0 + 16 * s;
            double2 v = make_double2(0.0, 0.0);
            if (kin && p < P) v = __ldcs(A + p * sa + k);
            ra[s] = make_double2(wk * v.x, wk * v.y);
        }
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const int q = q0 + r0 + 16 * s;
            rb[s] = (kin && q < Q) ? __ldcs(B + q * sb + k) : make_double2(0.0, 0.0);
        }
    };
    auto store = [&](int buf) {
#pragma unroll
        for (int s = 0; s < 4; ++s) *reinterpret_cast<double2*>(&sA[buf][(r0 + 16 * s) * MM_LD + 2 * kc]) = ra[s];
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            const int r = 2 * (r0 + 16 * s);
            *reinterpret_cast<double2*>(&sB[buf][r * MM_LD + 2 * kc]) = rb[s];
            *reinterpret_cast<double2*>(&sB[buf][(r + 1) * MM_LD + 2 * kc]) = make_double2(rb[s].y, -rb[s].x);
        }
    };

    double acc[4][4][2];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;

    const int64_t n_stages = (ke - kb + MM_KC - 1) / MM_KC;
    load(kb);
    store(0);
    __syncthreads();
    for (int64_t st = 0; st < n_stages; ++st) {
        const int buf = (int)(st & 1);
        if (st + 1 < n_stages) load(kb + (st + 1) * MM_KC);
        const double* a_s = sA[buf] + (wm * 32 + (lane >> 2)) * MM_LD + (lane & 3);
        const double* b_s = sB[buf] + (wn * 32 + (lane >> 2)) * MM_LD + (lane & 3);
#pragma unroll
        for (int ks = 0; ks < 2 * MM_KC / 4; ++ks) {
            double af[4], bf[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) af[i] = a_s[i * 8 * MM_LD + ks * 4];
#pragma unroll
            for (int j = 0; j < 4; ++j) bf[j] = b_s[j * 8 * MM_LD + ks * 4];
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) ip_dmma(acc[i][j][0], acc[i][j][1], af[i], bf[j]);
        }
        if (st + 1 < n_stages) store(buf ^ 1);
        __syncthreads();
    }

    // C fragment: row lane/4, columns 2 (lane%4) + {0, 1} = (Re, Im) of one q
    const int64_t ldc = 2 * (int64_t)Q;
    double* out = partial + (int64_t)blockIdx.y * P * ldc;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int col = tn * MM_BN + wn * 32 + j * 8 + 2 * (lane & 3);
        if (col >= ldc) continue;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int p = p0 + wm * 32 + i * 8 + (lane >> 2);
            if (p < P) *reinterpret_cast<double2*>(out + p * ldc + col) = make_double2(acc[i][j][0], acc[i][j][1]);
        }
    }
}

__global__ void __launch_bounds__(256)
inner_product_splitk_sum_kernel(const double* __restrict__ partial, int splits, int64_t len, double* __restrict__ G) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= len) return;
    double s = partial[e];
    for (int k = 1; k < splits; ++k) s += partial[(int64_t)k * len + e];
    G[e] = s;
}

struct MmGeom {
    int tiles_m, tiles_n, splits;
    int64_t k_per_split;
};

static MmGeom mm_geometry(int P, int Q, int64_t K) {
    MmGeom g;
    g.tiles_m = (P + MM_BM - 1) / MM_BM;
    g.tiles_n = (2 * Q + MM_BN - 1) / MM_BN;
    const int64_t tiles = (int64_t)g.tiles_m * g.tiles_n;
    const int64_t stages = (K + MM_KC - 1) / MM_KC;
    int64_t s = (148 * 8 + tiles - 1) / tiles;        // about two waves of 4 CTAs per SM
    const int64_t max_s = stages / 16 > 1 ? stages / 16 : 1;   // at least 16 stages per split
    if (s > max_s) s = max_s;
    if (s > 4096) s = 4096;
    const int64_t st_per = (stages + s - 1) / s;
    g.k_per_split = st_per * MM_KC;
    g.splits = (int)((K + g.k_per_split - 1) / g.k_per_split);
    return g;
}

}  // namespace scrib200

extern "C" size_t scrib200_inner_product_workspace_bytes(int64_t n_times, int n_cols, int n_batch) {
    using namespace scrib200;
    if (n_times <= 0 || n_cols <= 0 || n_batch <= 0) return 0;
    const IpGeom g = ip_geometry(n_times, n_cols, n_batch);
    return (size_t)n_batch * g.row_ctas * n_cols * sizeof(double2);
}

extern "C" int scrib200_inner_product(const double* a, int64_t lda, int a_col0, int64_t a_batch_stride, const double* b,
                                      int64_t ldb, int b_col0, int64_t b_batch_stride, int64_t n_times, int n_cols,
                                      int n_batch, const double* w, int conjugate, int per_column, double* out,
                                      void* workspace, size_t workspace_bytes, void* stream) {
    using namespace scrib200;
    SCRIB200_REQUIRE(a && b && w && out, "inner_product: null pointer");
    SCRIB200_REQUIRE(n_times >= 1 && n_cols >= 1 && n_batch >= 1 && n_batch <= 65535,
                     "inner_product: bad sizes n_times=%lld n_cols=%d n_batch=%d", (long long)n_times, n_cols, n_batch);
    SCRIB200_REQUIRE(a_col0 >= 0 && b_col0 >= 0 && lda >= a_col0 + n_cols && ldb >= b_col0 + n_cols,
                     "inner_product: column window [%d, %d) / [%d, %d) exceeds the row pitch %lld / %lld", a_col0,
                     a_col0 + n_cols, b_col0, b_col0 + n_cols, (long long)lda, (long long)ldb);
    SCRIB200_REQUIRE(aligned16(a) && aligned16(b) && aligned16(out) && aligned16(workspace),
                     "inner_product: pointers must be 16-byte aligned");
    const IpGeom g = ip_geometry(n_times, n_cols, n_batch);
    const size_t need = (size_t)n_batch * g.row_ctas * n_cols * sizeof(double2);
    SCRIB200_REQUIRE(workspace && workspace_bytes >= need, "inner_product: workspace of %zu bytes, %zu needed", workspace_bytes, need);
    const cudaStream_t s = (cudaStream_t)stream;
    double2* part = reinterpret_cast<double2*>(workspace);
    const double2* pa = reinterpret_cast<const double2*>(a) + a_col0;
    const double2* pb = reinterpret_cast<const double2*>(b) + b_col0;
    const dim3 grid(g.row_ctas, g.col_tiles, n_batch);
    if (conjugate)
        inner_product_kernel<true><<<grid, IP_THREADS, 0, s>>>(pa, lda, a_batch_stride, pb, ldb, b_batch_stride, n_times,
                                                              n_cols, w, g.rows_per_cta, part);
    else
        inner_product_kernel<false><<<grid, IP_THREADS, 0, s>>>(pa, lda, a_batch_stride, pb, ldb, b_batch_stride, n_times,
                                                               n_cols, w, g.rows_per_cta, part);
    SCRIB200_CHECK_LAUNCH("inner_product");
    if (per_column)
        inner_product_columns_kernel<<<dim3(g.col_tiles, n_batch), IP_THREADS, 0, s>>>(part, g.row_ctas, n_cols,
                                                                                    reinterpret_cast<double2*>(out));
    else
        inner_product_scalar_kernel<<<n_batch, IP_RED, 0, s>>>(part, g.row_ctas, n_cols, reinterpret_cast<double2*>(out));
    SCRIB200_CHECK_LAUNCH("inner_product_reduce");
    return SCRIB200_OK;
}

extern "C" size_t scrib200_inner_product_matrix_workspace_bytes(int P, int Q, int64_t n_times, int n_cols) {
    using namespace scrib200;
    if (P <= 0 || Q <= 0 || n_times <= 0 || n_cols <= 0) return 0;
    if (P == 1 || Q == 1) return scrib200_inner_product_workspace_bytes(n_times, n_cols, P > Q ? P : Q);
    const MmGeom g = mm_geometry(P, Q, n_times * n_cols);
    return (size_t)g.splits * P * 2 * (size_t)Q * sizeof(double);
}

extern "C" int scrib200_inner_product_matrix(const double* A, int P, int64_t a_stride, const double* B, int Q,
                                             int64_t b_stride, int64_t n_times, int n_cols, const double* w, double* G,
                                             void* workspace, size_t workspace_bytes, void* stream) {
    using namespace scrib200;
    SCRIB200_REQUIRE(A && B && w && G, "inner_product_matrix: null pointer");
    SCRIB200_REQUIRE(P >= 1 && Q >= 1 && n_times >= 1 && n_cols >= 1, "inner_product_matrix: bad sizes P=%d Q=%d n_times=%lld n_cols=%d",
                     P, Q, (long long)n_times, n_cols);
    const int64_t K = n_times * n_cols;
    SCRIB200_REQUIRE(a_stride >= K && b_stride >= K, "inner_product_matrix: waveform strides %lld / %lld below n_times * n_cols = %lld",
                     (long long)a_stride, (long long)b_stride, (long long)K);
    // a single row or column of G is a matrix-vector product: HBM-bound, so it takes the streaming kernel (one batch entry
    // per waveform of the longer side, the other operand broadcast with batch stride 0)
    if (P == 1 || Q == 1) {
        const int nb = P > Q ? P : Q;
        return scrib200_inner_product(A, n_cols, 0, P == 1 ? 0 : a_stride, B, n_cols, 0, Q == 1 ? 0 : b_stride, n_times, n_cols,
                                      nb, w, 1, 0, G, workspace, workspace_bytes, stream);
    }
    SCRIB200_REQUIRE(K < ((int64_t)1 << 31), "inner_product_matrix: n_times * n_cols = %lld must be below 2^31", (long long)K);
    SCRIB200_REQUIRE(aligned16(A) && aligned16(B) && aligned16(G) && aligned16(workspace),
                     "inner_product_matrix: pointers must be 16-byte aligned");
    const MmGeom g = mm_geometry(P, Q, K);
    const size_t need = (size_t)g.splits * P * 2 * (size_t)Q * sizeof(double);
    SCRIB200_REQUIRE(workspace && workspace_bytes >= need, "inner_product_matrix: workspace of %zu bytes, %zu needed",
                     workspace_bytes, need);
    const cudaStream_t s = (cudaStream_t)stream;
    double* part = reinterpret_cast<double*>(workspace);
    inner_product_dmma_kernel<<<dim3(g.tiles_m * g.tiles_n, g.splits), 128, 0, s>>>(
        reinterpret_cast<const double2*>(A), P, a_stride, reinterpret_cast<const double2*>(B), Q, b_stride, n_cols, K, w,
        g.k_per_split, g.tiles_m, part);
    SCRIB200_CHECK_LAUNCH("inner_product_matrix");
    const int64_t len = (int64_t)P * 2 * Q;
    inner_product_splitk_sum_kernel<<<(unsigned)((len + 255) / 256), 256, 0, s>>>(part, g.splits, len, G);
    SCRIB200_CHECK_LAUNCH("inner_product_matrix_reduce");
    return SCRIB200_OK;
}
