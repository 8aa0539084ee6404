// linalg.cu — sm_100a kernels for the linear-algebra half of ORC's SIMPLE loop
// (src/linear_algebra.rs): SpMV with fused BiCGSTAB epilogues, fused vector updates, Jacobi scaling,
// Jacobi / Gauss-Seidel smoothers, the "Strongest" restriction as a sync-free dataflow kernel, the
// Galerkin triple product with nalgebra-sparse's symbolic-union pattern, and the 3-level multigrid driver.
//
// Everything is fp64 and HBM-bandwidth bound (SpMV: 2 flop / 12 B): no tensor cores. Rounding follows
// the reference: one rounding per operator, no FMA contraction (this file is compiled with -fmad=false),
// in-row sums in ascending column order. Only the global reductions (dot products) are summed in a
// different — but fixed, deterministic — order than nalgebra's 8-accumulator dot.
#include "linalg.cuh"
#include "dist.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include <algorithm>
#include <cfloat>
#include <cstring>
#include <cstdlib>
#include <climits>

namespace orc {

// device scalar slots (Ctx::d_scal)
enum Scal : int { S_RHO = 0, S_ALPHA, S_OMEGA, S_BETA, S_RHO_PREV, S_TMP0, S_TMP1, S_JAC_INIT, S_NORM, S_MAXABS, S_COUNT };

// =================================================================================================
// small utilities
// =================================================================================================
__global__ void k_fill(double* y, double v, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) y[i] = v;
}
__global__ void k_add_inplace(double* y, const double* x, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) y[i] = y[i] + x[i];
}
__global__ void k_scale_inplace(double* y, double s, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) y[i] = y[i] * s;
}
__global__ void k_sumsq(const double* x, int64_t n, double* partials, unsigned int* counter, double* out) {
    __shared__ double sh[32];
    double a = 0.;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) a += x[i] * x[i];
    double s = block_sum(a, sh);
    if (threadIdx.x == 0) partials[blockIdx.x] = s;
    if (last_block_done(counter)) {
        double t = sum_partials(partials, gridDim.x, sh);
        if (threadIdx.x == 0) *out = sqrt(t);
    }
}
void dev_fill(Ctx& c, double* y, double v, int64_t n) {
    if (n <= 0) return;
    k_fill<<<grid_for(n, 256, 1184), 256, 0, c.stream>>>(y, v, n);
    c.after_launch("k_fill");
}
void dev_axpy_inplace(Ctx& c, double* y, const double* x, int64_t n) {
    if (n <= 0) return;
    k_add_inplace<<<grid_for(n, 256, 1184), 256, 0, c.stream>>>(y, x, n);
    c.after_launch("k_add_inplace");
}
void dev_scale(Ctx& c, double* y, double s, int64_t n) {
    if (n <= 0) return;
    k_scale_inplace<<<grid_for(n, 256, 1184), 256, 0, c.stream>>>(y, s, n);
    c.after_launch("k_scale_inplace");
}
double dev_norm_host(Ctx& c, const double* x, int64_t n) {
    k_sumsq<<<grid_for(std::max<int64_t>(n, 1), 256, 1184), 256, 0, c.stream>>>(x, n, c.d_partials, c.d_counter, c.d_scal + S_NORM);
    c.after_launch("k_sumsq");
    double h = 0.;
    ORC_CUDA(cudaMemcpyAsync(&h, c.d_scal + S_NORM, sizeof(double), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    return h;
}

// =================================================================================================
// CSR plumbing
// =================================================================================================
CsrPtr csr_alloc(Ctx& c, int64_t nrows, int64_t ncols, int64_t nnz) {
    CsrPtr a(new DCsr());
    a->ctx = &c; a->nrows = nrows; a->ncols = ncols; a->nnz = nnz;
    a->rowptr = c.alloc_n<int>((size_t)nrows + 1);
    a->col = c.alloc_n<int>((size_t)std::max<int64_t>(nnz, 1));
    a->val = c.alloc_n<double>((size_t)std::max<int64_t>(nnz, 1));
    return a;
}
CsrPtr csr_like(Ctx& c, const DCsr& a) {
    CsrPtr b(new DCsr());
    b->ctx = &c; b->nrows = a.nrows; b->ncols = a.ncols; b->nnz = a.nnz;
    b->rowptr = a.rowptr; b->col = a.col; b->diag = a.diag;
    b->own_pattern = false; b->own_diag = false;
    b->sym = a.sym; b->full_diag = a.full_diag; b->max_row = a.max_row; b->simplex = a.simplex; b->hint = a.hint;
    b->val = c.alloc_n<double>((size_t)std::max<int64_t>(a.nnz, 1));
    return b;
}

__global__ void k_find_diag(int n, const int* __restrict__ rowptr, const int* __restrict__ col, int* __restrict__ diag, int* missing) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int lo = rowptr[i], hi = rowptr[i + 1], e = hi;
    while (lo < hi) {  // lower_bound(col[lo..hi), i)
        int mid = (lo + hi) >> 1;
        if (col[mid] < i) lo = mid + 1; else hi = mid;
    }
    int d = (lo < e && col[lo] == i) ? lo : -1;
    diag[i] = d;
    if (d < 0 && e > rowptr[i]) atomicAdd(missing, 1);  // only NON-EMPTY rows without a diagonal change A' = P^-1 A's pattern
}
void csr_ensure_diag(Ctx& c, DCsr& a) {
    if (a.diag) return;
    a.diag = c.alloc_n<int>((size_t)std::max<int64_t>(a.nrows, 1));
    a.own_diag = true;
    DBuf<int> miss(&c, 1);
    miss.zero();
    if (a.nrows > 0) {
        k_find_diag<<<(int)((a.nrows + 255) / 256), 256, 0, c.stream>>>((int)a.nrows, a.rowptr, a.col, a.diag, miss);
        c.after_launch("k_find_diag");
    }
    int h = 0;
    miss.download(&h);
    c.sync();
    a.full_diag = (h == 0) ? 1 : 0;
}

__global__ void k_check_sym(int n, const int* __restrict__ rowptr, const int* __restrict__ col, int* asym) {
    // one warp per 32 rows would be better; this runs once per user-supplied matrix only
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    for (int k = rowptr[i]; k < rowptr[i + 1]; ++k) {
        int j = col[k];
        if (j == i) continue;
        if (j >= n) { atomicAdd(asym, 1); continue; }
        int lo = rowptr[j], hi = rowptr[j + 1], e = hi;
        while (lo < hi) { int mid = (lo + hi) >> 1; if (col[mid] < i) lo = mid + 1; else hi = mid; }
        if (!(lo < e && col[lo] == i)) atomicAdd(asym, 1);
    }
}
__global__ void k_max_row(int n, const int* __restrict__ rowptr, int* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int m = (i < n) ? rowptr[i + 1] - rowptr[i] : 0;
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_down_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0) atomicMax(out, m);
}
void csr_ensure_max_row(Ctx& c, DCsr& a) {   // fills a.max_row if unknown (one small launch + read-back)
    if (a.max_row >= 0) return;
    a.max_row = 0;
    if (a.nrows == 0) return;
    DBuf<int> m(&c, 1);
    m.zero();
    k_max_row<<<(int)((a.nrows + 255) / 256), 256, 0, c.stream>>>((int)a.nrows, a.rowptr, m);
    c.after_launch("k_max_row");
    m.download(&a.max_row);
    c.sync();
}
void csr_check_symmetry(Ctx& c, DCsr& a) {
    if (a.sym >= 0) return;
    if (a.nrows != a.ncols) { a.sym = 0; return; }
    DBuf<int> asym(&c, 1);
    asym.zero();
    if (a.nrows > 0) {
        k_check_sym<<<(int)((a.nrows + 255) / 256), 256, 0, c.stream>>>((int)a.nrows, a.rowptr, a.col, asym);
        c.after_launch("k_check_sym");
    }
    int h = 0;
    asym.download(&h);
    c.sync();
    a.sym = (h == 0) ? 1 : 0;
}

// out = &a * sa + &b * sb for matrices that share their pattern (solver.rs:310-311). nalgebra-sparse: `&Csr * scalar` maps
// v -> v * scalar; `&x + &y` zero-fills the union pattern and runs c = 0 * c + 1 * x, then c = 1 * c + 1 * y.
__global__ void k_csr_blend(int64_t n, const double* __restrict__ a, double sa, const double* __restrict__ b, double sb, double* __restrict__ out) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double v = 0.;
        v = v + 1. * (a[i] * sa);
        v = v + 1. * (b[i] * sb);
        out[i] = v;
    }
}
void csr_blend(Ctx& c, const DCsr& a, double sa, const DCsr& b, double sb, DCsr& out) {
    ORC_REQUIRE(a.rowptr == b.rowptr && a.col == b.col && out.rowptr == a.rowptr && out.col == a.col && a.nnz == b.nnz && out.nnz == a.nnz,
                ORC_E_INVALID, "csr_blend: the matrices must share one pattern");
    if (a.nnz == 0) return;
    k_csr_blend<<<grid_for(a.nnz, 256, c.sm_count * 8), 256, 0, c.stream>>>(a.nnz, a.val, sa, b.val, sb, out.val);
    c.after_launch("k_csr_blend");
}

// bitwise comparison of two value arrays (NaNs with equal payloads compare equal, +0 and -0 differ: "identical" means
// that every later kernel sees the same bits)
__global__ void k_bits_differ(int64_t n, const unsigned long long* __restrict__ a, const unsigned long long* __restrict__ b, int* out) {
    int d = 0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) d |= (a[i] != b[i]);
    if (__syncthreads_or(d) && threadIdx.x == 0) *out = 1;
}
bool csr_values_identical(Ctx& c, const DCsr& a, const DCsr& b) {
    if (a.nnz != b.nnz || a.nrows != b.nrows || a.ncols != b.ncols) return false;
    if (a.rowptr != b.rowptr || a.col != b.col) return false;  // only matrices that SHARE their pattern arrays are compared
    if (a.val == b.val || a.nnz == 0) return true;
    DBuf<int> flag(&c, 1);
    flag.zero();
    k_bits_differ<<<grid_for(a.nnz, 256, c.sm_count * 8), 256, 0, c.stream>>>(a.nnz, reinterpret_cast<const unsigned long long*>(a.val),
                                                                          reinterpret_cast<const unsigned long long*>(b.val), flag);
    c.after_launch("k_bits_differ");
    int h = 1;
    flag.download(&h);
    c.sync();
    return h == 0;
}

// =================================================================================================
// SpMV: y = A x.  (&CsrMatrix * &DVector == spmm_csr_dense(beta=0, alpha=1): per row
// acc = 0; for k ascending: acc += a_ik * x_k; y_i = acc.)
//
// Two kernels (picked by the average row length): one thread per row for the fine level, G lanes per row for the AMG coarse
// levels; both keep the in-row sum in ascending-k order per lane. Epilogues fuse the BiCGSTAB / Jacobi vector work and the dot
// products that follow each SpMV in the reference (linear_algebra.rs:250-268, 199-202), so x, y are touched once. Vectors come
// as batches of K = 1 or 3 systems (Cell<K> below).
// =================================================================================================
constexpr int SPMV_BLOCK = 256;

enum Epi : int {
    EP_NONE = 0,
    EP_SUM_ALPHA,    // nu = A p;          alpha = rho / sum(nu)                        (:256-257; r_hat_0 == 1)
    EP_DOTS_OMEGA,   // t = A s;           omega = (t.s) / (t.t)                        (:260-261)
    EP_RESID_INIT,   // r = b - A x; p = r; rho = sum(r)                                (:250-254)
    EP_RESID,        // r = b - A x                                                     (:283)
    EP_RESID_NORM,   // ||b - A x||  -> S_NORM, NaN -> DF_MG_NAN                        (:97-105)
    EP_JACOBI,       // xn = w * (b0 - A0 x) + x * (1 - w); NaN scan of x               (:192-200)
    EP_JACOBI_RES    // r = ||b' - A' xn||, max|xn|, x = xn, convergence latch          (:202-216)
};

// ---- right-hand-side batches -----------------------------------------------------------------------------------------
// K = 1: plain vectors. K = 3: three systems that share ONE matrix are solved in lockstep (the u, v, w momentum systems of
// a SIMPLE iteration have bit-identical matrices unless the scheme is TVD, discretization.rs:217-286; the reference's
// BiCGSTAB is unguarded, so all three run exactly `iterations` iterations). Their vectors are interleaved in 32-byte
// cells [x_u, x_v, x_w, 0]: a gather of column j fetches one aligned sector — the same sector count as a scalar gather —
// and the matrix is streamed once instead of three times. Every system keeps its own scalars (slot block k * SCAL_STRIDE)
// and its own block partials; the per-system arithmetic, including the reduction trees, is the K = 1 arithmetic bit for bit.
constexpr int SCAL_STRIDE = 16;  // doubles per system in Ctx::d_scal (S_COUNT <= 16, 3 systems + 16 staging slots <= 64)
constexpr int S_STAGE = 48;      // K = 3, multi-GPU: local totals staged contiguously for ONE allreduce: [q * 3 + k]
template <int K> struct Cell;
template <> struct Cell<1> {
    static constexpr int S = 1;
    static __device__ __forceinline__ void ld(const double* p, size_t i, double (&v)[1]) { v[0] = p[i]; }
    static __device__ __forceinline__ void st(double* p, size_t i, const double (&v)[1]) { p[i] = v[0]; }
};
struct alignas(32) D4 { double a, b, c, d; };  // one 256-bit access (LDG.E.ENL2.256 / STG.E.ENL2.256 on sm_100a): a gather of a
                                               // cell costs one L1 wavefront, like a scalar gather
template <> struct Cell<3> {
    static constexpr int S = 4;
    static __device__ __forceinline__ void ld(const double* p, size_t i, double (&v)[3]) {
        const D4 q = reinterpret_cast<const D4*>(p)[i];
        v[0] = q.a; v[1] = q.b; v[2] = q.c;
    }
    static __device__ __forceinline__ void st(double* p, size_t i, const double (&v)[3]) {
        D4 q;
        q.a = v[0]; q.b = v[1]; q.c = v[2]; q.d = 0.;
        reinterpret_cast<D4*>(p)[i] = q;
    }
};
static inline int vstride(int K) { return K == 1 ? 1 : 4; }
// where the fused kernels publish local totals for a multi-GPU solve (quantity q of system k)
template <int K> __device__ __forceinline__ int stage_slot(int q, int k) { return K == 1 ? S_TMP0 + q : S_STAGE + q * 3 + k; }

struct SpmvArgs {
    int n;
    const int* rowptr;
    const int* col;
    const double* val;
    const double* x;
    double* y;          // primary output (may be null for EP_RESID_NORM)
    const double* b;    // rhs for residual-type epilogues
    double* y2;         // second output (p for EP_RESID_INIT, x for EP_JACOBI_RES)
    double* scal;
    double* partials;
    unsigned int* counter;
    int* flags;
    double w, one_minus_w, threshold;
    int iter;
    int defer;  // EP_JACOBI_RES: leave the convergence decision to k_dot_ref (reference-order norm)
    int dist;   // multi-GPU: publish the LOCAL totals (stage_slot); the scalars are derived after the allreduce
    int row0;   // Jacobi epilogues: kernel row i is row i + row0 of the vectors (a partition solves its owned rows only)
    int nv;     // virtual blocks of this launch (Ctx::kVirtualBlocks): the unit of the fused reductions
};

// per-row epilogue and the fused reductions, shared by the two SpMV kernels
template <int EPI, int K>
__device__ __forceinline__ void spmv_row_epilogue(const SpmvArgs& a, int i, const double (&acc)[K], double (&acc0)[K], double (&acc1)[K],
                                                  int& nanflag) {
    using C = Cell<K>;
    if (EPI == EP_NONE) {
        C::st(a.y, i, acc);
    } else if (EPI == EP_SUM_ALPHA) {
        C::st(a.y, i, acc);
#pragma unroll
        for (int k = 0; k < K; ++k) acc0[k] += acc[k];
    } else if (EPI == EP_DOTS_OMEGA) {
        C::st(a.y, i, acc);
        double xi[K];
        C::ld(a.x, i, xi);
#pragma unroll
        for (int k = 0; k < K; ++k) { acc0[k] += acc[k] * xi[k]; acc1[k] += acc[k] * acc[k]; }
    } else if (EPI == EP_RESID_INIT) {
        double bi[K], r[K];
        C::ld(a.b, i, bi);
#pragma unroll
        for (int k = 0; k < K; ++k) { r[k] = bi[k] - acc[k]; acc0[k] += r[k]; }
        C::st(a.y, i, r);
        C::st(a.y2, i, r);
    } else if (EPI == EP_RESID) {
        double bi[K], r[K];
        C::ld(a.b, i, bi);
#pragma unroll
        for (int k = 0; k < K; ++k) r[k] = bi[k] - acc[k];
        C::st(a.y, i, r);
    } else if (EPI == EP_RESID_NORM) {
        double bi[K];
        C::ld(a.b, i, bi);
#pragma unroll
        for (int k = 0; k < K; ++k) { const double r = bi[k] - acc[k]; acc0[k] += r * r; }
    } else if (EPI == EP_JACOBI) {  // K == 1 only (launch_spmv)
        const int g = i + a.row0;
        double xi = a.x[g];
        if (xi != xi) nanflag = 1;
        a.y[g] = a.w * (a.b[g] - acc[0]) + xi * a.one_minus_w;
    } else if (EPI == EP_JACOBI_RES) {  // K == 1 only
        const int g = i + a.row0;
        double xi = a.x[g];
        double r = a.b[g] - acc[0];
        acc0[0] += r * r;
        if (xi != xi) nanflag = 1; else acc1[0] = fmax(acc1[0], fabs(xi));
        a.y2[g] = xi;
    }
}
// number of fused sums of an epilogue: quantity q of system k lives in partial lane q * K + k (K = 3: at most 6 of 8 lanes)
template <int EPI, int K> struct EpiSums {
    static constexpr int NQ = (EPI == EP_DOTS_OMEGA) ? 2 * K : (EPI == EP_NONE || EPI == EP_RESID || EPI == EP_JACOBI) ? 0 : K;
    static constexpr bool parked = NQ > 0 && EPI != EP_JACOBI_RES;   // barrier-free path (vb_park / vb_publish)
    static constexpr int SH = parked ? kMaxLocalVb * NQ * kWarpsPerBlock + 32 * NQ : 32;   // doubles of shared memory
};
// end of ONE virtual block `vb` (the lv-th of this real block)
template <int EPI, int K>
__device__ __forceinline__ void spmv_block_partials(const SpmvArgs& a, int vb, int lv, double (&acc0)[K], double (&acc1)[K], int nanflag,
                                                    double* sh) {
    const int t = threadIdx.x;
    if (EPI == EP_NONE || EPI == EP_RESID) return;
    if (EPI == EP_JACOBI) {
        if (nanflag) atomicOr(a.flags, DF_NAN_JACOBI);
        return;
    }
    if (EPI == EP_JACOBI_RES) {  // single system, rare: plain block reductions
        double s0 = block_sum(acc0[0], sh);
        if (t == 0) a.partials[vb] = s0;
        double m1 = block_max(acc1[0], sh);
        if (t == 0) a.partials[Ctx::kMaxBlocks + vb] = m1;
        int anyn = __syncthreads_or(nanflag);
        if (t == 0) a.partials[2 * Ctx::kMaxBlocks + vb] = anyn ? 1. : 0.;
        return;
    }
    if (EPI == EP_DOTS_OMEGA) {
        double v[2 * K];
#pragma unroll
        for (int k = 0; k < K; ++k) { v[k] = acc0[k]; v[K + k] = acc1[k]; }
        vb_park<2 * K>(sh, lv, v);
    } else {
        vb_park<K>(sh, lv, acc0);
    }
}
// The Jacobi decision that follows the residual (linear_algebra.rs:202-216) from the totals of the scaled system: sum of r^2, max |xn|
// over the rows that are not NaN, and the number of NaN rows. One thread; the single-GPU residual kernel and k_jacobi_decide share it.
__device__ __forceinline__ void jacobi_decide(double* scal, int* flags, int iter, double threshold, double sum_r2, double max_abs, double nan_rows) {
    double r = sqrt(sum_r2);
    scal[S_NORM] = r;
    // `initial_residual` starts at 0 in every call (:170) and is taken at iter_num == 1 (:208, Q9)
    const double initial = (iter == 0) ? 0. : scal[S_JAC_INIT];
    if (iter == 1) {
        scal[S_JAC_INIT] = r;
    } else if (r / initial < threshold) {
        atomicOr(flags, DF_CONVERGED);
        return;  // `break` precedes the magnitude check (:209-216)
    }
    if (nan_rows == 0. && max_abs > 1e10) atomicOr(flags, DF_JACOBI_HUGE);  // a NaN maximum compares false in the reference
}

// the last block to finish combines the partials of all virtual blocks in a fixed order and derives the scalars that
// follow in the reference
template <int EPI, int K>
__device__ __forceinline__ void spmv_finalize(const SpmvArgs& a, int n_local, double* sh) {
    const int t = threadIdx.x;
    constexpr int NQ = EpiSums<EPI, K>::NQ;
    if constexpr (NQ == 0) {
        return;
    } else {
    if constexpr (EpiSums<EPI, K>::parked) vb_publish<NQ>(sh, n_local, blockIdx.x, gridDim.x, a.partials);
    const int G = a.nv;
    if (!last_block_done(a.counter)) return;
    double T0[K], T1[K];
    double T2 = 0.;
    if constexpr (EPI == EP_JACOBI_RES) {
        T0[0] = sum_partials(a.partials, G, sh);
        T1[0] = max_partials(a.partials + Ctx::kMaxBlocks, G, sh);
        T2 = sum_partials(a.partials + 2 * Ctx::kMaxBlocks, G, sh);
    } else {
        double T[NQ];
        sum_partials_n<NQ>(a.partials, G, T, sh + kMaxLocalVb * NQ * kWarpsPerBlock);
#pragma unroll
        for (int k = 0; k < K; ++k) { T0[k] = T[k]; T1[k] = (EPI == EP_DOTS_OMEGA) ? T[(K + k) % NQ] : 0.; }
    }
    if (t != 0) return;
#pragma unroll
    for (int k = 0; k < K; ++k) {
        double* scal = a.scal + k * SCAL_STRIDE;
        if (a.dist && EPI == EP_JACOBI_RES) {  // the three local totals that k_jacobi_decide reduces: sum at S_TMP0.., max at S_MAXABS
            scal[S_TMP0] = T0[0]; scal[S_TMP1] = T2; scal[S_MAXABS] = T1[0];
            return;
        }
        if (a.dist) { a.scal[stage_slot<K>(0, k)] = T0[k]; a.scal[stage_slot<K>(1, k)] = T1[k]; continue; }
        if (EPI == EP_SUM_ALPHA) {
            scal[S_ALPHA] = scal[S_RHO] / T0[k];
        } else if (EPI == EP_DOTS_OMEGA) {
            scal[S_OMEGA] = T0[k] / T1[k];
        } else if (EPI == EP_RESID_INIT) {
            scal[S_RHO] = T0[k];
        } else if (EPI == EP_RESID_NORM) {
            double nrm = sqrt(T0[k]);
            scal[S_NORM] = nrm;
            if (nrm != nrm) atomicOr(a.flags, DF_MG_NAN);
        } else if (EPI == EP_JACOBI_RES) {
            if (a.defer) { scal[S_MAXABS] = T1[0]; scal[S_TMP1] = T2; return; }
            jacobi_decide(scal, a.flags, a.iter, a.threshold, T0[0], T1[0], T2);
        }
    }
    }
}

// ---- short rows (fine level: 7 nnz/row hex, 5 tet): one thread per row, in-row sum in ascending-k order (bit-exact).
// Measured on B200 (scripts/lab/spmv_lab.cu, 128^3 7-point matrix, 217 MB): thread-per-row 39 us (5.5 TB/s) vs 47-59 us for
// shared-memory staged variants and 57 us for 4 lanes per row — consecutive rows are consecutive in (val, col), so the L1
// absorbs the 56-byte stride and every sector is used; the streaming ceiling of the same grid is 29 us. ----
template <int EPI, int K>
__global__ void __launch_bounds__(SPMV_BLOCK, (K == 1 ? 8 : 6)) k_spmv(const SpmvArgs a) {
    __shared__ double sh[EpiSums<EPI, K>::SH];
    if (EPI == EP_JACOBI || EPI == EP_JACOBI_RES) {
        if (*(volatile int*)a.flags & DF_CONVERGED) return;  // the reference broke out of its loop (:209-212)
    }
    int lv = 0;
    for (int vb = blockIdx.x; vb < a.nv; vb += gridDim.x, ++lv) {
        double acc0[K], acc1[K];  // per-thread partials of the fused reductions
#pragma unroll
        for (int k = 0; k < K; ++k) { acc0[k] = 0.; acc1[k] = 0.; }
        int nanflag = 0;
        for (int i = vb * SPMV_BLOCK + threadIdx.x; i < a.n; i += a.nv * SPMV_BLOCK) {
            const int lo = a.rowptr[i], hi = a.rowptr[i + 1];
            double acc[K];
#pragma unroll
            for (int k = 0; k < K; ++k) acc[k] = 0.;
            for (int q = lo; q < hi; ++q) {
                const double v = a.val[q];
                double xv[K];
                Cell<K>::ld(a.x, a.col[q], xv);
#pragma unroll
                for (int k = 0; k < K; ++k) acc[k] += v * xv[k];
            }
            spmv_row_epilogue<EPI, K>(a, i, acc, acc0, acc1, nanflag);
        }
        spmv_block_partials<EPI, K>(a, vb, lv, acc0, acc1, nanflag, sh);
    }
    spmv_finalize<EPI, K>(a, lv, sh);
}

// ---- long rows (AMG coarse levels: 17 / 44 / 111 entries per row measured at 128^3): G lanes per row, coalesced along the
// row, UN independent (val, col) loads in flight per lane before the dependent gathers of x, per-lane partial sums in
// ascending k followed by a fixed shuffle tree. Deterministic, but not the ascending-k order of the reference: values agree
// to rounding (DESIGN.md §5; aggregates and Galerkin products do not depend on SpMV results, so they stay bit-exact).
// What bounds it (profiles/r1_spmv_k3_ncu.txt): the L1 data pipe, not HBM — a scattered gather costs one L1 wavefront per
// distinct 32-byte sector (one system: 0.7 sectors per entry; three systems: exactly one, the 32-byte cell), ncu shows
// l1tex__data_pipe_lsu_wavefronts at 86-90 % of peak with DRAM at 32-55 %. Measured on the real 128^3 hierarchy
// (profiles/r1_level_bench.txt): 55 / 72 / 88 us per launch for one system (4.0-4.3 TB/s), 90 / 117 / 137 us for three
// (1.8-1.9 x the throughput of three launches). A serial tail loop instead of the predicated body costs 10-25 %. ----
template <int EPI, int G, int UN, int K>
__global__ void __launch_bounds__(SPMV_BLOCK, (K == 1 ? 8 : 6)) k_spmv_vec(const SpmvArgs a) {
    __shared__ double sh[EpiSums<EPI, K>::SH];
    if (EPI == EP_JACOBI || EPI == EP_JACOBI_RES) {
        if (*(volatile int*)a.flags & DF_CONVERGED) return;
    }
    const int t = threadIdx.x, gl = t & (G - 1);
    constexpr int RPB = SPMV_BLOCK / G;
    const int ngroups = (a.n + RPB - 1) / RPB;
    int lv = 0;
    for (int vb = blockIdx.x; vb < a.nv; vb += gridDim.x, ++lv) {
        double acc0[K], acc1[K];
#pragma unroll
        for (int k = 0; k < K; ++k) { acc0[k] = 0.; acc1[k] = 0.; }
        int nanflag = 0;
        for (int grp = vb; grp < ngroups; grp += a.nv) {
            const int i = grp * RPB + t / G;
            double acc[K];
#pragma unroll
            for (int k = 0; k < K; ++k) acc[k] = 0.;
            if (i < a.n) {
                const int lo = a.rowptr[i], hi = a.rowptr[i + 1];
                for (int q = lo + gl; q < hi; q += UN * G) {  // fully predicated body: no serial tail
                    double v[UN], xv[UN][K];
                    int cc[UN];
                    bool ok[UN];
#pragma unroll
                    for (int u = 0; u < UN; ++u) {
                        ok[u] = q + u * G < hi;
                        v[u] = ok[u] ? a.val[q + u * G] : 0.;
                        cc[u] = ok[u] ? a.col[q + u * G] : 0;   // inactive slots gather column 0 (always in range, also for rectangular matrices)
                    }
#pragma unroll
                    for (int u = 0; u < UN; ++u) Cell<K>::ld(a.x, cc[u], xv[u]);
#pragma unroll
                    for (int u = 0; u < UN; ++u)
                        if (ok[u]) {
#pragma unroll
                            for (int k = 0; k < K; ++k) acc[k] += v[u] * xv[u][k];
                        }
                }
            }
#pragma unroll
            for (int k = 0; k < K; ++k) {
#pragma unroll
                for (int o = G / 2; o > 0; o >>= 1) acc[k] += __shfl_down_sync(0xffffffffu, acc[k], o, G);
            }
            if (i < a.n && gl == 0) spmv_row_epilogue<EPI, K>(a, i, acc, acc0, acc1, nanflag);
        }
        spmv_block_partials<EPI, K>(a, vb, lv, acc0, acc1, nanflag, sh);
    }
    spmv_finalize<EPI, K>(a, lv, sh);
}

// how many blocks of a kernel one SM keeps resident (queried once per instantiation)
template <auto Kern>
static int resident_blocks(const Ctx& c, int block) {
    static int per_sm = 0;
    if (per_sm == 0) {
        int v = 0;
        ORC_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, Kern, block, 0));
        per_sm = std::max(v, 1);
    }
    return per_sm * c.sm_count;
}
// real blocks for nv virtual ones: what fits on the device, but never more than kMaxLocalVb virtual blocks per real block
static int virtual_grid(int nv, int resident) { return std::max(std::min(nv, resident), (nv + kMaxLocalVb - 1) / kMaxLocalVb); }
template <auto Kern>
static void launch_virtual(Ctx& c, SpmvArgs& a, int64_t tiles) {
    a.nv = (int)std::max<int64_t>(1, std::min<int64_t>(tiles, Ctx::kVirtualBlocks));
    const int grid = virtual_grid(a.nv, resident_blocks<Kern>(c, SPMV_BLOCK));
    Kern<<<grid, SPMV_BLOCK, 0, c.stream>>>(a);
}

static int spmv_grid(const Ctx& c, int64_t n) {
    int64_t tiles = (n + SPMV_BLOCK - 1) / SPMV_BLOCK;
    int64_t cap = (int64_t)c.sm_count * 8;  // 8 resident 256-thread blocks per SM
    return (int)std::max<int64_t>(1, std::min(tiles, cap));
}
template <int EPI, int K>
static void launch_spmv_k(Ctx& c, const DCsr& A, SpmvArgs a) {
    a.n = (int)A.nrows; a.rowptr = A.rowptr; a.col = A.col; a.val = A.val;
    a.scal = c.d_scal; a.partials = c.d_partials; a.counter = c.d_counter; a.flags = c.d_flags;
    // SURVEY.md §8d: values+cols and rowptr once, x and y once per system
    ProfScope ps(c, PC_SPMV, 12. * (double)A.nnz + 4. * (double)A.nrows + 16. * (double)K * (double)A.nrows,
                 (double)K * (12. * (double)A.nnz + 20. * (double)A.nrows),    // ... and as K SpMVs of the reference
                 (int64_t)A.nnz * 8 + K);
    if (c.prof.enabled) c.prof.rows_of[A.nnz] = A.nrows;
    const double avg = A.nrows > 0 ? (double)A.nnz / (double)A.nrows : 0.;
    auto tiles = [&](int rows_per_block) { return (A.nrows + rows_per_block - 1) / rows_per_block; };
    // the lanes-per-row choice fixes the in-row summation tree, so it is the same for K = 1 and K = 3 (bit-identical systems);
    // loads in flight per lane: 4 for one system, 2 for three (measured: profiles/r1_level_bench.txt)
    constexpr int UN = (K == 1) ? 4 : 2;
    if (avg < 10. || c.exact_order) {
        launch_virtual<k_spmv<EPI, K>>(c, a, tiles(SPMV_BLOCK));
    } else if (avg < 32.) {
        launch_virtual<k_spmv_vec<EPI, 4, UN, K>>(c, a, tiles(SPMV_BLOCK / 4));
    } else {
        launch_virtual<k_spmv_vec<EPI, 8, UN, K>>(c, a, tiles(SPMV_BLOCK / 8));
    }
    c.after_launch("k_spmv");
}
template <int EPI>
static void launch_spmv(Ctx& c, const DCsr& A, SpmvArgs a, int K = 1) {
    if (K == 1) { launch_spmv_k<EPI, 1>(c, A, a); return; }
    ORC_REQUIRE(K == 3 && !c.exact_order, ORC_E_INTERNAL, "SpMV batches hold 1 or 3 systems");
    if constexpr (EPI == EP_JACOBI || EPI == EP_JACOBI_RES) throw Error(ORC_E_INTERNAL, "Jacobi epilogues are single-system");
    else launch_spmv_k<EPI, 3>(c, A, a);
}
void spmv(Ctx& c, const DCsr& A, const double* x, double* y, int K) {
    if (A.nrows == 0) return;
    SpmvArgs a{};
    a.x = x; a.y = y;
    launch_spmv<EP_NONE>(c, A, a, K);
}

// =================================================================================================
// BiCGSTAB (linear_algebra.rs:247-269): unguarded, r_hat_0 == 1, exactly `iterations` iterations.
// Five launches per iteration; every scalar (rho, alpha, omega, beta) lives on the device, so the loop
// never synchronises with the host.
// =================================================================================================
template <int K>
__global__ void k_bicg_s(int64_t n, const double* __restrict__ r, const double* __restrict__ nu, double* __restrict__ s, const double* scal) {
    double alpha[K];
#pragma unroll
    for (int k = 0; k < K; ++k) alpha[k] = scal[k * SCAL_STRIDE + S_ALPHA];
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double ri[K], ni[K], si[K];
        Cell<K>::ld(r, i, ri);
        Cell<K>::ld(nu, i, ni);
#pragma unroll
        for (int k = 0; k < K; ++k) si[k] = ri[k] - alpha[k] * ni[k];  // s = &r - alpha * &nu  (:259)
        Cell<K>::st(s, i, si);
    }
}
template <int K>
__global__ void __launch_bounds__(256, (K == 1 ? 8 : 6)) k_bicg_xr(int64_t n, double* __restrict__ x, const double* __restrict__ p, const double* __restrict__ s,
                          const double* __restrict__ tv, double* __restrict__ r, double* scal, double* partials, unsigned int* counter,
                          int nv, int64_t own_lo = 0, int64_t own_hi = INT64_MAX, int dist = 0) {
    __shared__ double sh[kMaxLocalVb * K * kWarpsPerBlock + 32 * K];
    double alpha[K], omega[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { alpha[k] = scal[k * SCAL_STRIDE + S_ALPHA]; omega[k] = scal[k * SCAL_STRIDE + S_OMEGA]; }
    int lv = 0;
    for (int vb = blockIdx.x; vb < nv; vb += gridDim.x, ++lv) {  // virtual blocks: the reduction does not depend on the launch geometry
        double acc[K];
#pragma unroll
        for (int k = 0; k < K; ++k) acc[k] = 0.;
        for (int64_t i = vb * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)nv * blockDim.x) {
            double xi[K], pi[K], si[K], ti[K], ri[K];
            Cell<K>::ld(x, i, xi);
            Cell<K>::ld(p, i, pi);
            Cell<K>::ld(s, i, si);
            Cell<K>::ld(tv, i, ti);
            const bool own = (i >= own_lo && i < own_hi);  // rho = r_hat_0 . r  (:265); halo entries belong to another rank
#pragma unroll
            for (int k = 0; k < K; ++k) {
                const double h = xi[k] + alpha[k] * pi[k];   // h = &x + alpha * &p      (:258)
                xi[k] = h + omega[k] * si[k];                // x = &h + omega * &s      (:262)
                ri[k] = si[k] - omega[k] * ti[k];            // r = &s - omega * &t      (:263)
                if (own) acc[k] += ri[k];
            }
            Cell<K>::st(x, i, xi);
            Cell<K>::st(r, i, ri);
        }
        vb_park<K>(sh, lv, acc);
    }
    vb_publish<K>(sh, lv, blockIdx.x, gridDim.x, partials);
    if (last_block_done(counter)) {
        double T[K];
        sum_partials_n<K>(partials, nv, T, sh + kMaxLocalVb * K * kWarpsPerBlock);
        if (threadIdx.x == 0) {
#pragma unroll
            for (int k = 0; k < K; ++k) {
                if (dist) { scal[stage_slot<K>(0, k)] = T[k]; continue; }
                double* sc = scal + k * SCAL_STRIDE;
                double rho_prev = sc[S_RHO];
                sc[S_RHO_PREV] = rho_prev;
                sc[S_RHO] = T[k];
                sc[S_BETA] = T[k] / rho_prev * alpha[k] / omega[k];  // beta = rho / rho_prev * alpha / omega  (:266)
            }
        }
    }
}
template <int K>
__global__ void k_bicg_p(int64_t n, const double* __restrict__ r, double* __restrict__ p, const double* __restrict__ nu, const double* scal) {
    double beta[K], omega[K];
#pragma unroll
    for (int k = 0; k < K; ++k) { beta[k] = scal[k * SCAL_STRIDE + S_BETA]; omega[k] = scal[k * SCAL_STRIDE + S_OMEGA]; }
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double ri[K], pi[K], ni[K];
        Cell<K>::ld(r, i, ri);
        Cell<K>::ld(p, i, pi);
        Cell<K>::ld(nu, i, ni);
#pragma unroll
        for (int k = 0; k < K; ++k) pi[k] = ri[k] + beta[k] * (pi[k] - omega[k] * ni[k]);  // p = &r + beta * (p - omega * &nu)  (:267)
        Cell<K>::st(p, i, pi);
    }
}
// (b_u, b_v, b_w) <-> interleaved cells
__global__ void k_pack3(int64_t n, const double* __restrict__ a, const double* __restrict__ b, const double* __restrict__ c3, double* __restrict__ out) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const double v[3] = {a[i], b[i], c3[i]};
        Cell<3>::st(out, i, v);
    }
}
__global__ void k_unpack3(int64_t n, const double* __restrict__ in, double* __restrict__ a, double* __restrict__ b, double* __restrict__ c3) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double v[3];
        Cell<3>::ld(in, i, v);
        a[i] = v[0]; b[i] = v[1]; c3[i] = v[2];
    }
}
void pack3(Ctx& c, int64_t n, const double* a, const double* b, const double* c3, double* out) {
    if (n <= 0) return;
    k_pack3<<<grid_for(n, 256, c.sm_count * 8), 256, 0, c.stream>>>(n, a, b, c3, out);
    c.after_launch("k_pack3");
}
void unpack3(Ctx& c, int64_t n, const double* in, double* a, double* b, double* c3) {
    if (n <= 0) return;
    k_unpack3<<<grid_for(n, 256, c.sm_count * 8), 256, 0, c.stream>>>(n, in, a, b, c3);
    c.after_launch("k_unpack3");
}

// ---- reference-order reductions (orc_settings.reduction_mode == ORC_REDUCE_REFERENCE_ORDER) ----------------------------
// nalgebra's dot (base/blas.rs): eight interleaved accumulators over chunks of 8, combined as
// res += acc0+acc4; res += acc1+acc5; res += acc2+acc6; res += acc3+acc7; then the tail in order. Each accumulator is a
// sequential chain of n/8 additions, so the kernel is latency bound by construction (8 lanes of one warp): it exists to make
// the whole solve bit-identical to the reference on small meshes, where the unguarded BiCGSTAB (Q8) amplifies the last
// bit of every dot product into the leading digits of the result. Large meshes use the fused tree reductions instead.
enum DotOp : int { DOT_RHO_INIT = 0, DOT_ALPHA, DOT_TS, DOT_OMEGA, DOT_BETA, DOT_JACOBI_DECIDE, DOT_STORE };
__global__ void k_dot_ref(int64_t n, const double* __restrict__ a, const double* __restrict__ b, double* scal, int* flags, int op, int iter,
                          double threshold) {
    if (op == DOT_JACOBI_DECIDE && (*(volatile int*)flags & DF_CONVERGED)) return;
    const int lane = threadIdx.x;
    const int64_t m = n - (n % 8);
    double acc = 0.;
    if (lane < 8) {
        int64_t i = lane;
        for (; i + 56 < m; i += 64) {  // 8 loads in flight, then the dependent chain
            double pr[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) pr[u] = a[i + 8 * u] * (b ? b[i + 8 * u] : 1.);
#pragma unroll
            for (int u = 0; u < 8; ++u) acc += pr[u];
        }
        for (; i < m; i += 8) acc += a[i] * (b ? b[i] : 1.);
    }
    double a0 = __shfl_sync(0xffffffffu, acc, 0), a1 = __shfl_sync(0xffffffffu, acc, 1), a2 = __shfl_sync(0xffffffffu, acc, 2),
           a3 = __shfl_sync(0xffffffffu, acc, 3), a4 = __shfl_sync(0xffffffffu, acc, 4), a5 = __shfl_sync(0xffffffffu, acc, 5),
           a6 = __shfl_sync(0xffffffffu, acc, 6), a7 = __shfl_sync(0xffffffffu, acc, 7);
    if (lane != 0) return;
    double res = 0.;
    res += a0 + a4; res += a1 + a5; res += a2 + a6; res += a3 + a7;
    for (int64_t i = m; i < n; ++i) res += a[i] * (b ? b[i] : 1.);
    switch (op) {
        case DOT_RHO_INIT: scal[S_RHO] = res; break;
        case DOT_ALPHA: scal[S_ALPHA] = scal[S_RHO] / res; break;
        case DOT_TS: scal[S_TMP0] = res; break;
        case DOT_OMEGA: scal[S_OMEGA] = scal[S_TMP0] / res; break;
        case DOT_BETA: {  // k_bicg_xr has saved the previous rho in S_RHO_PREV
            const double rho_prev = scal[S_RHO_PREV];
            scal[S_RHO] = res;
            scal[S_BETA] = res / rho_prev * scal[S_ALPHA] / scal[S_OMEGA];
            break;
        }
        case DOT_JACOBI_DECIDE: {
            const double r = sqrt(res);
            scal[S_NORM] = r;
            const double initial = (iter == 0) ? 0. : scal[S_JAC_INIT];
            if (iter == 1) {
                scal[S_JAC_INIT] = r;
            } else if (r / initial < threshold) {
                atomicOr(flags, DF_CONVERGED);
                break;
            }
            if (scal[S_TMP1] == 0. && scal[S_MAXABS] > 1e10) atomicOr(flags, DF_JACOBI_HUGE);
            break;
        }
        default: scal[S_NORM] = res;
    }
}
static void dot_ref(Ctx& c, int64_t n, const double* a, const double* b, int op, int iter = 0, double thr = 0.) {
    k_dot_ref<<<1, 32, 0, c.stream>>>(n, a, b, c.d_scal, c.d_flags, op, iter, thr);
    c.after_launch("k_dot_ref");
}
static void bicgstab_reference_order(Ctx& c, const DCsr& A, const double* b, double* x, uint64_t iterations) {
    const int64_t n = A.nrows;
    DBuf<double> r(&c, n), p(&c, n), nu(&c, n), s(&c, n), tv(&c, n);
    const int vg = grid_for(n, 256, Ctx::kVirtualBlocks), xr_cap = resident_blocks<k_bicg_xr<1>>(c, 256);
    { SpmvArgs a{}; a.x = x; a.y = r; a.y2 = p; a.b = b; launch_spmv<EP_RESID_INIT>(c, A, a); }   // r = b - A x; p = r
    dot_ref(c, n, r, nullptr, DOT_RHO_INIT);                                                       // rho = r . r_hat_0
    for (uint64_t it = 0; it < iterations; ++it) {
        { SpmvArgs a{}; a.x = p; a.y = nu; launch_spmv<EP_NONE>(c, A, a); }
        dot_ref(c, n, nu, nullptr, DOT_ALPHA);                                                     // alpha = rho / (r_hat_0 . nu)
        k_bicg_s<1><<<vg, 256, 0, c.stream>>>(n, r, nu, s, c.d_scal);
        c.after_launch("k_bicg_s");
        { SpmvArgs a{}; a.x = s; a.y = tv; launch_spmv<EP_NONE>(c, A, a); }
        dot_ref(c, n, tv, s, DOT_TS);
        dot_ref(c, n, tv, tv, DOT_OMEGA);                                                          // omega = (t.s) / (t.t)
        k_bicg_xr<1><<<virtual_grid(vg, xr_cap), 256, 0, c.stream>>>(n, x, p, s, tv, r, c.d_scal, c.d_partials, c.d_counter, vg);
        c.after_launch("k_bicg_xr");
        dot_ref(c, n, r, nullptr, DOT_BETA);                                                       // rho, beta in reference order
        k_bicg_p<1><<<vg, 256, 0, c.stream>>>(n, r, p, nu, c.d_scal);
        c.after_launch("k_bicg_p");
    }
}

// =================================================================================================
// Multi-GPU solves (SURVEY.md §8e): rows partitioned by contiguous cell ranges, halo exchange before every SpMV (C1), one
// small allreduce per scalar (C2). Local totals are published by the fused kernels; k_dist_scalar derives alpha/omega/
// beta/rho from the reduced values with the reference's formulas, so the loop still never synchronises with the host.
// =================================================================================================
enum DistOp : int { DO_RHO_INIT = 0, DO_ALPHA, DO_OMEGA, DO_BETA, DO_NORMCHK };
// With peer windows (dist.cuh) the allreduce of the staged totals happens in this same launch: one warp exchanges the `count * K`
// doubles with every peer's mailbox, sums them in rank order, then threads 0 .. K-1 derive the scalars.
template <int K>
__global__ void k_dist_scalar(double* scal_all, int* flags, int op, PeerAr pa, int count) {
    if (pa.nranks > 1) peer_allreduce_warp(pa, scal_all + (K == 1 ? (int)S_TMP0 : S_STAGE), count * K, 0, flags);
    const int k = threadIdx.x;
    if (k >= K) return;
    double* scal = scal_all + k * SCAL_STRIDE;
    const double t0 = scal_all[stage_slot<K>(0, k)], t1 = scal_all[stage_slot<K>(1, k)];
    switch (op) {
        case DO_RHO_INIT: scal[S_RHO] = t0; break;
        case DO_ALPHA: scal[S_ALPHA] = scal[S_RHO] / t0; break;
        case DO_OMEGA: scal[S_OMEGA] = t0 / t1; break;
        case DO_BETA: {
            const double rho_prev = scal[S_RHO];
            scal[S_RHO_PREV] = rho_prev;
            scal[S_RHO] = t0;
            scal[S_BETA] = t0 / rho_prev * scal[S_ALPHA] / scal[S_OMEGA];
            break;
        }
        default: {
            const double nrm = sqrt(t0);
            scal[S_NORM] = nrm;
            if (nrm != nrm) atomicOr(flags, DF_MG_NAN);
        }
    }
}
// `count` quantities per system were published by a fused kernel (stage_slot): ONE allreduce for all systems
template <int K>
static void dist_scalar(Ctx& c, const DistEnv& env, int count, int op) {
    PeerAr pa;   // nranks == 1: the totals are already reduced (NCCL below)
    if (env.comm->peer.on) {
        pa = env.comm->next_allreduce();
    } else {
        env.comm->allreduce(c, c.d_scal + (K == 1 ? (int)S_TMP0 : S_STAGE), count * K, 0);
    }
    ProfScope ps(c, PC_OTHER, 0.);
    k_dist_scalar<K><<<1, 32, 0, c.stream>>>(c.d_scal, c.d_flags, op, pa, count);
    c.after_launch("k_dist_scalar");
}

// On a partition (env->on()): A's rows are the local cells incl. halo (halo rows are empty). The halo of every SpMV input is
// exchanged first, the fused kernels publish local totals (SpmvArgs::dist) and dist_scalar reduces them across the ranks.
template <int K>
static void bicgstab_k(Ctx& c, const DCsr& A, const double* b, double* x, uint64_t iterations, const DistEnv* env) {
    const bool dist = env && env->on();
    const int64_t n = A.nrows;
    constexpr int S = Cell<K>::S;
    DBuf<double> r(&c, n * S), p(&c, n * S), nu(&c, n * S), s(&c, n * S), tv(&c, n * S);
    if (dist) for (DBuf<double>* v : {&r, &p, &nu, &s, &tv}) v->zero();
    const int64_t own_lo = dist ? env->halo->own_lo : 0, own_hi = dist ? env->halo->own_hi : n;   // rho sums the owned rows
    auto exchange = [&](double* v) { if (dist) env->halo->exchange(c, *env->comm, v, S); };
    auto reduce = [&](int count, int op) { if (dist) dist_scalar<K>(c, *env, count, op); };
    const int vg = grid_for(n, 256, Ctx::kVirtualBlocks), xr_cap = resident_blocks<k_bicg_xr<K>>(c, 256);
    // algorithmic bytes of the call: per iteration 2 SpMVs (matrix once, x and y per system) + the three vector kernels
    // (s: 3 passes, x/r: 6, p: 4 — `h` is fused away; the reference's model has 14 passes), plus the initial residual
    const double spmv_b = 12. * (double)A.nnz + 4. * (double)n + 16. * K * (double)n;
    ProfScope whole(c, PC_BICG, (double)iterations * (2. * spmv_b + 104. * K * (double)n) + spmv_b + 16. * K * (double)n,
                    (double)iterations * K * (24. * (double)A.nnz + 152. * (double)n), (int64_t)A.nnz * 8 + K + 4);
    if (c.prof.enabled) c.prof.rows_of[A.nnz] = A.nrows;
    exchange(x);
    { SpmvArgs a{}; a.x = x; a.y = r; a.y2 = p; a.b = b; a.dist = dist; launch_spmv<EP_RESID_INIT>(c, A, a, K); }
    reduce(1, DO_RHO_INIT);
    for (uint64_t it = 0; it < iterations; ++it) {
        exchange(p);
        { SpmvArgs a{}; a.x = p; a.y = nu; a.dist = dist; launch_spmv<EP_SUM_ALPHA>(c, A, a, K); }
        reduce(1, DO_ALPHA);
        {
            ProfScope ps(c, PC_VECTOR, 24. * K * (double)n);
            k_bicg_s<K><<<vg, 256, 0, c.stream>>>(n, r, nu, s, c.d_scal);
            c.after_launch("k_bicg_s");
        }
        exchange(s);
        { SpmvArgs a{}; a.x = s; a.y = tv; a.dist = dist; launch_spmv<EP_DOTS_OMEGA>(c, A, a, K); }
        reduce(2, DO_OMEGA);
        {
            ProfScope ps(c, PC_VECTOR, 48. * K * (double)n);
            k_bicg_xr<K><<<virtual_grid(vg, xr_cap), 256, 0, c.stream>>>(n, x, p, s, tv, r, c.d_scal, c.d_partials, c.d_counter, vg, own_lo,
                                                                          own_hi, dist);
            c.after_launch("k_bicg_xr");
        }
        reduce(1, DO_BETA);
        {
            ProfScope ps(c, PC_VECTOR, 32. * K * (double)n);
            k_bicg_p<K><<<vg, 256, 0, c.stream>>>(n, r, p, nu, c.d_scal);
            c.after_launch("k_bicg_p");
        }
    }
}
void bicgstab(Ctx& c, const DCsr& A, const double* b, double* x, uint64_t iterations, int K, const DistEnv* env) {
    const bool dist = env && env->on();
    const int64_t n = A.nrows;
    ORC_REQUIRE(A.nrows == A.ncols, ORC_E_INVALID, "bicgstab: matrix must be square");
    if (n == 0 && !dist) return;   // a rank without cells still takes part in the collectives
    if (c.exact_order) {
        ORC_REQUIRE(!dist, ORC_E_UNSUPPORTED, "reference-order reductions are single-GPU only");
        ORC_REQUIRE(K == 1, ORC_E_UNSUPPORTED, "reference-order reductions solve one system at a time");
        if (small_solve_ok(c, A)) bicgstab_small(c, A, b, x, iterations);   // one launch, same arithmetic (small.cu)
        else bicgstab_reference_order(c, A, b, x, iterations);
        return;
    }
    if (K == 1) bicgstab_k<1>(c, A, b, x, iterations, env);
    else bicgstab_k<3>(c, A, b, x, iterations, env);
}

// =================================================================================================
// Jacobi preconditioner (linear_algebra.rs:157-168): A' = P^-1 A with P^-1 = diagonal_as_csr().map(1/v)
// (an SpGEMM in the reference: c_ij = (1 * pinv_i) * a_ij), b' = P^-1 b (an SpMV: 0 + pinv_i * b_i).
// Rows whose diagonal is not stored have an empty P^-1 row, hence an empty A' row and b'_i = 0.
// =================================================================================================
template <int K>
__global__ void __launch_bounds__(SPMV_BLOCK) k_jacobi_scale(int n, const int* __restrict__ rowptr, const int* __restrict__ diag,
                                                             const double* __restrict__ val, const double* __restrict__ b,
                                                             double* __restrict__ val_out, double* __restrict__ b_out) {
    __shared__ int rp[SPMV_BLOCK + 1];
    __shared__ double pinv[SPMV_BLOCK];
    const int t = threadIdx.x;
    const int ntiles = (n + SPMV_BLOCK - 1) / SPMV_BLOCK;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int r0 = tile * SPMV_BLOCK;
        const int nr = min(SPMV_BLOCK, n - r0);
        __syncthreads();
        for (int q = t; q <= nr; q += SPMV_BLOCK) rp[q] = rowptr[r0 + q];
        if (t < nr) {
            int d = diag[r0 + t];
            double pi = (d >= 0) ? 1. / val[d] : 0.;
            pinv[t] = pi;
            if (b_out) {
                double bi[K], bo[K];
                Cell<K>::ld(b, r0 + t, bi);
#pragma unroll
                for (int k = 0; k < K; ++k) bo[k] = (d >= 0) ? 0. + pi * bi[k] : 0.;
                Cell<K>::st(b_out, r0 + t, bo);
            }
        }
        __syncthreads();
        const int kbeg = rp[0], kend = rp[nr];
        for (int k = kbeg + t; k < kend; k += SPMV_BLOCK) {
            int lo = 0, hi = nr;  // row of entry k: last r with rp[r] <= k
            while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (rp[mid] <= k) lo = mid; else hi = mid; }
            val_out[k] = 0. + (1. * pinv[lo]) * val[k];
        }
    }
}
// compaction for the rare case of rows without a stored diagonal (their A' row is empty)
__global__ void k_row_keep_counts(int n, const int* rowptr, const int* diag, int* cnt) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) cnt[i] = diag[i] >= 0 ? rowptr[i + 1] - rowptr[i] : 0;
}
__global__ void k_row_compact(int n, const int* rowptr, const int* diag, const int* col, const double* val, const int* rowptr_out,
                              int* col_out, double* val_out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || diag[i] < 0) return;
    int o = rowptr_out[i];
    for (int k = rowptr[i]; k < rowptr[i + 1]; ++k, ++o) { col_out[o] = col[k]; val_out[o] = val[k]; }
}
static void exclusive_scan_to_rowptr(Ctx& c, const int* counts, int* rowptr, int64_t n) {
    // rowptr[0..n] = exclusive scan of counts[0..n) with the total in rowptr[n]; counts must have n+1 slots (last = 0)
    size_t tmp_bytes = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, counts, rowptr, (int)(n + 1), c.stream);
    DBuf<char> tmp(&c, tmp_bytes);
    ORC_CUDA(cub::DeviceScan::ExclusiveSum(tmp.p, tmp_bytes, counts, rowptr, (int)(n + 1), c.stream));
    ++c.launches;
}

CsrPtr jacobi_scale(Ctx& c, DCsr& A, const double* b, double* b_out, int K) {
    ORC_REQUIRE(A.nrows == A.ncols, ORC_E_INVALID, "jacobi_scale: matrix must be square");
    csr_ensure_diag(c, A);
    CsrPtr out = csr_like(c, A);
    if (A.nrows == 0) return out;
    if (K == 1) k_jacobi_scale<1><<<spmv_grid(c, A.nrows), SPMV_BLOCK, 0, c.stream>>>((int)A.nrows, A.rowptr, A.diag, A.val, b, out->val, b_out);
    else k_jacobi_scale<3><<<spmv_grid(c, A.nrows), SPMV_BLOCK, 0, c.stream>>>((int)A.nrows, A.rowptr, A.diag, A.val, b, out->val, b_out);
    c.after_launch("k_jacobi_scale");
    if (A.full_diag == 1) return out;
    // slow path: drop the rows whose diagonal is not stored
    const int n = (int)A.nrows;
    DBuf<int> cnt(&c, (size_t)n + 1);
    cnt.zero();
    k_row_keep_counts<<<(n + 255) / 256, 256, 0, c.stream>>>(n, A.rowptr, A.diag, cnt);
    c.after_launch("k_row_keep_counts");
    DBuf<int> rp(&c, (size_t)n + 1);
    exclusive_scan_to_rowptr(c, cnt, rp, n);
    int nnz = 0;
    ORC_CUDA(cudaMemcpyAsync(&nnz, rp.p + n, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    CsrPtr packed = csr_alloc(c, A.nrows, A.ncols, nnz);
    ORC_CUDA(cudaMemcpyAsync(packed->rowptr, rp.p, sizeof(int) * ((size_t)n + 1), cudaMemcpyDeviceToDevice, c.stream));
    k_row_compact<<<(n + 255) / 256, 256, 0, c.stream>>>(n, A.rowptr, A.diag, A.col, out->val, packed->rowptr, packed->col, packed->val);
    c.after_launch("k_row_compact");
    packed->hint = A.hint; packed->sym = -1; packed->max_row = A.max_row; packed->simplex = A.simplex;
    return packed;
}

// =================================================================================================
// Jacobi (linear_algebra.rs:172-218)
// =================================================================================================
__global__ void k_jacobi_prepare(int lo, int hi, const int* __restrict__ rowptr, const int* __restrict__ col, const int* __restrict__ diag,
                                 const double* __restrict__ val, const double* __restrict__ b, double* __restrict__ val0,
                                 double* __restrict__ b0, int* flags) {
    // a_prime = v / a(i,i) off the diagonal, 0 on it; b_prime = b / a(i,i). a.get(i,i) panics if not stored. Rows [lo, hi).
    int i = lo + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= hi) return;
    int d = diag[i];
    if (d < 0) { atomicOr(flags, DF_MISSING_ENTRY); return; }
    double aii = val[d];
    for (int k = rowptr[i]; k < rowptr[i + 1]; ++k) val0[k] = (col[k] == i) ? 0. : val[k] / aii;
    b0[i] = b[i] / aii;
}
__global__ void k_clear_latch(int* f) { atomicAnd(f, ~DF_CONVERGED); }
// On a partition the update is row-local and a partition keeps the column order of every row, so the iterates are the single-GPU
// fast mode's bit for bit; only the residual norm that decides the break is summed per rank and then across ranks. Every rank takes
// that decision (the latch, the magnitude check) from the same reduced bits.
__global__ void k_jacobi_decide(double* scal, int* flags, PeerAr pa_sum, PeerAr pa_max, int iter, double threshold) {
    if (pa_sum.nranks > 1) {   // peer path: the two allreduces in this launch (sum of r^2 and NaN rows, then max |xn|)
        peer_allreduce_warp(pa_sum, scal + S_TMP0, 2, 0, flags);
        peer_allreduce_warp(pa_max, scal + S_MAXABS, 1, 2, flags);
    }
    if (threadIdx.x != 0) return;
    if (*(volatile int*)flags & DF_CONVERGED) return;   // latched: the residual kernel published nothing
    jacobi_decide(scal, flags, iter, threshold, scal[S_TMP0], scal[S_MAXABS], scal[S_TMP1]);
}
static void jacobi(Ctx& c, DCsr& A, const double* b, double* x, const SolveParams& sp, const DistEnv* env) {
    const bool dist = env && env->on();
    const int64_t n = A.nrows;   // on a partition: local cells incl. halo; halo rows are empty and store no diagonal
    if (n == 0 && !dist) return;
    const int64_t lo = dist ? env->halo->own_lo : 0, nown = dist ? env->halo->own_hi - lo : n;   // the rows this rank solves
    csr_ensure_diag(c, A);
    CsrPtr A0 = csr_like(c, A);
    DBuf<double> b0(&c, (size_t)std::max<int64_t>(n, 1)), xn(&c, (size_t)std::max<int64_t>(n, 1));
    if (dist) xn.zero();
    if (nown > 0) {
        k_jacobi_prepare<<<(int)((nown + 255) / 256), 256, 0, c.stream>>>((int)lo, (int)(lo + nown), A.rowptr, A.col, A.diag, A.val, b, A0->val, b0,
                                                                          c.d_flags);
        c.after_launch("k_jacobi_prepare");
    }
    // the owned rows as a matrix of their own: row i of the view is row lo + i (SpmvArgs::row0), columns stay local ids
    auto owned_rows = [&](const DCsr& M) {
        DCsr v;   // no context: the view frees nothing
        v.nrows = nown; v.ncols = M.ncols; v.nnz = M.nnz; v.rowptr = M.rowptr + lo; v.col = M.col; v.val = M.val;
        return v;
    };
    const DCsr A0v = owned_rows(*A0), Av = owned_rows(A);
    for (uint64_t it = 0; it < sp.iterations; ++it) {
        if (dist) env->halo->exchange(c, *env->comm, x);
        if (nown > 0) {
            SpmvArgs a{};
            a.x = x; a.y = xn; a.b = b0; a.w = sp.relaxation; a.one_minus_w = 1. - sp.relaxation; a.row0 = (int)lo;
            launch_spmv<EP_JACOBI>(c, A0v, a);
        }
        if (dist) env->halo->exchange(c, *env->comm, xn);
        if (nown > 0) {
            SpmvArgs r{};
            r.x = xn; r.y2 = x; r.b = b; r.iter = (int)it; r.threshold = sp.threshold; r.defer = c.exact_order ? 1 : 0; r.dist = dist;
            r.row0 = (int)lo;
            launch_spmv<EP_JACOBI_RES>(c, Av, r);
        } else {
            ORC_CUDA(cudaMemsetAsync(c.d_scal + S_TMP0, 0, 2 * sizeof(double), c.stream));   // a rank without cells adds nothing
            ORC_CUDA(cudaMemsetAsync(c.d_scal + S_MAXABS, 0, sizeof(double), c.stream));
        }
        if (c.exact_order) {  // r = (b' - A' x).norm() in nalgebra's accumulation order decides the break (:202-212); one GPU only
            SpmvArgs q{};
            q.x = x; q.y = xn; q.b = b;
            launch_spmv<EP_RESID>(c, A, q);
            dot_ref(c, n, xn, xn, DOT_JACOBI_DECIDE, (int)it, sp.threshold);
        }
        if (dist) {   // the residual kernel published the local totals: reduce them and decide on every rank
            Comm& cm = *env->comm;
            PeerAr ps, pm;   // nranks == 1: NCCL has reduced the totals already
            if (cm.peer.on) {
                ps = cm.next_allreduce();
                pm = cm.next_allreduce();
            } else {
                cm.allreduce(c, c.d_scal + S_TMP0, 2, 0);
                cm.allreduce(c, c.d_scal + S_MAXABS, 1, 2);
            }
            ProfScope pscope(c, PC_OTHER, 0.);
            k_jacobi_decide<<<1, 32, 0, c.stream>>>(c.d_scal, c.d_flags, ps, pm, (int)it, sp.threshold);
            c.after_launch("k_jacobi_decide");
        }
    }
    // clear the convergence latch (stream ordered) so that later solves start fresh
    k_clear_latch<<<1, 1, 0, c.stream>>>(c.d_flags);
    c.after_launch("k_clear_latch");
}

// =================================================================================================
// Gauss-Seidel (linear_algebra.rs:219-246), intended semantics (the reference arm cannot run: Q10):
// forward sweep in row order, x_i = x_i (1-w) + w (b_i - sum_{j != i} a_ij x_j) / a_ii with the newest x.
// Exact parallelisation: a sync-free dataflow sweep. A warp owns a chunk of consecutive rows and walks
// them in order; a row waits until every stored lower neighbour has been updated in this sweep.
// Chunks are handed out through an atomic ticket, so every chunk a warp can wait on is already owned
// by a resident warp (forward progress without a cooperative launch).
// =================================================================================================
constexpr int DF_CHUNK = 8;             // rows per warp-chunk in the dataflow kernels
constexpr long long SPIN_LIMIT = 1ll << 22;

__global__ void k_gs_sweep(int n, const int* __restrict__ rowptr, const int* __restrict__ col, const double* __restrict__ val,
                           const int* __restrict__ diag, const double* __restrict__ b, double* x, double w, double one_minus_w,
                           int* done, int sweep, unsigned int* ticket, int* flags) {
    const int lane = threadIdx.x & 31;
    const int nchunks = (n + DF_CHUNK - 1) / DF_CHUNK;
    for (;;) {
        unsigned int chunk = 0;
        if (lane == 0) chunk = atomicAdd(ticket, 1u);
        chunk = __shfl_sync(0xffffffffu, chunk, 0);
        if ((int)chunk >= nchunks) return;
        const int r0 = chunk * DF_CHUNK, r1 = min(n, r0 + DF_CHUNK);
        for (int i = r0; i < r1; ++i) {
            const int lo = rowptr[i], hi = rowptr[i + 1];
            double sum = 0.;
            for (int base = lo; base < hi; base += 32) {
                const int k = base + lane;
                double pr = 0.;
                int j = -1;
                if (k < hi) {
                    j = col[k];
                    if (j != i) {
                        if (j < i && j < r0) {  // rows of this chunk below i were finished by this warp already
                            long long spins = 0;
                            while (*(volatile int*)(done + j) < sweep) {
                                if ((++spins & 1023) == 0 && (spins > SPIN_LIMIT || (*(volatile int*)flags & DF_SPIN))) { atomicOr(flags, DF_SPIN); break; }
                            }
                            __threadfence();
                        }
                        pr = val[k] * __ldcg(x + j);
                    }
                }
                const int cnt = min(32, hi - base);
                for (int l = 0; l < cnt; ++l) {  // ordered sum, identical in every lane
                    double v = __shfl_sync(0xffffffffu, pr, l);
                    int jj = __shfl_sync(0xffffffffu, j, l);
                    if (jj != i) sum += v;
                }
            }
            if (lane == 0) {
                const int d = diag[i];
                if (d < 0) {
                    atomicOr(flags, DF_MISSING_ENTRY);
                } else {
                    double xi = __ldcg(x + i) * one_minus_w + w * (b[i] - sum) / val[d];
                    if (xi != xi) atomicOr(flags, DF_GS_NAN);
                    __stcg(x + i, xi);
                }
                __threadfence();
                *(volatile int*)(done + i) = sweep;
            }
            __syncwarp();
        }
    }
}
__global__ void k_gs_serial(int n, const int* rowptr, const int* col, const double* val, const int* diag, const double* b, double* x,
                            double w, double one_minus_w, int* flags) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    for (int i = 0; i < n; ++i) {
        double sum = 0.;
        for (int k = rowptr[i]; k < rowptr[i + 1]; ++k)
            if (col[k] != i) sum += val[k] * x[col[k]];
        int d = diag[i];
        if (d < 0) { atomicOr(flags, DF_MISSING_ENTRY); return; }
        double xi = x[i] * one_minus_w + w * (b[i] - sum) / val[d];
        if (xi != xi) atomicOr(flags, DF_GS_NAN);
        x[i] = xi;
    }
}
// ---- multicolour variant (a different ordering): the greedy colouring in row order, colour(i) = the smallest colour that no stored
// lower neighbour j < i has. It is built in rounds: row i is coloured in the first round in which every lower neighbour was coloured
// in an EARLIER round (`coloured_in`, -1 while uncoloured). A neighbour coloured in the same round, or a racing read of its write,
// reads as `round` or -1 and defers i, so each row sees the final colours of all its lower neighbours: the result is the sequential
// greedy colouring whatever the thread timing. On a structurally symmetric pattern it is a proper colouring (an upper neighbour j of
// i has i as a lower neighbour), so the rows of one colour are independent. st[0] counts the rows left, st[1] = 1 + the largest colour.
__global__ void k_colour_round(int n, const int* __restrict__ rowptr, const int* __restrict__ col, int* colour, int* coloured_in, int round,
                               int* st) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || coloured_in[i] >= 0) return;
    const int lo = rowptr[i], hi = rowptr[i + 1];
    for (int k = lo; k < hi; ++k) {
        int j = col[k];
        if (j < i) { int rj = ((volatile int*)coloured_in)[j]; if (rj < 0 || rj >= round) { atomicAdd(st, 1); return; } }
    }
    // smallest colour unused by the lower neighbours, 64 candidates per pass (it is at most their number, so the loop ends)
    int c = 0;
    for (int base = 0;; base += 64) {
        unsigned long long used = 0;
        for (int k = lo; k < hi; ++k) {
            int j = col[k];
            if (j < i) { int d = colour[j] - base; if (d >= 0 && d < 64) used |= 1ull << d; }
        }
        if (~used) { c = base + __ffsll((long long)~used) - 1; break; }
    }
    colour[i] = c;
    coloured_in[i] = round;
    atomicMax(st + 1, c + 1);
}
__global__ void k_gs_colour(int n, const int* __restrict__ rowptr, const int* __restrict__ col, const double* __restrict__ val,
                            const int* __restrict__ diag, const double* __restrict__ b, double* x, double w, double one_minus_w,
                            const int* __restrict__ colour, int which, int* flags) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || colour[i] != which) return;
    double sum = 0.;
    for (int k = rowptr[i]; k < rowptr[i + 1]; ++k)
        if (col[k] != i) sum += val[k] * x[col[k]];
    int d = diag[i];
    if (d < 0) { atomicOr(flags, DF_MISSING_ENTRY); return; }
    double xi = x[i] * one_minus_w + w * (b[i] - sum) / val[d];
    if (xi != xi) atomicOr(flags, DF_GS_NAN);
    x[i] = xi;
}

static int dataflow_grid(const Ctx& c, int64_t nchunks, int warps_per_block) {
    int64_t blocks = (nchunks + warps_per_block - 1) / warps_per_block;
    int64_t cap = (int64_t)c.sm_count * (64 / warps_per_block);
    return (int)std::max<int64_t>(1, std::min(blocks, cap));
}

static void gauss_seidel(Ctx& c, DCsr& A, const double* b, double* x, const SolveParams& sp) {
    if (sp.gs_mode == ORC_GS_REFERENCE_PANIC) throw Error(ORC_E_GS_MAINTENANCE, "Gauss-Seidel out for maintenance :)");
    const int n = (int)A.nrows;
    if (n == 0) return;
    csr_ensure_diag(c, A);
    const double w = sp.relaxation, omw = 1. - sp.relaxation;
    if (sp.gs_mode == ORC_GS_MULTICOLOUR) {
        // a one-sided entry (i stores j, j does not store i) could give i and j one colour, and one sweep would then write x_j
        // while another row of the colour reads it
        csr_check_symmetry(c, A);
        ORC_REQUIRE(A.sym == 1, ORC_E_UNSUPPORTED,
                    "multicolour Gauss-Seidel needs a structurally symmetric pattern ((i, j) stored exactly when (j, i) is stored)");
        DBuf<int> colour(&c, n), coloured_in(&c, n), st(&c, 2);
        ORC_CUDA(cudaMemsetAsync(coloured_in.p, 0xff, sizeof(int) * (size_t)n, c.stream));
        int ncol = 0;
        for (int round = 0;; ++round) {
            // every round colours at least the lowest uncoloured row
            ORC_REQUIRE(round < n, ORC_E_INTERNAL, "multicolour GS: colouring did not terminate");
            st.zero();
            k_colour_round<<<(n + 255) / 256, 256, 0, c.stream>>>(n, A.rowptr, A.col, colour, coloured_in, round, st);
            c.after_launch("k_colour_round");
            int h[2] = {0, 0};
            st.download(h);
            c.sync();
            ncol = std::max(ncol, h[1]);
            if (h[0] == 0) break;
        }
        for (uint64_t it = 0; it < sp.iterations; ++it)
            for (int q = 0; q < ncol; ++q) {
                k_gs_colour<<<(n + 255) / 256, 256, 0, c.stream>>>(n, A.rowptr, A.col, A.val, A.diag, b, x, w, omw, colour, q, c.d_flags);
                c.after_launch("k_gs_colour");
            }
        return;
    }
    csr_check_symmetry(c, A);
    if (A.sym != 1) {  // the dataflow sweep needs (i,j) stored <=> (j,i) stored; otherwise walk the rows serially
        for (uint64_t it = 0; it < sp.iterations; ++it) {
            k_gs_serial<<<1, 32, 0, c.stream>>>(n, A.rowptr, A.col, A.val, A.diag, b, x, w, omw, c.d_flags);
            c.after_launch("k_gs_serial");
        }
        return;
    }
    if (gs_small_ok(c, A, sp.iterations)) {  // all sweeps in one launch, ready flags in shared memory (small.cu)
        gauss_seidel_small(c, A, b, x, w, omw, sp.iterations);
        return;
    }
    DBuf<int> done(&c, n);
    DBuf<unsigned int> ticket(&c, 1);
    done.zero();
    const int nchunks = (n + DF_CHUNK - 1) / DF_CHUNK;
    for (uint64_t it = 0; it < sp.iterations; ++it) {
        ticket.zero();
        k_gs_sweep<<<dataflow_grid(c, nchunks, 8), 256, 0, c.stream>>>(n, A.rowptr, A.col, A.val, A.diag, b, x, w, omw, done, (int)it + 1,
                                                                         ticket, c.d_flags);
        c.after_launch("k_gs_sweep");
    }
}

// =================================================================================================
// build_restriction_matrix, "Strongest" (linear_algebra.rs:30-60) — a sequential greedy in the reference:
// row i picks argmin a_ij over stored j != i that no earlier row has picked (strict <, first minimum
// wins, start value f64::MAX), then marks j as combined. Pushes (i/2, i, 1) and (i/2, j, 1).
//
// Exact parallelisation (bit-identical aggregates) as a sync-free dataflow kernel. Row i evaluates its best
// candidate j* among the columns that are not combined yet, and may commit to it as soon as every row k < i
// that also stores column j* ("lower toucher") has decided — for a structurally symmetric matrix those rows are
// the entries k < i, k != j* of row j*, so the wait is one parallel scan of `decided[]` over row j*.
// Why this is the sequential answer: a row k > i can only take a column of row i after i itself has decided
// (i is a lower toucher of that column), so every column seen as combined was taken by a row < i; columns are
// never un-combined, so everything that beat j* stays unavailable; and once all lower touchers of j* have
// decided without taking it, nobody below i ever will. If j* was taken while waiting, the row re-evaluates.
// Only the chain through the best candidate is waited on. Rows are handed out in chunks through an atomic
// ticket, so every row a warp can wait on is already owned by a resident warp (forward progress).
// =================================================================================================
// `state[k]`: 0 = row k undecided, 1 = decided without a pick, 2 + j = decided and picked column j. Flag and payload
// share one word, so a single store publishes the decision and a single load observes it: no fences on the critical
// path (one L2 round trip per dependency hop). `combined[]` is only a monotone hint for the candidate scan.
constexpr int DFR_WARPS = 8;     // warps per block of the restriction kernel
constexpr int DFR_SM_BLOCKS = 8;   // resident blocks per SM: 8 warps x 8 blocks = 2048 threads, a full SM
// Ticket shape: rows a warp handles ONE AFTER THE OTHER per block ticket (a ticket covers WARPS * rows consecutive rows). A row that
// waits for its warp has not even issued its loads when the row it depends on decides; with more than one row per warp the front of
// a dependency chain therefore pays a whole row latency every WARPS rows instead of one flag round trip per hop
// (scripts/lab/restriction_sim.py: 50 ns per row with 4, 0.6 ns with 1 on a 150 x 150 x 3 tet slab). Measured
// (profiles/r2_restriction_rows.txt): Kuhn-split tets are chain bound — one row per warp is up to 60 x faster (slab: 1053 -> 17.5 ms
// per hierarchy); the hex boxes are throughput bound — four rows per warp are 1.6 x faster (5.2 vs 8.3 ms), because a block whose
// warps hold one row each idles until its slowest row is done. The aggregates do not depend on the shape. The rule: hierarchies of
// simplex meshes (fine-matrix rows of <= 5 entries; DCsr::simplex is inherited by every matrix derived from the fine one) take one
// row per warp, everything else four; the one-block kernel for small systems always takes four. (A tuner that timed both shapes on
// the first builds was tried and dropped: the momentum and the pressure matrix of a size prefer different shapes and the first
// iterations are not representative, so it cost the hex bench 6-27 ms per iteration.)
static int dfr_rows_for(Ctx& c, DCsr& A) {
    if (A.simplex < 0) { csr_ensure_max_row(c, A); A.simplex = (A.max_row <= 5) ? 1 : 0; }
    return A.simplex == 1 ? 1 : 4;
}
// The body is shared by the grid-wide kernel (state in global memory: one L2 round trip per dependency hop) and the one-block
// kernel for small systems (state in shared memory: ~30 cycles per hop; on the reference's 2-D meshes the hops form one long chain).
template <int WARPS>
__device__ __forceinline__ void strongest_dataflow_body(int n, const int* __restrict__ rowptr, const int* __restrict__ col,
                                                        const double* __restrict__ val, int* state, int* combined, int* pick, int* picked_by,
                                                        unsigned int* ticket, int* flags, unsigned int* s_chunk_p, int rows_per_warp) {
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int BCH = WARPS * rows_per_warp;
    const int nchunks = (n + BCH - 1) / BCH;
    for (;;) {
        __syncthreads();
        if (threadIdx.x == 0) *s_chunk_p = atomicAdd(ticket, 1u);
        __syncthreads();
        const unsigned int chunk = *s_chunk_p;
        if ((int)chunk >= nchunks) return;
        const int r0 = chunk * BCH;
        // consecutive rows (which usually depend on each other) go to different warps, so that their loads overlap
        for (int i = r0 + wib; i < min(n, r0 + BCH); i += WARPS) {
            const int lo = rowptr[i], hi = rowptr[i + 1];
            int chosen = -1;
            bool give_up = false;
            // Rows of up to 32 entries (the fine level and the first coarse level) live in registers, one entry per lane, together
            // with the row bounds of the entry's column (the candidate's row is needed right after the choice): a row costs five
            // dependent memory latencies instead of eight, a retry one (the refreshed `combined` hints).
            const bool in_regs = (hi - lo) <= 32;
            int e_j = -1, e_lo = 0, e_hi = 0;
            double e_v = 0.;
            bool e_free = false;
            if (in_regs && lo + lane < hi) {
                e_j = col[lo + lane];
                e_v = val[lo + lane];
                e_free = (e_j != i);
                if (e_free) { e_lo = rowptr[e_j]; e_hi = rowptr[e_j + 1]; }
            }
            for (;;) {
                double best = DBL_MAX;   // strongest_coeff starts at Float::MAX
                int best_k = INT_MAX;    // position in the row: the FIRST minimum wins
                if (in_regs) {
                    if (e_free && *(volatile int*)(combined + e_j) != 0) e_free = false;
                    if (e_free) { best = e_v; best_k = lo + lane; }
                } else {
                    for (int k = lo + lane; k < hi; k += 32) {
                        const int j = col[k];
                        const double v = val[k];   // loaded alongside the column, not behind the `combined` check
                        if (j != i && *(volatile int*)(combined + j) == 0) {
                            if (v < best) { best = v; best_k = k; }  // a lane sees ascending k, so ties keep the first
                        }
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {  // warp argmin on (value, position)
                    double ov = __shfl_down_sync(0xffffffffu, best, o);
                    int ok = __shfl_down_sync(0xffffffffu, best_k, o);
                    if (ok != INT_MAX && (best_k == INT_MAX || ov < best || (ov == best && ok < best_k))) { best = ov; best_k = ok; }
                }
                best_k = __shfl_sync(0xffffffffu, best_k, 0);
                if (best_k == INT_MAX) break;  // nothing available: row i pushes nothing
                int j, jlo, jhi;
                if (in_regs) {
                    const int src = best_k - lo;   // the lane that holds the winning entry
                    j = __shfl_sync(0xffffffffu, e_j, src);
                    jlo = __shfl_sync(0xffffffffu, e_lo, src);
                    jhi = __shfl_sync(0xffffffffu, e_hi, src);
                } else {
                    j = col[best_k];
                    jlo = rowptr[j]; jhi = rowptr[j + 1];
                }
                // every row that can take j before row i is a LOWER TOUCHER of j: a row k < i, k != j stored in row j
                // (structural symmetry). Wait for their decisions and see whether one of them picked j.
                // The warp polls all of them together and stops as soon as ONE of them reports "picked j": a taken candidate needs
                // nothing from the other lower touchers, and waiting for those as well would make row i depend on rows that have
                // no say in its decision (on the Kuhn-split tet slabs of the 8-GPU runs those extra waits chained every row to the
                // previous one: 290 ns per row, 750 ms per restriction matrix).
                int taken = 0, bad = 0;
                for (int base = jlo; base < jhi && !taken; base += 32) {
                    const int kk = base + lane;
                    int k = INT_MAX;
                    if (kk < jhi) k = col[kk];
                    const bool mine = (k < i && k != j);
                    long long spins = 0;
                    for (;;) {
                        int st = 1;
                        if (mine) st = *(volatile const int*)(state + k);
                        const unsigned int took = __ballot_sync(0xffffffffu, mine && st == 2 + j);
                        const unsigned int pending = __ballot_sync(0xffffffffu, mine && st == 0);
                        if (took) { taken = 1; break; }
                        if (!pending) break;
                        if ((++spins & 1023) == 0) {
                            int stop = 0;
                            if (spins > SPIN_LIMIT) { atomicOr(flags, DF_SPIN); stop = 1; }
                            else if (*(volatile int*)flags & DF_SPIN) stop = 1;
                            if (__any_sync(0xffffffffu, stop)) { bad = 1; break; }
                        }
                    }
                    if (bad) break;
                    if (__any_sync(0xffffffffu, k >= i)) break;
                }
                if (bad) { give_up = true; break; }
                if (!taken) { chosen = j; break; }
                if (lane == 0) *(volatile int*)(combined + j) = 1;  // make the hint visible to this warp's next scan
                if (in_regs && e_j == j) e_free = false;
                __syncwarp();
            }
            if (lane == 0) {
                if (chosen >= 0) {
                    *(volatile int*)(combined + chosen) = 1;
                    picked_by[chosen] = i;
                }
                pick[i] = chosen;
                *(volatile int*)(state + i) = (chosen >= 0 && !give_up) ? 2 + chosen : 1;
            }
            __syncwarp();
        }
    }
}
__global__ void __launch_bounds__(DFR_WARPS * 32) k_strongest_dataflow(int n, const int* __restrict__ rowptr, const int* __restrict__ col,
                                                                       const double* __restrict__ val, int* state, int* combined, int* pick,
                                                                       int* picked_by, unsigned int* ticket, int* flags, int rows_per_warp) {
    __shared__ unsigned int s_chunk;
    strongest_dataflow_body<DFR_WARPS>(n, rowptr, col, val, state, combined, pick, picked_by, ticket, flags, &s_chunk, rows_per_warp);
}
// one block, `state` and `combined` in shared memory (2 n ints): systems of up to kStrongestSmallRows rows
constexpr int kStrongestSmallRows = 24576;
__global__ void __launch_bounds__(1024, 1) k_strongest_small(int n, const int* __restrict__ rowptr, const int* __restrict__ col,
                                                             const double* __restrict__ val, int* pick, int* picked_by, int* flags, int rows_per_warp) {
    extern __shared__ int sm_state[];
    __shared__ unsigned int s_chunk, s_ticket;
    int* state = sm_state;
    int* combined = sm_state + n;
    for (int i = threadIdx.x; i < 2 * n; i += blockDim.x) sm_state[i] = 0;
    if (threadIdx.x == 0) s_ticket = 0u;
    __syncthreads();
    strongest_dataflow_body<32>(n, rowptr, col, val, state, combined, pick, picked_by, &s_ticket, flags, &s_chunk, rows_per_warp);
}
__global__ void k_strongest_serial(int n, const int* rowptr, const int* col, const double* val, int* combined, int* pick, int* picked_by) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    for (int i = 0; i < n; ++i) {
        double best = DBL_MAX;
        int bj = -1;
        for (int k = rowptr[i]; k < rowptr[i + 1]; ++k) {
            int j = col[k];
            if (combined[j] || j == i) continue;
            if (val[k] < best) { best = val[k]; bj = j; }
        }
        pick[i] = bj;
        if (bj >= 0) { combined[bj] = 1; picked_by[bj] = i; }
    }
}
// R row I collects the pushes of fine rows 2I and 2I+1; CsrMatrix::from(&Coo) sorts columns and sums duplicates.
__device__ __forceinline__ int restriction_row(int I, int nfine, const int* pick, int* cols, double* vals) {
    int m = 0;
    for (int i = 2 * I; i < 2 * I + 2 && i < nfine; ++i) {
        int pj = pick[i];
        if (pj < 0) continue;
        int cand[2] = {i, pj};
        for (int q = 0; q < 2; ++q) {
            int cc = cand[q], pos = 0;
            while (pos < m && cols[pos] < cc) ++pos;
            if (pos < m && cols[pos] == cc) { vals[pos] = vals[pos] + 1.0; continue; }
            for (int s = m; s > pos; --s) { cols[s] = cols[s - 1]; vals[s] = vals[s - 1]; }
            cols[pos] = cc; vals[pos] = 1.0; ++m;
        }
    }
    return m;
}
__global__ void k_restriction_counts(int ncoarse, int nfine, const int* pick, const int* picked_by, int* cnt_r, int* cnt_rt) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < ncoarse) {
        int cols[4]; double vals[4];
        cnt_r[t] = restriction_row(t, nfine, pick, cols, vals);
    }
    if (t < nfine) {
        int a = pick[t] >= 0 ? t / 2 : -1;
        int b = picked_by[t] >= 0 ? picked_by[t] / 2 : -1;
        cnt_rt[t] = (a >= 0) + (b >= 0) - ((a >= 0 && a == b) ? 1 : 0);
    }
}
__global__ void k_restriction_fill(int ncoarse, int nfine, const int* pick, const int* picked_by, const int* rp_r, int* col_r,
                                   double* val_r, const int* rp_rt, int* col_rt, double* val_rt) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t < ncoarse) {
        int cols[4]; double vals[4];
        int m = restriction_row(t, nfine, pick, cols, vals);
        int o = rp_r[t];
        for (int q = 0; q < m; ++q) { col_r[o + q] = cols[q]; val_r[o + q] = vals[q]; }
    }
    if (t < nfine) {  // R^T row t: transpose() keeps the summed values, columns sorted
        int a = pick[t] >= 0 ? t / 2 : -1;
        int b = picked_by[t] >= 0 ? picked_by[t] / 2 : -1;
        int o = rp_rt[t];
        if (a >= 0 && a == b) { col_rt[o] = a; val_rt[o] = 2.0; }
        else {
            int lo = (a >= 0 && (b < 0 || a < b)) ? a : b;
            int hi2 = (lo == a) ? b : a;
            if (lo >= 0) { col_rt[o] = lo; val_rt[o++] = 1.0; }
            if (hi2 >= 0) { col_rt[o] = hi2; val_rt[o] = 1.0; }
        }
    }
}

CsrPtr build_restriction(Ctx& c, DCsr& A, int method, CsrPtr* rt_out) {
    ORC_REQUIRE(A.nrows == A.ncols, ORC_E_INVALID, "build_restriction: matrix must be square");
    const int n = (int)A.ncols;
    const int nc = n / 2 + n % 2;
    DBuf<int> pick(&c, std::max(n, 1)), picked_by(&c, std::max(n, 1));
    ORC_CUDA(cudaMemsetAsync(picked_by.p, 0xff, sizeof(int) * (size_t)std::max(n, 1), c.stream));
    if (method == ORC_RESTRICT_INJECTION) {
        // R = [1 1 0 0 ..; 0 0 1 1 ..]: build directly as a CSR with two entries per row
        CsrPtr R = csr_alloc(c, nc, n, n);
        std::vector<int> rp(nc + 1), cl(std::max(n, 1));
        std::vector<double> vl(std::max(n, 1), 1.0);
        for (int r = 0; r <= nc; ++r) rp[r] = std::min(2 * r, n);
        for (int k = 0; k < n; ++k) cl[k] = k;
        ORC_CUDA(cudaMemcpyAsync(R->rowptr, rp.data(), sizeof(int) * (nc + 1), cudaMemcpyHostToDevice, c.stream));
        ORC_CUDA(cudaMemcpyAsync(R->col, cl.data(), sizeof(int) * std::max(n, 1), cudaMemcpyHostToDevice, c.stream));
        ORC_CUDA(cudaMemcpyAsync(R->val, vl.data(), sizeof(double) * std::max(n, 1), cudaMemcpyHostToDevice, c.stream));
        if (rt_out) {
            CsrPtr RT = csr_alloc(c, n, nc, n);
            std::vector<int> rpt(n + 1), clt(std::max(n, 1));
            for (int k = 0; k <= n; ++k) rpt[k] = k;
            for (int k = 0; k < n; ++k) clt[k] = k / 2;
            ORC_CUDA(cudaMemcpyAsync(RT->rowptr, rpt.data(), sizeof(int) * (n + 1), cudaMemcpyHostToDevice, c.stream));
            ORC_CUDA(cudaMemcpyAsync(RT->col, clt.data(), sizeof(int) * std::max(n, 1), cudaMemcpyHostToDevice, c.stream));
            ORC_CUDA(cudaMemcpyAsync(RT->val, vl.data(), sizeof(double) * std::max(n, 1), cudaMemcpyHostToDevice, c.stream));
            *rt_out = std::move(RT);
        }
        c.sync();
        return R;
    }
    ORC_REQUIRE(method == ORC_RESTRICT_STRONGEST, ORC_E_INVALID, "unknown restriction method");
    if (n > 0) {
        csr_check_symmetry(c, A);
        csr_ensure_max_row(c, A);
        DBuf<int> combined(&c, n);
        combined.zero();
        if (A.sym == 1 && n <= kStrongestSmallRows && small_enabled()) {
            static bool attr_set = false;
            if (!attr_set) {
                ORC_CUDA(cudaFuncSetAttribute(k_strongest_small, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(2 * kStrongestSmallRows * sizeof(int))));
                attr_set = true;
            }
            k_strongest_small<<<1, 1024, 2 * (size_t)n * sizeof(int), c.stream>>>(n, A.rowptr, A.col, A.val, pick, picked_by, c.d_flags, 4);
            c.after_launch("k_strongest_small");
        } else if (A.sym == 1) {
            DBuf<int> decided(&c, n);
            DBuf<unsigned int> ticket(&c, 1);
            decided.zero();
            ticket.zero();
            const int rows = dfr_rows_for(c, A);
            const int nchunks = (n + DFR_WARPS * rows - 1) / (DFR_WARPS * rows);
            k_strongest_dataflow<<<std::max(1, std::min(nchunks, c.sm_count * DFR_SM_BLOCKS)), DFR_WARPS * 32, 0, c.stream>>>(
                n, A.rowptr, A.col, A.val, decided, combined, pick, picked_by, ticket, c.d_flags, rows);
            c.after_launch("k_strongest_dataflow");
        } else {
            k_strongest_serial<<<1, 32, 0, c.stream>>>(n, A.rowptr, A.col, A.val, combined, pick, picked_by);
            c.after_launch("k_strongest_serial");
        }
    }
    DBuf<int> cnt_r(&c, (size_t)nc + 1), cnt_rt(&c, (size_t)n + 1), rp_r(&c, (size_t)nc + 1), rp_rt(&c, (size_t)n + 1);
    cnt_r.zero();
    cnt_rt.zero();
    if (n > 0) {
        k_restriction_counts<<<(n + 255) / 256, 256, 0, c.stream>>>(nc, n, pick, picked_by, cnt_r, cnt_rt);
        c.after_launch("k_restriction_counts");
    }
    exclusive_scan_to_rowptr(c, cnt_r, rp_r, nc);
    exclusive_scan_to_rowptr(c, cnt_rt, rp_rt, n);
    int nnz_r = 0, nnz_rt = 0;
    ORC_CUDA(cudaMemcpyAsync(&nnz_r, rp_r.p + nc, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    ORC_CUDA(cudaMemcpyAsync(&nnz_rt, rp_rt.p + n, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    CsrPtr R = csr_alloc(c, nc, n, nnz_r), RT = csr_alloc(c, n, nc, nnz_rt);
    ORC_CUDA(cudaMemcpyAsync(R->rowptr, rp_r.p, sizeof(int) * ((size_t)nc + 1), cudaMemcpyDeviceToDevice, c.stream));
    ORC_CUDA(cudaMemcpyAsync(RT->rowptr, rp_rt.p, sizeof(int) * ((size_t)n + 1), cudaMemcpyDeviceToDevice, c.stream));
    if (n > 0) {
        k_restriction_fill<<<(n + 255) / 256, 256, 0, c.stream>>>(nc, n, pick, picked_by, R->rowptr, R->col, R->val, RT->rowptr, RT->col, RT->val);
        c.after_launch("k_restriction_fill");
    }
    if (rt_out) *rt_out = std::move(RT);
    return R;
}

// =================================================================================================
// SpGEMM with nalgebra-sparse semantics (&Csr * &Csr): pattern = symbolic union of the B rows selected
// by A's row (nothing dropped, sorted); values c_ij = 0; for k ascending over row i of A:
// for j over row k of B: c_ij += (1 * a_ik) * b_kj.
//
// One warp per output row, one pass: every contribution (column j, term (1*a_ik)*b_kj) is gathered in
// k-major order, the warp sorts 64-bit keys (j << 32 | gather position) with a bitonic network in shared
// memory, and each distinct column then sums its run of terms IN KEY ORDER — i.e. in ascending k, the
// reference's accumulation order, so values are bit-identical without any search or atomics. Rows are
// written behind an upper-bound offset (sum of the selected B-row lengths) and compacted afterwards.
// =================================================================================================
constexpr int SG_WARPS = 4;
constexpr int SG_CAP = 512;  // contributions per warp held in shared memory (20 B each)

// maxcand[0] = longest candidate row; (maxcand[2], maxcand[3]) = 64-bit total of all candidates: the 32-bit scan that follows
// wraps silently once the total passes 2^32, so the callers check this total (x their expansion factor) against INT32_MAX.
__global__ void k_spgemm_cand(int n, const int* __restrict__ arp, const int* __restrict__ acol, const int* __restrict__ brp, int* cand,
                              int* maxcand) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    int tot = 0;
    if (i < n)
        for (int ka = arp[i]; ka < arp[i + 1]; ++ka) tot += brp[acol[ka] + 1] - brp[acol[ka]];
    if (i < n) cand[i] = tot;
    int m = tot;
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_down_sync(0xffffffffu, m, o));
    unsigned long long s = (unsigned long long)tot;
    for (int o = 16; o > 0; o >>= 1) s += __shfl_down_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0 && m > 0) {
        atomicMax(maxcand, m);
        atomicAdd(reinterpret_cast<unsigned long long*>(maxcand + 2), s);
    }
}

// Bitonic sort of P = 32 * NK keys held in registers (element r * 32 + lane lives in register r of `lane`): exchanges over a
// distance < 32 are warp shuffles, longer ones stay inside the thread. About a quarter of the instructions of the
// shared-memory network below (the Galerkin kernels are issue bound, not memory bound).
template <int NK, class KeyT>
__device__ __forceinline__ void warp_bitonic_sort_regs(KeyT (&key)[NK], int lane) {
#pragma unroll
    for (int k = 2; k <= 32 * NK; k <<= 1) {
#pragma unroll
        for (int j = k >> 1; j > 0; j >>= 1) {
            if (j >= 32) {
#pragma unroll
                for (int r = 0; r < NK; ++r) {
                    const int pr = r ^ (j >> 5);
                    if (pr > r) {
                        const bool up = (((r << 5) | lane) & k) == 0;
                        const KeyT a = key[r], b = key[pr];
                        if ((a > b) == up) { key[r] = b; key[pr] = a; }
                    }
                }
            } else {
#pragma unroll
                for (int r = 0; r < NK; ++r) {
                    const KeyT mine = key[r];
                    const KeyT other = __shfl_xor_sync(0xffffffffu, mine, j);
                    const bool up = (((r << 5) | lane) & k) == 0;
                    const bool lower = (lane & j) == 0;   // this element is the lower index of the pair
                    const bool take_min = (lower == up);
                    key[r] = take_min ? (mine < other ? mine : other) : (mine > other ? mine : other);
                }
            }
        }
    }
}
// buf[0 .. P) (P a power of two, 32 <= P <= 1024, padded with all-ones keys by the caller) sorted through registers
template <int NK, class KeyT>
__device__ __forceinline__ void warp_sort_via_regs(KeyT* buf, int lane) {
    KeyT key[NK];
#pragma unroll
    for (int r = 0; r < NK; ++r) key[r] = buf[r * 32 + lane];
    warp_bitonic_sort_regs<NK, KeyT>(key, lane);
#pragma unroll
    for (int r = 0; r < NK; ++r) buf[r * 32 + lane] = key[r];
    __syncwarp();
}
template <int PMAX, class KeyT>   // PMAX: largest P the caller can ask for (keeps the register footprint of short-row instantiations small)
__device__ __forceinline__ void warp_sort_keys(KeyT* buf, int P, int lane) {
    if (P == 32) { warp_sort_via_regs<1, KeyT>(buf, lane); return; }
    if constexpr (PMAX >= 64) { if (P == 64) { warp_sort_via_regs<2, KeyT>(buf, lane); return; } }
    if constexpr (PMAX >= 128) { if (P == 128) { warp_sort_via_regs<4, KeyT>(buf, lane); return; } }
    if constexpr (PMAX >= 256) { if (P == 256) { warp_sort_via_regs<8, KeyT>(buf, lane); return; } }
    if constexpr (PMAX >= 512) { if (P == 512) { warp_sort_via_regs<16, KeyT>(buf, lane); return; } }
    if constexpr (PMAX >= 1024) { if (P == 1024) { warp_sort_via_regs<32, KeyT>(buf, lane); return; } }
}
__device__ __forceinline__ void warp_bitonic_sort64(unsigned long long* buf, int P, int lane) {
    for (int k = 2; k <= P; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int idx = lane; idx < P; idx += 32) {
                int partner = idx ^ j;
                if (partner > idx) {
                    unsigned long long a = buf[idx], b = buf[partner];
                    bool up = (idx & k) == 0;
                    if ((a > b) == up) { buf[idx] = b; buf[partner] = a; }
                }
            }
            __syncwarp();
        }
}

__global__ void __launch_bounds__(SG_WARPS * 32) k_spgemm_rows(int n, const int* __restrict__ arp, const int* __restrict__ acol,
                                                               const double* __restrict__ aval, const int* __restrict__ brp,
                                                               const int* __restrict__ bcol, const double* __restrict__ bval,
                                                               const int* __restrict__ candptr, int* counts, int* tcol, double* tval,
                                                               unsigned long long* scratch_keys, double* scratch_vals, int* scratch_heads,
                                                               int scratch_stride) {
    __shared__ unsigned long long skeys[SG_WARPS][SG_CAP];
    __shared__ double svals[SG_WARPS][SG_CAP];
    __shared__ int sheads[SG_WARPS][SG_CAP];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int warp = blockIdx.x * SG_WARPS + wib, nwarps = gridDim.x * SG_WARPS;
    for (int i = warp; i < n; i += nwarps) {
        const int c0 = candptr[i];
        const int tot = candptr[i + 1] - c0;
        int P = 1;
        while (P < tot) P <<= 1;
        const bool in_smem = (P <= SG_CAP);
        unsigned long long* keys = in_smem ? skeys[wib] : scratch_keys + (size_t)warp * scratch_stride;
        double* vals = in_smem ? svals[wib] : scratch_vals + (size_t)warp * scratch_stride;
        int* heads = in_smem ? sheads[wib] : scratch_heads + (size_t)warp * scratch_stride;
        const int alo = arp[i], ahi = arp[i + 1];
        // ---- gather in k-major order ----
        if ((ahi - alo) <= 8) {  // R*A: few, long B rows -> lanes across a B row
            int off = 0;
            for (int ka = alo; ka < ahi; ++ka) {
                const int k = acol[ka];
                const double alpha_aik = 1. * aval[ka];
                const int bb = brp[k], len = brp[k + 1] - bb;
                for (int q = lane; q < len; q += 32) {
                    keys[off + q] = ((unsigned long long)(unsigned int)bcol[bb + q] << 32) | (unsigned int)(off + q);
                    vals[off + q] = alpha_aik * bval[bb + q];
                }
                off += len;
            }
        } else {  // (RA)*R^T: many, short B rows -> lanes across A's row behind a warp prefix sum
            int off = 0;
            for (int base = alo; base < ahi; base += 32) {
                const int ka = base + lane;
                int len = 0, bb = 0;
                double alpha_aik = 0.;
                if (ka < ahi) { const int k = acol[ka]; bb = brp[k]; len = brp[k + 1] - bb; alpha_aik = 1. * aval[ka]; }
                int incl = len;
                for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
                const int my = off + incl - len;
                for (int q = 0; q < len; ++q) {
                    keys[my + q] = ((unsigned long long)(unsigned int)bcol[bb + q] << 32) | (unsigned int)(my + q);
                    vals[my + q] = alpha_aik * bval[bb + q];
                }
                off += __shfl_sync(0xffffffffu, incl, 31);
            }
        }
        for (int idx = tot + lane; idx < P; idx += 32) keys[idx] = ~0ull;
        __syncwarp();
        warp_bitonic_sort64(keys, P, lane);
        // ---- run heads (distinct columns), in order ----
        int nuniq = 0;
        for (int base = 0; base < tot; base += 32) {
            const int idx = base + lane;
            bool head = false;
            if (idx < tot) head = (idx == 0) || ((keys[idx - 1] >> 32) != (keys[idx] >> 32));
            const unsigned int mask = __ballot_sync(0xffffffffu, head);
            if (head) heads[nuniq + __popc(mask & ((1u << lane) - 1u))] = idx;
            nuniq += __popc(mask);
        }
        __syncwarp();
        // ---- each distinct column sums its run in key order == ascending k ----
        for (int q = lane; q < nuniq; q += 32) {
            const int b = heads[q], e = (q + 1 < nuniq) ? heads[q + 1] : tot;
            double acc = 0. * 0.;
            for (int idx = b; idx < e; ++idx) acc += vals[(unsigned int)(keys[idx] & 0xffffffffull)];
            tcol[c0 + q] = (int)(keys[b] >> 32);
            tval[c0 + q] = acc;
        }
        if (lane == 0) counts[i] = nuniq;
        __syncwarp();
    }
}
__global__ void k_spgemm_compact(int n, const int* __restrict__ candptr, const int* __restrict__ crp, const int* __restrict__ tcol,
                                 const double* __restrict__ tval, int* ccol, double* cval) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int i = warp; i < n; i += nwarps) {
        const int s = candptr[i], d = crp[i], len = crp[i + 1] - d;
        for (int q = lane; q < len; q += 32) { ccol[d + q] = tcol[s + q]; cval[d + q] = tval[s + q]; }
    }
}

CsrPtr spgemm(Ctx& c, const DCsr& A, const DCsr& B) {
    ORC_REQUIRE(A.ncols == B.nrows, ORC_E_INVALID, "spgemm: dimension mismatch");
    const int n = (int)A.nrows;
    DBuf<int> cand(&c, (size_t)n + 1), candptr(&c, (size_t)n + 1), counts(&c, (size_t)n + 1), rp(&c, (size_t)n + 1), maxc(&c, 4);
    cand.zero();
    counts.zero();
    maxc.zero();
    int hmax = 0, htot = 0;
    int hm4[4] = {0, 0, 0, 0};
    if (n > 0) {
        k_spgemm_cand<<<(n + 255) / 256, 256, 0, c.stream>>>(n, A.rowptr, A.col, B.rowptr, cand, maxc);
        c.after_launch("k_spgemm_cand");
    }
    exclusive_scan_to_rowptr(c, cand, candptr, n);
    maxc.download(hm4);
    ORC_CUDA(cudaMemcpyAsync(&htot, candptr.p + n, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    hmax = hm4[0];
    unsigned long long tot64 = 0;
    memcpy(&tot64, hm4 + 2, sizeof(tot64));
    ORC_REQUIRE(tot64 <= (unsigned long long)INT32_MAX, ORC_E_INVALID, "spgemm: intermediate product exceeds 2^31 entries");
    const int grid = std::max(1, std::min((n + SG_WARPS - 1) / SG_WARPS, c.sm_count * 8));
    DBuf<unsigned long long> skeys;
    DBuf<double> svals;
    DBuf<int> sheads;
    int stride = 0;
    if (hmax > SG_CAP) {
        stride = 1;
        while (stride < hmax) stride <<= 1;
        const size_t tot = (size_t)grid * SG_WARPS * stride;
        skeys.alloc(&c, tot); svals.alloc(&c, tot); sheads.alloc(&c, tot);
    }
    DBuf<int> tcol(&c, (size_t)std::max(htot, 1));
    DBuf<double> tval(&c, (size_t)std::max(htot, 1));
    if (n > 0) {
        k_spgemm_rows<<<grid, SG_WARPS * 32, 0, c.stream>>>(n, A.rowptr, A.col, A.val, B.rowptr, B.col, B.val, candptr, counts, tcol, tval,
                                                            skeys.p, svals.p, sheads.p, stride);
        c.after_launch("k_spgemm_rows");
    }
    exclusive_scan_to_rowptr(c, counts, rp, n);
    int nnz = 0;
    ORC_CUDA(cudaMemcpyAsync(&nnz, rp.p + n, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    CsrPtr C = csr_alloc(c, A.nrows, B.ncols, nnz);
    ORC_CUDA(cudaMemcpyAsync(C->rowptr, rp.p, sizeof(int) * ((size_t)n + 1), cudaMemcpyDeviceToDevice, c.stream));
    if (n > 0 && nnz > 0) {
        k_spgemm_compact<<<std::max(1, std::min((n + 7) / 8, c.sm_count * 8)), 256, 0, c.stream>>>(n, candptr, C->rowptr, tcol, tval, C->col, C->val);
        c.after_launch("k_spgemm_compact");
    }
    return C;
}

// ---- fused Galerkin triple product: (R*A)*R^T for one coarse row per warp, the intermediate row of R*A never leaves shared
// memory. Both products keep nalgebra's semantics (symbolic-union pattern, terms summed in ascending k): phase 1 sorts the
// terms (1*r_Ii)*a_ij by (j, gather position) and sums each run -> row I of R*A; phase 2 expands every (j, v) of that row
// through row j of R^T (at most two entries), sorts by (J, position) and sums each run -> row I of R*A*R^T. ----
constexpr int GK_WARPS = 4;
// CAP1 = phase-1 term limit per row (template parameter, picked from the longest row of the launch so that short-row
// levels keep a high occupancy); phase 2 can produce up to twice as many terms.
// shared memory per warp: keys and values for up to 2 * cap1 terms, run heads (16 bit), the cap1-entry row of R*A
template <class KeyT>
constexpr size_t gk_smem_per_warp(int cap1) { return (size_t)(2 * cap1) * (sizeof(KeyT) + 8 + 2) + (size_t)cap1 * (4 + 8); }
constexpr int gk_log2(int v) { int b = 0; while ((1 << b) < v) ++b; return b; }

// Keys are (column << POSB) | gather position, POSB = log2(2 * CAP1). KeyT = 32 bit whenever the columns fit into 32 - POSB bits
// (every level of the meshes here: half the shuffles and half the key memory), 64 bit otherwise.
template <class KeyT, int POSB>
__device__ __forceinline__ int warp_runs(const KeyT* keys, int tot, unsigned short* heads, int lane) {
    int nuniq = 0;
    for (int base = 0; base < tot; base += 32) {
        const int idx = base + lane;
        bool head = false;
        if (idx < tot) head = (idx == 0) || ((keys[idx - 1] >> POSB) != (keys[idx] >> POSB));
        const unsigned int mask = __ballot_sync(0xffffffffu, head);
        if (head) heads[nuniq + __popc(mask & ((1u << lane) - 1u))] = (unsigned short)idx;
        nuniq += __popc(mask);
    }
    __syncwarp();
    return nuniq;
}

template <int GK_CAP1, class KeyT>
__global__ void __launch_bounds__(GK_WARPS * 32) k_galerkin_rows(int nc, const int* __restrict__ rrp, const int* __restrict__ rcol,
                                                                 const double* __restrict__ rval, const int* __restrict__ arp,
                                                                 const int* __restrict__ acol, const double* __restrict__ aval,
                                                                 const int* __restrict__ trp, const int* __restrict__ tcol_,
                                                                 const double* __restrict__ tval_, const int* __restrict__ outptr, int* counts,
                                                                 int* ocol, double* oval, int* maxrow) {
    extern __shared__ __align__(16) unsigned char gk_smem[];
    constexpr int GK_CAP = 2 * GK_CAP1, POSB = gk_log2(GK_CAP);
    constexpr KeyT POSMASK = (KeyT)((1u << POSB) - 1u), SENTINEL = (KeyT)~(KeyT)0;
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    unsigned char* base_ptr = gk_smem + (size_t)wib * gk_smem_per_warp<KeyT>(GK_CAP1);
    double* vals = reinterpret_cast<double*>(base_ptr);                                    // 2 CAP1 doubles
    double* ra_val = vals + GK_CAP;                                                        // CAP1 doubles
    KeyT* keys = reinterpret_cast<KeyT*>(ra_val + GK_CAP1);                                // 2 CAP1 keys
    int* ra_col = reinterpret_cast<int*>(keys + GK_CAP);                                   // CAP1 ints
    unsigned short* heads = reinterpret_cast<unsigned short*>(ra_col + GK_CAP1);           // 2 CAP1 shorts
    const int warp = blockIdx.x * GK_WARPS + wib, nwarps = gridDim.x * GK_WARPS;
    int wmax = 0;   // longest output row this warp produced
    for (int I = warp; I < nc; I += nwarps) {
        // ---- phase 1: row I of R*A ----
        int tot = 0;
        for (int kr = rrp[I]; kr < rrp[I + 1]; ++kr) {  // at most four entries, ascending fine row
            const int i = rcol[kr];
            const double alpha = 1. * rval[kr];
            const int bb = arp[i], len = arp[i + 1] - bb;
            for (int q = lane; q < len; q += 32) {
                keys[tot + q] = ((KeyT)(unsigned int)acol[bb + q] << POSB) | (KeyT)(unsigned int)(tot + q);
                vals[tot + q] = alpha * aval[bb + q];
            }
            tot += len;
        }
        int P = 32;
        while (P < tot) P <<= 1;
        for (int idx = tot + lane; idx < P; idx += 32) keys[idx] = SENTINEL;
        __syncwarp();
        warp_sort_keys<GK_CAP, KeyT>(keys, P, lane);
        const int n1 = warp_runs<KeyT, POSB>(keys, tot, heads, lane);
        for (int q = lane; q < n1; q += 32) {
            const int b = heads[q], e = (q + 1 < n1) ? heads[q + 1] : tot;
            double acc = 0. * 0.;
            for (int idx = b; idx < e; ++idx) acc += vals[(unsigned int)(keys[idx] & POSMASK)];
            ra_col[q] = (int)(keys[b] >> POSB);
            ra_val[q] = acc;
        }
        __syncwarp();
        // ---- phase 2: row I of (R*A)*R^T ----
        int tot2 = 0;
        for (int base = 0; base < n1; base += 32) {
            const int q = base + lane;
            int len = 0, bb = 0;
            double alpha = 0.;
            if (q < n1) { const int j = ra_col[q]; bb = trp[j]; len = trp[j + 1] - bb; alpha = 1. * ra_val[q]; }
            int incl = len;
            for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
            const int my = tot2 + incl - len;
            for (int e = 0; e < len; ++e) {
                keys[my + e] = ((KeyT)(unsigned int)tcol_[bb + e] << POSB) | (KeyT)(unsigned int)(my + e);
                vals[my + e] = alpha * tval_[bb + e];
            }
            tot2 += __shfl_sync(0xffffffffu, incl, 31);
        }
        P = 32;
        while (P < tot2) P <<= 1;
        for (int idx = tot2 + lane; idx < P; idx += 32) keys[idx] = SENTINEL;
        __syncwarp();
        warp_sort_keys<GK_CAP, KeyT>(keys, P, lane);
        const int n2 = warp_runs<KeyT, POSB>(keys, tot2, heads, lane);
        const int o0 = outptr[I];
        for (int q = lane; q < n2; q += 32) {
            const int b = heads[q], e = (q + 1 < n2) ? heads[q + 1] : tot2;
            double acc = 0. * 0.;
            for (int idx = b; idx < e; ++idx) acc += vals[(unsigned int)(keys[idx] & POSMASK)];
            ocol[o0 + q] = (int)(keys[b] >> POSB);
            oval[o0 + q] = acc;
        }
        if (lane == 0) counts[I] = n2;
        wmax = max(wmax, n2);
        __syncwarp();
    }
    if (lane == 0 && wmax > 0) atomicMax(maxrow, wmax);
}
__global__ void k_double_counts(int n, const int* in, int* out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = 2 * in[i];
}

CsrPtr galerkin(Ctx& c, const DCsr& R, const DCsr& RT, const DCsr& A) {
    ORC_REQUIRE(R.ncols == A.nrows && A.ncols == RT.nrows, ORC_E_INVALID, "galerkin: dimension mismatch");
    const int nc = (int)R.nrows;
    // upper bounds: phase 1 gathers cand1 = sum of the selected A-row lengths; phase 2 at most 2 terms per entry of R*A
    DBuf<int> cand(&c, (size_t)nc + 1), cand2(&c, (size_t)nc + 1), outptr(&c, (size_t)nc + 1), counts(&c, (size_t)nc + 1), rp(&c, (size_t)nc + 1), maxc(&c, 4);
    cand.zero(); cand2.zero(); counts.zero(); maxc.zero();
    int hmax = 0, htot = 0;
    int hm4[4] = {0, 0, 0, 0};
    if (nc > 0) {
        k_spgemm_cand<<<(nc + 255) / 256, 256, 0, c.stream>>>(nc, R.rowptr, R.col, A.rowptr, cand, maxc);
        c.after_launch("k_spgemm_cand");
        k_double_counts<<<(nc + 255) / 256, 256, 0, c.stream>>>(nc, cand, cand2);
        c.after_launch("k_double_counts");
    }
    exclusive_scan_to_rowptr(c, cand2, outptr, nc);
    maxc.download(hm4);
    ORC_CUDA(cudaMemcpyAsync(&htot, outptr.p + nc, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    hmax = hm4[0];
    unsigned long long tot64 = 0;
    memcpy(&tot64, hm4 + 2, sizeof(tot64));
    const bool too_many = 2ull * tot64 > (unsigned long long)INT32_MAX;   // the scanned counts are 2 * cand
    bool rt_short = true;  // R^T rows hold at most two entries when R comes from build_restriction; verify cheaply via nnz
    if (RT.nnz > 2 * RT.nrows) rt_short = false;
    if (hmax > 512 || too_many || !rt_short) {  // very long rows / foreign R: the generic two-step path
        CsrPtr RA = spgemm(c, R, A);          // &restriction_matrix * a
        CsrPtr Ac = spgemm(c, *RA, RT);       // (...) * &restriction_matrix.transpose()
        Ac->sym = A.sym;
        Ac->hint = A.hint; Ac->hint.shift = A.hint.shift + 1;
        Ac->simplex = A.simplex;
        return Ac;
    }
    DBuf<int> tcol(&c, (size_t)std::max(htot, 1));
    DBuf<double> tval(&c, (size_t)std::max(htot, 1));
    if (nc > 0) {
        static const bool force64 = [] { const char* e = getenv("ORC_B200_GALERKIN_KEY64"); return e && atoi(e) != 0; }();  // tests
        auto launch = [&](auto kernel, size_t smem_per_warp) {
            const size_t smem = smem_per_warp * GK_WARPS;
            ORC_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            const int grid = std::max(1, std::min((nc + GK_WARPS - 1) / GK_WARPS, c.sm_count * 8));
            kernel<<<grid, GK_WARPS * 32, smem, c.stream>>>(nc, R.rowptr, R.col, R.val, A.rowptr, A.col, A.val, RT.rowptr, RT.col, RT.val, outptr,
                                                            counts, tcol, tval, maxc.p + 1);
            c.after_launch("k_galerkin_rows");
        };
        // 32-bit keys need (largest column + 1) << log2(2 * cap1) to stay below the all-ones sentinel
        const int64_t maxcol = std::max<int64_t>(A.ncols, RT.ncols);
        auto go = [&](auto k32, auto k64, int cap1) {
            const bool fits = !force64 && (maxcol + 1) < ((int64_t)1 << (32 - gk_log2(2 * cap1)));
            if (fits) launch(k32, gk_smem_per_warp<unsigned int>(cap1));
            else launch(k64, gk_smem_per_warp<unsigned long long>(cap1));
        };
        if (hmax <= 32) go(k_galerkin_rows<32, unsigned int>, k_galerkin_rows<32, unsigned long long>, 32);
        else if (hmax <= 64) go(k_galerkin_rows<64, unsigned int>, k_galerkin_rows<64, unsigned long long>, 64);
        else if (hmax <= 128) go(k_galerkin_rows<128, unsigned int>, k_galerkin_rows<128, unsigned long long>, 128);
        else if (hmax <= 256) go(k_galerkin_rows<256, unsigned int>, k_galerkin_rows<256, unsigned long long>, 256);
        else go(k_galerkin_rows<512, unsigned int>, k_galerkin_rows<512, unsigned long long>, 512);
    }
    exclusive_scan_to_rowptr(c, counts, rp, nc);
    int nnz = 0, max_row = 0;
    ORC_CUDA(cudaMemcpyAsync(&nnz, rp.p + nc, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    ORC_CUDA(cudaMemcpyAsync(&max_row, maxc.p + 1, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    CsrPtr Ac = csr_alloc(c, R.nrows, RT.ncols, nnz);
    Ac->max_row = max_row;
    Ac->simplex = A.simplex;
    Ac->hint = A.hint; Ac->hint.shift = A.hint.shift + 1;
    ORC_CUDA(cudaMemcpyAsync(Ac->rowptr, rp.p, sizeof(int) * ((size_t)nc + 1), cudaMemcpyDeviceToDevice, c.stream));
    if (nc > 0 && nnz > 0) {
        k_spgemm_compact<<<std::max(1, std::min((nc + 7) / 8, c.sm_count * 8)), 256, 0, c.stream>>>(nc, outptr, Ac->rowptr, tcol, tval, Ac->col, Ac->val);
        c.after_launch("k_spgemm_compact");
    }
    Ac->sym = A.sym;  // R A R^T of a structurally symmetric A is structurally symmetric
    return Ac;
}

// =================================================================================================
// multigrid_solve (linear_algebra.rs:66-141) and iterative_solve (:144-299)
// =================================================================================================
static void residual(Ctx& c, const DCsr& A, const double* b, const double* x, double* r, int K = 1) {
    if (A.nrows == 0) return;
    SpmvArgs a{};
    a.x = x; a.y = r; a.b = b;
    launch_spmv<EP_RESID>(c, A, a, K);
}
static void residual_norm_check(Ctx& c, const DCsr& A, const double* b, const double* x, int K = 1) {
    // error_magnitude = (&r_prime - &a_prime * &e_prime).norm(); NaN -> "Multigrid diverged" (:97-105)
    if (A.nrows == 0) return;
    SpmvArgs a{};
    a.x = x; a.b = b;
    launch_spmv<EP_RESID_NORM>(c, A, a, K);
}


// =================================================================================================
// Locality ordering of the coarse levels (no counterpart in the reference: a storage order, not an algorithm change).
//
// What bounds the coarse-level gather SpMVs is the number of distinct 128-byte lines a warp instruction touches (~2 cycles of
// the L1 data pipe each; profiles/r2_staged_spmv_lab_v2.txt). The aggregates are numbered by the reference's rule (coarse row
// I = fine rows 2I, 2I+1 plus their picks), i.e. x-fastest with the x extent halving per level, while the picks widen the
// stencil in y and z: on level 3 of the 128^3 box a row's ~100 columns come in runs of <= 3. Stored along the Morton curve of
// the aggregate positions the same rows touch 20-36 % fewer lines (scripts/lab/reorder_analysis.py; measured on B200,
// profiles/r2_reorder_lab.txt: level 2 / 3 three-system SpMV 109 -> 89 us / 121 -> 91 us, one system 66 -> 53 / 78 -> 58 us).
//
// So a level's smoother runs on  P (D^-1 A) P^T  y = P D^-1 b,  x = P^T y:  the Jacobi-scaled copy that iterative_solve makes
// anyway (linear_algebra.rs:157-168) is WRITTEN in the permuted order (rows permuted, columns renumbered and re-sorted), once
// per level instead of once per smoothing call. The hierarchy itself (aggregates, Galerkin products — both depend on the
// numbering) is built from the matrices in the reference's numbering and stays bit-exact; entry values are the same
// products, only the summation order inside the already toleranced coarse SpMVs / dot products changes (DESIGN.md §5).
// Needs positions (DCsr::hint: mesh matrices have them); reference-order mode never reorders.
// =================================================================================================
static int reorder_min_level() {   // ORC_B200_REORDER=0 switches the ordering off, =l applies it from coarse level l on (default 1)
    const char* e = getenv("ORC_B200_REORDER");   // read per call (a few times per solve): tests switch it inside one process
    return e ? atoi(e) : 1;
}
constexpr int64_t kReorderMinRows = 16384;   // below this a level is launch bound, not gather bound
constexpr int RO_WARPS = 8, RO_CAP = 512, RO_POSB = 9;   // rows of up to 512 entries (longer rows: the level keeps its order)

__device__ __forceinline__ unsigned int morton_spread10(unsigned int v) {   // 10 bits -> every third bit
    v &= 0x3ffu;
    v = (v | (v << 16)) & 0x030000ffu;
    v = (v | (v << 8)) & 0x0300f00fu;
    v = (v | (v << 4)) & 0x030c30c3u;
    v = (v | (v << 2)) & 0x09249249u;
    return v;
}
__global__ void k_morton_keys(int n, PosHint h, unsigned int* keys, int* ids) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t f = min((int64_t)i << h.shift, h.n - 1);
    const double q[3] = {(h.x[f] - h.lo[0]) * h.inv[0], (h.y[f] - h.lo[1]) * h.inv[1], (h.z[f] - h.lo[2]) * h.inv[2]};
    unsigned int key = 0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const int v = q[a] >= 1023. ? 1023 : (q[a] > 0. ? (int)q[a] : 0);   // NaN -> 0
        key |= morton_spread10((unsigned int)v) << a;
    }
    keys[i] = key;
    ids[i] = i;
}
// iperm[perm[r]] = r; cnt[r] = entries of the scaled row perm[r] (a row without a stored diagonal is empty, like in jacobi_scale)
__global__ void k_perm_inverse_counts(int n, const int* __restrict__ perm, const int* __restrict__ rowptr, const int* __restrict__ diag, int* iperm, int* cnt) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const int i = perm[r];
    iperm[i] = r;
    cnt[r] = diag[i] >= 0 ? rowptr[i + 1] - rowptr[i] : 0;
}
// One warp per row of the permuted matrix: scale (the same products as k_jacobi_scale), renumber the columns, sort them.
template <int K, class KeyT>
__global__ void __launch_bounds__(RO_WARPS * 32) k_scale_permute_rows(int n, const int* __restrict__ rowptr, const int* __restrict__ col,
                                                                      const int* __restrict__ diag, const double* __restrict__ val,
                                                                      const int* __restrict__ perm, const int* __restrict__ iperm,
                                                                      const int* __restrict__ rp_out, int* __restrict__ col_out,
                                                                      double* __restrict__ val_out, const double* __restrict__ b,
                                                                      double* __restrict__ b_out) {
    __shared__ KeyT skeys[RO_WARPS][RO_CAP];
    constexpr KeyT SENTINEL = (KeyT)~(KeyT)0, POSMASK = (KeyT)(RO_CAP - 1);
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int warp = blockIdx.x * RO_WARPS + wib, nwarps = gridDim.x * RO_WARPS;
    KeyT* keys = skeys[wib];
    for (int r = warp; r < n; r += nwarps) {
        const int i = perm[r];
        const int lo = rowptr[i], len = rowptr[i + 1] - lo, d = diag[i];
        const double pinv = (d >= 0) ? 1. / val[d] : 0.;
        if (lane == 0) {
            double bi[K], bo[K];
            Cell<K>::ld(b, i, bi);
#pragma unroll
            for (int k = 0; k < K; ++k) bo[k] = (d >= 0) ? 0. + pinv * bi[k] : 0.;
            Cell<K>::st(b_out, r, bo);
        }
        if (d < 0) continue;
        int P = 32;
        while (P < len) P <<= 1;
        for (int q = lane; q < P; q += 32) keys[q] = q < len ? (((KeyT)(unsigned int)iperm[col[lo + q]] << RO_POSB) | (KeyT)(unsigned int)q) : SENTINEL;
        __syncwarp();
        warp_sort_keys<RO_CAP, KeyT>(keys, P, lane);
        const int o = rp_out[r];
        for (int q = lane; q < len; q += 32) {
            const KeyT key = keys[q];
            col_out[o + q] = (int)(key >> RO_POSB);
            val_out[o + q] = 0. + (1. * pinv) * val[lo + (int)(key & POSMASK)];
        }
        __syncwarp();
    }
}
template <int K>
__global__ void k_permute_cells(int64_t n, const int* __restrict__ perm, const double* __restrict__ in, double* __restrict__ out, int scatter) {
    for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x) {
        double v[K];
        if (scatter) { Cell<K>::ld(in, r, v); Cell<K>::st(out, perm[r], v); }
        else { Cell<K>::ld(in, perm[r], v); Cell<K>::st(out, r, v); }
    }
}
struct ReorderedLevel {
    DBuf<int> perm;      // row r of the stored system is row perm[r] of the level
    CsrPtr A;            // P (D^-1 A) P^T, columns sorted
    DBuf<double> b, x;   // P D^-1 b, and the iterate in stored order
    bool on() const { return (bool)A; }
};
static bool reorder_applies(const Ctx& c, const DCsr& A, int level, const SolveParams& sp) {
    const int lmin = reorder_min_level();
    return lmin > 0 && level >= lmin && !sp.exact_order && sp.mg_smoother == ORC_SOLVER_BICGSTAB && sp.preconditioner == ORC_PC_JACOBI &&
           A.hint.on() && A.nrows == A.ncols && A.nrows >= kReorderMinRows && A.max_row > 0 && A.max_row <= RO_CAP;
}
static void permute_cells(Ctx& c, int64_t n, const int* perm, const double* in, double* out, bool scatter, int K) {
    if (n == 0) return;
    ProfScope ps(c, PC_VECTOR, (16. * K + 4.) * (double)n);
    if (K == 1) k_permute_cells<1><<<grid_for(n, 256, c.sm_count * 8), 256, 0, c.stream>>>(n, perm, in, out, scatter ? 1 : 0);
    else k_permute_cells<3><<<grid_for(n, 256, c.sm_count * 8), 256, 0, c.stream>>>(n, perm, in, out, scatter ? 1 : 0);
    c.after_launch("k_permute_cells");
}
static void build_reordered(Ctx& c, DCsr& A, const double* b, int K, ReorderedLevel& ro) {
    const int n = (int)A.nrows;
    const int S = vstride(K);
    csr_ensure_diag(c, A);
    DBuf<unsigned int> k_in(&c, (size_t)n), k_out(&c, (size_t)n);
    DBuf<int> ids(&c, (size_t)n), iperm(&c, (size_t)n), cnt(&c, (size_t)n + 1);
    ro.perm.alloc(&c, (size_t)n);
    k_morton_keys<<<(n + 255) / 256, 256, 0, c.stream>>>(n, A.hint, k_in, ids);
    c.after_launch("k_morton_keys");
    size_t tmp_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, k_in.p, k_out.p, ids.p, ro.perm.p, n, 0, 30, c.stream);
    DBuf<char> tmp(&c, tmp_bytes);
    ORC_CUDA(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, k_in.p, k_out.p, ids.p, ro.perm.p, n, 0, 30, c.stream));   // stable: ties keep the row order
    ++c.launches;
    cnt.zero();
    k_perm_inverse_counts<<<(n + 255) / 256, 256, 0, c.stream>>>(n, ro.perm, A.rowptr, A.diag, iperm, cnt);
    c.after_launch("k_perm_inverse_counts");
    ro.A = csr_alloc(c, n, n, A.nnz);   // nnz is an upper bound when rows without a diagonal are dropped; kernels read rowptr
    exclusive_scan_to_rowptr(c, cnt, ro.A->rowptr, n);
    ro.A->sym = A.sym; ro.A->max_row = A.max_row;
    ro.b.alloc(&c, (size_t)n * S); ro.x.alloc(&c, (size_t)n * S);
    const int grid = std::max(1, std::min((n + RO_WARPS - 1) / RO_WARPS, c.sm_count * 8));
    auto go = [&](auto kern) {
        kern<<<grid, RO_WARPS * 32, 0, c.stream>>>(n, A.rowptr, A.col, A.diag, A.val, ro.perm, iperm, ro.A->rowptr, ro.A->col, ro.A->val, b, ro.b.p);
        c.after_launch("k_scale_permute_rows");
    };
    const bool key32 = (int64_t)n < ((int64_t)1 << (32 - RO_POSB)) - 1;
    if (K == 1) { if (key32) go(k_scale_permute_rows<1, unsigned int>); else go(k_scale_permute_rows<1, unsigned long long>); }
    else { if (key32) go(k_scale_permute_rows<3, unsigned int>); else go(k_scale_permute_rows<3, unsigned long long>); }
}
// one smoothing call of multigrid_solve on the stored system: x (level order) in and out
static void reordered_smooth(Ctx& c, ReorderedLevel& ro, double* x, uint64_t iterations, bool x_is_zero, int K) {
    const int64_t n = ro.A->nrows;
    if (x_is_zero) ro.x.zero();
    else permute_cells(c, n, ro.perm, x, ro.x, false, K);
    bicgstab(c, *ro.A, ro.b, ro.x, iterations, K);
    permute_cells(c, n, ro.perm, ro.x, x, true, K);
}

// K systems (vectors of K-cells, see Cell<K>) share the hierarchy: aggregates, Galerkin products and scaled copies depend
// on the matrix only, so they are built once per call for all of them.
static void multigrid_solve(Ctx& c, DCsr& A, const double* r, double* out /* len A.ncols */, int level, const SolveParams& sp,
                            MgTrace* trace, int K = 1) {
    const int S = vstride(K);
    CsrPtr RT, R;
    {
        ProfScope ps(c, PC_RESTRICT, 0.);
        R = build_restriction(c, A, ORC_RESTRICT_STRONGEST, &RT);              // :80
    }
    const int64_t nc = R->nrows;
    DBuf<double> r_prime(&c, std::max<int64_t>(nc, 1) * S), e_prime(&c, std::max<int64_t>(nc, 1) * S);
    spmv(c, *R, r, r_prime, K);                                                 // :82
    CsrPtr Ac;
    {
        ProfScope ps(c, PC_GALERKIN, 0.);
        Ac = galerkin(c, *R, *RT, A);                                           // :84
    }
    if (trace) { trace->rows.push_back(Ac->nrows); trace->nnz.push_back(Ac->nnz); }
    e_prime.zero();                                                             // :86
    SolveParams smooth = sp;
    smooth.method = sp.mg_smoother;
    ReorderedLevel ro;
    if (reorder_applies(c, *Ac, level, sp)) {
        ProfScope ps(c, PC_SCALE, 0.);
        build_reordered(c, *Ac, r_prime, K, ro);
    }
    if (ro.on()) reordered_smooth(c, ro, e_prime, smooth.iterations, true, K);
    else iterative_solve(c, *Ac, r_prime, e_prime, smooth, nullptr, K);         // :87-96
    residual_norm_check(c, *Ac, r_prime, e_prime, K);                           // :97-105
    if (level < sp.mg_levels && Ac->nrows > 16) {                               // :109
        DBuf<double> corr(&c, std::max<int64_t>(nc, 1) * S);
        multigrid_solve(c, *Ac, r_prime, corr, level + 1, sp, trace, K);        // :110-121 (r_prime, not the residual: Q11)
        dev_axpy_inplace(c, e_prime, corr, nc * S);
        SolveParams post = smooth;
        post.threshold = sp.threshold / 10.;
        if (ro.on()) reordered_smooth(c, ro, e_prime, post.iterations, false, K);
        else iterative_solve(c, *Ac, r_prime, e_prime, post, nullptr, K);       // :123-132
    }
    spmv(c, *RT, e_prime, out, K);                                              // :140
    if (trace && trace->keep) {
        // stored coarse-first in recursion order; the caller reverses nothing: index l = level-1 is fixed below
        trace->restriction.resize(std::max<size_t>(trace->restriction.size(), (size_t)level));
        trace->coarse.resize(std::max<size_t>(trace->coarse.size(), (size_t)level));
        trace->restriction[level - 1] = std::move(R);
        trace->coarse[level - 1] = std::move(Ac);
    }
}

// Can `sp` be run on a batch of three systems? Needs a lockstep method: the unguarded BiCGSTAB (alone or as the Multigrid
// smoother). Jacobi breaks out per system, Gauss-Seidel is a dataflow sweep over one vector.
bool solve_batchable(const SolveParams& sp) {
    if (sp.exact_order) return false;
    if (sp.method == ORC_SOLVER_BICGSTAB) return true;
    return sp.method == ORC_SOLVER_MULTIGRID && sp.mg_smoother == ORC_SOLVER_BICGSTAB;
}

// rows/columns [lo, hi) of A as a standalone CSR with indices shifted to 0 (the rank's diagonal block)
__global__ void k_block_counts(int lo, int hi, const int* __restrict__ rowptr, const int* __restrict__ col, int* cnt) {
    int i = lo + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= hi) return;
    int m = 0;
    for (int k = rowptr[i]; k < rowptr[i + 1]; ++k) m += (col[k] >= lo && col[k] < hi);
    cnt[i - lo] = m;
}
__global__ void k_block_fill(int lo, int hi, const int* __restrict__ rowptr, const int* __restrict__ col, const double* __restrict__ val,
                             const int* __restrict__ rp_out, int* col_out, double* val_out) {
    int i = lo + blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= hi) return;
    int o = rp_out[i - lo];
    for (int k = rowptr[i]; k < rowptr[i + 1]; ++k)
        if (col[k] >= lo && col[k] < hi) { col_out[o] = col[k] - lo; val_out[o] = val[k]; ++o; }
}
static CsrPtr extract_block(Ctx& c, const DCsr& A, int64_t lo, int64_t hi) {
    const int n = (int)(hi - lo);
    DBuf<int> cnt(&c, (size_t)n + 1), rp(&c, (size_t)n + 1);
    cnt.zero();
    if (n > 0) {
        k_block_counts<<<(n + 255) / 256, 256, 0, c.stream>>>((int)lo, (int)hi, A.rowptr, A.col, cnt);
        c.after_launch("k_block_counts");
    }
    exclusive_scan_to_rowptr(c, cnt, rp, n);
    int nnz = 0;
    ORC_CUDA(cudaMemcpyAsync(&nnz, rp.p + n, sizeof(int), cudaMemcpyDeviceToHost, c.stream));
    c.sync();
    CsrPtr B = csr_alloc(c, n, n, nnz);
    ORC_CUDA(cudaMemcpyAsync(B->rowptr, rp.p, sizeof(int) * ((size_t)n + 1), cudaMemcpyDeviceToDevice, c.stream));
    if (n > 0) {
        k_block_fill<<<(n + 255) / 256, 256, 0, c.stream>>>((int)lo, (int)hi, A.rowptr, A.col, A.val, B->rowptr, B->col, B->val);
        c.after_launch("k_block_fill");
    }
    B->sym = A.sym;
    B->max_row = A.max_row;   // an upper bound is all the users need
    B->simplex = A.simplex;
    if (A.hint.on() && A.hint.shift == 0 && hi <= A.hint.n) {   // the block's rows keep their places
        B->hint = A.hint;
        B->hint.x += lo; B->hint.y += lo; B->hint.z += lo; B->hint.n = hi - lo;
    }
    return B;
}

void iterative_solve(Ctx& c, DCsr& A, const double* b, double* x, const SolveParams& sp, MgTrace* trace, int K, const DistEnv* env) {
    const bool dist = env && env->on();
    ORC_REQUIRE(A.nrows == A.ncols, ORC_E_INVALID, "iterative_solve: matrix must be square");
    ORC_REQUIRE(!(dist && sp.exact_order), ORC_E_UNSUPPORTED, "reference-order reductions are single-GPU only");
    ORC_REQUIRE(K == 1 || (K == 3 && solve_batchable(sp)), ORC_E_UNSUPPORTED, "this solver cannot run three systems in lockstep");
    const int64_t n = A.nrows;
    const int S = vstride(K);
    c.exact_order = sp.exact_order;
    CsrPtr a_tmp;
    DBuf<double> b_tmp;
    DCsr* Ap = &A;
    const double* bp = b;
    if (sp.preconditioner == ORC_PC_JACOBI) {  // :157-168; row-local, so a partition needs no communication
        b_tmp.alloc(&c, std::max<int64_t>(n, 1) * S);
        ProfScope ps(c, PC_SCALE, 0.);
        a_tmp = jacobi_scale(c, A, b, b_tmp, K);
        Ap = a_tmp.get();
        bp = b_tmp;
    }
    switch (sp.method) {
        case ORC_SOLVER_JACOBI: jacobi(c, *Ap, bp, x, sp, env); break;
        case ORC_SOLVER_GAUSS_SEIDEL:   // the sweep is one dependency chain over all rows: it has no partitioned form
            ORC_REQUIRE(!dist, ORC_E_UNSUPPORTED, "multi-GPU solves support Jacobi, BiCGSTAB and Multigrid");
            gauss_seidel(c, *Ap, bp, x, sp);
            break;
        case ORC_SOLVER_BICGSTAB: bicgstab(c, *Ap, bp, x, sp.iterations, K, env); break;
        case ORC_SOLVER_MULTIGRID: {  // :270-296
            // on a partition the coarse correction is the reference's multigrid_solve on this rank's diagonal block (rows [lo, lo + nown)):
            // aggregates never cross the partition (C4)
            const int64_t lo = dist ? env->halo->own_lo : 0, nown = dist ? env->halo->own_hi - lo : n;
            if (trace) { trace->rows.clear(); trace->nnz.clear(); trace->rows.push_back(nown); trace->nnz.push_back(Ap->nnz); }
            SolveParams pre = sp;
            pre.method = sp.mg_smoother;
            ORC_REQUIRE(!dist || pre.method == ORC_SOLVER_BICGSTAB, ORC_E_UNSUPPORTED, "multi-GPU multigrid needs the BiCGSTAB smoother");
            iterative_solve(c, *Ap, bp, x, pre, nullptr, K, env);   // preconditions AGAIN (Q7), globally on a partition
            DBuf<double> r(&c, std::max<int64_t>(n, 1) * S), corr(&c, std::max<int64_t>(nown, 1) * S);
            CsrPtr Aloc;
            if (dist) {
                r.zero();
                env->halo->exchange(c, *env->comm, x, S);
            }
            residual(c, *Ap, bp, x, r, K);
            if (dist) Aloc = extract_block(c, *Ap, lo, lo + nown);
            multigrid_solve(c, dist ? *Aloc : *Ap, r.p + lo * S, corr, 1, sp, trace, K);
            dev_axpy_inplace(c, x + lo * S, corr, nown * S);
            break;
        }
        default: throw Error(ORC_E_UNSUPPORTED, dist ? "multi-GPU solves support Jacobi, BiCGSTAB and Multigrid" : "unsupported solution method");
    }
}

void check_solver_flags(Ctx& c) {
    int f = c.read_flags();
    if (f == 0) return;
    c.clear_flags();
    throw_for_flags(f);
}
void throw_for_flags(int f) {
    f &= ~DF_CONVERGED;
    if (f == 0) return;
    if (f & DF_SPIN) throw Error(ORC_E_INTERNAL, "dataflow kernel exceeded its spin bound");
    if (f & DF_MISSING_ENTRY) throw Error(ORC_E_MISSING_ENTRY, "Tried to access CsrMatrix element that hasn't been stored yet.");
    if (f & DF_UNSUPPORTED_BC) throw Error(ORC_E_UNSUPPORTED, "unsupported face zone type");
    if (f & DF_SINGULAR) throw Error(ORC_E_INVALID, "called `Option::unwrap()` on a `None` value (singular least-squares gradient system)");
    if (f & DF_NAN_JACOBI) throw Error(ORC_E_JACOBI_DIVERGED, "diverged");
    if (f & DF_JACOBI_HUGE) throw Error(ORC_E_JACOBI_DIVERGED, "Diverged - max solution value > 10^10");
    if (f & DF_GS_NAN) throw Error(ORC_E_GS_DIVERGED, "****** Solution diverged ******");
    if (f & DF_MG_NAN) throw Error(ORC_E_MG_DIVERGED, "Multigrid diverged");
}

}  // namespace orc
