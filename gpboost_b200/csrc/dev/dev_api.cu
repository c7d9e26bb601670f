// Device engine for the Vecchia-approximated Gaussian process: C ABI of include/gpboost_b200_dev.h.
// sm_100a only; there is no CPU fallback (every entry fails loudly without a CUDA device).
#include "../../../include/gpboost_b200_dev.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <numeric>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "knn.cuh"
#include "vecchia_factor.cuh"
#include "vecchia_big.cuh"
#include "vecchia_nll2.cuh"

namespace {

thread_local std::string g_last_error;

int fail(const std::string& msg) {
  g_last_error = msg;
  return -1;
}

#define CUDA_TRY(expr)                                                                              \
  do {                                                                                              \
    cudaError_t err__ = (expr);                                                                     \
    if (err__ != cudaSuccess) {                                                                     \
      return fail(std::string("CUDA error at " __FILE__ ":") + std::to_string(__LINE__) + ": " +    \
                  cudaGetErrorString(err__));                                                       \
    }                                                                                               \
  } while (0)

// ---- small kernels around the factor kernel -------------------------------------------------------

// y_ord[i] = y_orig[perm[i]]  (the per-cluster re-ordering SetY does, re_model_template.h:6185-6200)
__global__ void gather_perm_kernel(const double* __restrict__ src, const int32_t* __restrict__ perm,
                                   double* __restrict__ dst, int64_t n) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    dst[i] = src[perm[i]];
}

// fixed-order reduction of the per-warp partial sums: deterministic for a given grid
__global__ void reduce_partials_kernel(const double* __restrict__ partials, int64_t nrows, double* __restrict__ out) {
  __shared__ double sh[256];
  for (int k = 0; k < gpb::kNumAcc; ++k) {
    double s = 0.;
    for (int64_t r = threadIdx.x; r < nrows; r += blockDim.x) s += partials[r * gpb::kNumAcc + k];
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int o = blockDim.x / 2; o > 0; o >>= 1) {
      if (threadIdx.x < o) sh[threadIdx.x] += sh[threadIdx.x + o];
      __syncthreads();
    }
    if (threadIdx.x == 0) out[k] = sh[0];
    __syncthreads();
  }
}

// y_aux = B^T u with u = D^-1 B y (CalcYAux, re_model_template.h:9772), gather form over the CSC view of
// B's pattern: one warp per column, deterministic; result scattered back to the original observation order.
__global__ void bt_apply_kernel(const double* __restrict__ A, const double* __restrict__ u,
                                const int32_t* __restrict__ colptr, const int32_t* __restrict__ csc_pos,
                                const int32_t* __restrict__ perm, double* __restrict__ out_orig, int64_t n, int m,
                                int64_t row_begin, int64_t row_end, double scale) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t j = warp; j < n; j += nwarps) {
    const int32_t b = colptr[j], e = colptr[j + 1];
    double s = 0.;
    for (int32_t p = b + lane; p < e; p += 32) {
      const int32_t pos = csc_pos[p];
      s -= A[pos] * u[pos / m];
    }
    s = gpb::warp_sum(s);
    if (lane == 0) {
      if (j >= row_begin && j < row_end) s += u[j];  // unit diagonal of B
      out_orig[perm[j]] = s * scale;
    }
  }
}

__global__ void fill_kernel(double* p, int64_t n, double v) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) p[i] = v;
}

// FP64 FMA throughput probe: 8 independent dependent-chains per thread, no memory traffic. Gives the measured
// DFMA peak of this chip that the factor kernel (FP64-pipe bound) is compared against in bench.py.
__global__ void fp64_peak_kernel(double* out, int iters, double a, double b) {
  double x0 = threadIdx.x, x1 = x0 + 1., x2 = x0 + 2., x3 = x0 + 3., x4 = x0 + 4., x5 = x0 + 5., x6 = x0 + 6., x7 = x0 + 7.;
  for (int i = 0; i < iters; ++i) {
    x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
    x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
  }
  if (x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7 == 12345.678) out[0] = x0;
}

using FactorKernel = void (*)(const gpb::FactorArgs);

template <int COV, int MODE, int DIM>
FactorKernel pick_cap(int m) {
  if (m <= 10) return gpb::vecchia_factor_kernel<COV, MODE, DIM, 10>;
  if (m <= 20) return gpb::vecchia_factor_kernel<COV, MODE, DIM, 20>;
  return gpb::vecchia_factor_kernel<COV, MODE, DIM, 30>;
}
template <int COV, int MODE>
FactorKernel pick_dim(int d, int m) {
  return d == 2 ? pick_cap<COV, MODE, 2>(m) : pick_cap<COV, MODE, 0>(m);
}
template <int COV>
FactorKernel pick_mode(int mode, int d, int m) {
  switch (mode) {
    case gpb::MODE_NLL: return pick_dim<COV, gpb::MODE_NLL>(d, m);
    case gpb::MODE_STORE: return pick_dim<COV, gpb::MODE_STORE>(d, m);
    case gpb::MODE_GRAD: return pick_dim<COV, gpb::MODE_GRAD>(d, m);
    default: return pick_dim<COV, gpb::MODE_STORE_GRAD>(d, m);
  }
}
FactorKernel pick_kernel(int cov, int mode, int d, int m) {
  switch (cov) {
    case gpb::COV_EXPONENTIAL: return pick_mode<gpb::COV_EXPONENTIAL>(mode, d, m);
    case gpb::COV_MATERN15: return pick_mode<gpb::COV_MATERN15>(mode, d, m);
    case gpb::COV_MATERN25: return pick_mode<gpb::COV_MATERN25>(mode, d, m);
    default: return pick_mode<gpb::COV_GAUSSIAN>(mode, d, m);
  }
}

using BigKernel = void (*)(const gpb::BigArgs);
template <int COV>
BigKernel pick_big_mode(int mode) {
  switch (mode) {
    case gpb::BIG_NLL: return gpb::vecchia_big_kernel<COV, gpb::BIG_NLL>;
    case gpb::BIG_STORE: return gpb::vecchia_big_kernel<COV, gpb::BIG_STORE>;
    case gpb::BIG_GRAD: return gpb::vecchia_big_kernel<COV, gpb::BIG_GRAD>;
    default: return gpb::vecchia_big_kernel<COV, gpb::BIG_PRED>;
  }
}
BigKernel pick_big_kernel(int cov, int mode) {
  switch (cov) {
    case gpb::COV_EXPONENTIAL: return pick_big_mode<gpb::COV_EXPONENTIAL>(mode);
    case gpb::COV_MATERN15: return pick_big_mode<gpb::COV_MATERN15>(mode);
    case gpb::COV_MATERN25: return pick_big_mode<gpb::COV_MATERN25>(mode);
    default: return pick_big_mode<gpb::COV_GAUSSIAN>(mode);
  }
}

}  // namespace

struct gpb_laplace_state;

struct gpbdev_vecchia {
  gpb_laplace_state* lap = nullptr;  // Laplace-Vecchia buffers (laplace.cuh), lazy
  gpbdev_allreduce_fn allreduce = nullptr;  // device collective hook (row-sharded engines)
  void* allreduce_ctx = nullptr;
  int device = 0;
  int64_t n = 0;
  int d = 0, m = 0;
  int64_t row_begin = 0, row_end = 0;
  int num_sms = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  double* coords = nullptr;   // n x d
  int32_t* nn = nullptr;      // n x m
  int32_t* perm = nullptr;    // n
  double* y_in = nullptr;     // n staging (original order)
  double* y = nullptr;        // n ordered
  double* A = nullptr;        // n x m   (lazy)
  double* Dinv = nullptr;     // n       (lazy)
  double* u = nullptr;        // n       (lazy)
  double* dA = nullptr;       // n x m   (lazy, MODE_STORE_GRAD)
  double* dD = nullptr;       // n       (lazy, MODE_STORE_GRAD)
  double* yaux = nullptr;     // n       (lazy, original order)
  int32_t* colptr = nullptr;  // n + 1   (lazy)
  int32_t* csc_pos = nullptr; // nnz     (lazy)
  int32_t* csc_row = nullptr; // nnz     (lazy, Laplace): row of every CSC entry (= csc_pos / m)
  double* A_csc = nullptr;    // nnz     (lazy, Laplace): A in CSC order, refreshed after every latent factorisation
  double* partials = nullptr;
  double* sums = nullptr;     // kNumAcc (device)
  double* sums_host = nullptr;  // pinned
  double* stage_host = nullptr; // pinned n doubles
  double* flush = nullptr;
  int64_t flush_n = 0;
  int grid_cap = 0;
  int64_t launches = 0;
  bool factor_stored = false;
  // parameters of the stored factor and of the last pass (whose sums sit in `sums`): a STORE request for exactly this state is
  // already satisfied — the gradient pass of the two-observation kernel writes A, D^-1, u as well once the buffers exist
  int stored_cov = -1, last_cov = -1;
  bool stored_latent = false, last_latent = false;
  double stored_var = 0., stored_range = 0., last_var = 0., last_range = 0.;
  int knn_replayed = 0;  // queries whose neighbour set was re-derived by the exact replay of the reference walk
  std::vector<int32_t> nn_host;  // kept for the lazy CSC build
};

namespace {

void laplace_release(gpbdev_vecchia* h);  // laplace.cuh

int ensure_store_buffers(gpbdev_vecchia* h) {
  if (h->A) return 0;
  CUDA_TRY(cudaMalloc(&h->A, sizeof(double) * h->n * h->m));
  CUDA_TRY(cudaMalloc(&h->Dinv, sizeof(double) * h->n));
  CUDA_TRY(cudaMalloc(&h->u, sizeof(double) * h->n));
  CUDA_TRY(cudaMemsetAsync(h->A, 0, sizeof(double) * h->n * h->m, h->stream));
  CUDA_TRY(cudaMemsetAsync(h->u, 0, sizeof(double) * h->n, h->stream));
  CUDA_TRY(cudaMemsetAsync(h->Dinv, 0, sizeof(double) * h->n, h->stream));
  return 0;
}

// CSC view of the pattern of B restricted to this shard's rows: for column j the positions i*m+k with nn[i,k]==j
int ensure_csc(gpbdev_vecchia* h) {
  if (h->colptr) return 0;
  const int64_t n = h->n;
  const int m = h->m;
  if (h->nn_host.empty()) {
    h->nn_host.resize((size_t)n * m);
    CUDA_TRY(cudaMemcpy(h->nn_host.data(), h->nn, sizeof(int32_t) * n * m, cudaMemcpyDeviceToHost));
  }
  std::vector<int32_t> colptr(n + 1, 0);
  for (int64_t i = h->row_begin; i < h->row_end; ++i)
    for (int k = 0; k < m; ++k) {
      const int32_t j = h->nn_host[(size_t)i * m + k];
      if (j >= 0) ++colptr[j + 1];
    }
  for (int64_t j = 0; j < n; ++j) colptr[j + 1] += colptr[j];
  std::vector<int32_t> pos((size_t)colptr[n]);
  std::vector<int32_t> fill(colptr.begin(), colptr.end() - 1);
  for (int64_t i = h->row_begin; i < h->row_end; ++i)
    for (int k = 0; k < m; ++k) {
      const int32_t j = h->nn_host[(size_t)i * m + k];
      if (j >= 0) pos[fill[j]++] = (int32_t)(i * m + k);
    }
  CUDA_TRY(cudaMalloc(&h->colptr, sizeof(int32_t) * (n + 1)));
  CUDA_TRY(cudaMalloc(&h->csc_pos, sizeof(int32_t) * std::max<size_t>(pos.size(), 1)));
  CUDA_TRY(cudaMemcpy(h->colptr, colptr.data(), sizeof(int32_t) * (n + 1), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(h->csc_pos, pos.data(), sizeof(int32_t) * pos.size(), cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMalloc(&h->yaux, sizeof(double) * n));
  return 0;
}

int launch_eval(gpbdev_vecchia* h, int cov_type, double var, double range, int mode, bool latent = false) {
  if (cov_type < 0 || cov_type > 3) return fail("gpbdev_vecchia_eval: unknown covariance id");
  if (mode < 0 || mode > 3) return fail("gpbdev_vecchia_eval: unknown mode");
  if (!(var > 0.) || !(range > 0.)) return fail("gpbdev_vecchia_eval: covariance parameters must be positive");
  CUDA_TRY(cudaSetDevice(h->device));
  // GPBoost iteration: OptimCovPar's last accepted trial was a gradient pass at the final parameters on this response, and
  // CalcGradient asks for the factor at the same state right after (regression_objective.hpp:164-165): nothing to recompute.
  // GPB200_GRAD_STORES=0 switches the shortcut (and the extra stores of the gradient pass) off.
  static const bool grad_stores = []() { const char* e = std::getenv("GPB200_GRAD_STORES"); return !(e && std::string(e) == "0"); }();
  if (mode == gpb::MODE_STORE && !latent && grad_stores && h->factor_stored && h->stored_cov == cov_type && h->stored_latent == latent &&
      h->stored_var == var && h->stored_range == range && h->last_cov == cov_type && h->last_latent == latent && h->last_var == var &&
      h->last_range == range)
    return 0;
  if (mode == gpb::MODE_STORE || mode == gpb::MODE_STORE_GRAD) {
    if (ensure_store_buffers(h)) return -1;
  }
  h->last_cov = cov_type; h->last_latent = latent; h->last_var = var; h->last_range = range;
  if (mode == gpb::MODE_STORE || mode == gpb::MODE_STORE_GRAD) { h->stored_cov = cov_type; h->stored_latent = latent; h->stored_var = var; h->stored_range = range; }
  if (mode == gpb::MODE_STORE_GRAD && !h->dA) {
    CUDA_TRY(cudaMalloc(&h->dA, sizeof(double) * h->n * h->m));
    CUDA_TRY(cudaMalloc(&h->dD, sizeof(double) * h->n));
    CUDA_TRY(cudaMemsetAsync(h->dA, 0, sizeof(double) * h->n * h->m, h->stream));
    CUDA_TRY(cudaMemsetAsync(h->dD, 0, sizeof(double) * h->n, h->stream));
  }
  gpb::FactorArgs a;
  a.coords = h->coords; a.nn = h->nn; a.y = h->y;
  a.A = h->A; a.Dinv = h->Dinv; a.w = h->u;
  if (mode == gpb::MODE_GRAD && !grad_stores) a.A = nullptr;  // (only the two-observation gradient pass looks at it)
  a.partials = h->partials;
  a.n = h->n; a.row_begin = h->row_begin; a.row_end = h->row_end;
  a.m = h->m; a.d = h->d; a.var = var; a.range = range;
  a.diag_nb = latent ? var * (1. + 1e-10) : var + 1.;
  a.diag_obs = latent ? var : var + 1.;
  if (mode == gpb::MODE_STORE_GRAD) {
    CUDA_TRY(cudaMemcpyToSymbolAsync(gpb::g_factor_dA, &h->dA, sizeof(double*), 0, cudaMemcpyHostToDevice, h->stream));
    CUDA_TRY(cudaMemcpyToSymbolAsync(gpb::g_factor_dD, &h->dD, sizeof(double*), 0, cudaMemcpyHostToDevice, h->stream));
  }
  if (latent && mode == gpb::MODE_GRAD) return fail("gpbdev_vecchia_eval: the gradient pass assumes a Gaussian likelihood");
  if (h->m > gpb::kMaxNeighbors) {  // 30 < num_neighbors <= 60: shared-memory kernel (vecchia_big.cuh), same sums and factor layout
    if (mode == gpb::MODE_STORE_GRAD) return fail("gpbdev_vecchia_eval: the factor derivative (non-Gaussian likelihoods) supports num_neighbors <= 30");
    gpb::BigArgs b;
    b.coords = h->coords; b.y = h->y; b.nn = h->nn; b.qcoords = nullptr;
    b.A = h->A; b.Dinv = h->Dinv; b.w = h->u; b.pred_mean = nullptr; b.pred_var = nullptr; b.partials = h->partials;
    b.row_begin = h->row_begin; b.row_end = h->row_end; b.m = h->m; b.d = h->d;
    b.var = var; b.range = range; b.diag_nb = a.diag_nb; b.diag_obs = a.diag_obs;
    const int bmode = mode == gpb::MODE_NLL ? gpb::BIG_NLL : (mode == gpb::MODE_STORE ? gpb::BIG_STORE : gpb::BIG_GRAD);
    const int warps = bmode == gpb::BIG_GRAD ? 2 : 4;
    BigKernel bk = pick_big_kernel(cov_type, bmode);
    const size_t bsmem = gpb::big_smem_bytes(bmode, warps, h->d);
    CUDA_TRY(cudaFuncSetAttribute(bk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem));
    int grid = std::min(h->num_sms, (int)((h->grid_cap * gpb::kWarpsPerBlock) / warps));  // one CTA per SM; partials has grid_cap * 4 rows
    grid = std::max(grid, 1);
    bk<<<grid, warps * 32, bsmem, h->stream>>>(b);
    CUDA_TRY(cudaGetLastError());
    reduce_partials_kernel<<<1, 256, 0, h->stream>>>(h->partials, (int64_t)grid * warps, h->sums);
    CUDA_TRY(cudaGetLastError());
    h->launches += 2;
    if (h->allreduce && !latent) {
      if (h->allreduce(h->allreduce_ctx, h->sums, gpb::kNumAcc, (void*)h->stream)) return fail("gpbdev_vecchia_eval: device all-reduce failed");
    }
    if (mode == gpb::MODE_STORE) h->factor_stored = true;
    return 0;
  }
  // likelihood and gradient passes at the headline shape (d = 2, 20 < m <= 30): two observations per warp (vecchia_nll2.cuh);
  // GPB200_NLL_KERNEL=1 keeps the one-observation kernel
  static const bool nll1_only = []() { const char* e = std::getenv("GPB200_NLL_KERNEL"); return e && std::string(e) == "1"; }();
  if ((mode == gpb::MODE_NLL || mode == gpb::MODE_STORE || (mode == gpb::MODE_GRAD && !latent)) && h->d == 2 && h->m > 20 && !nll1_only) {
    FactorKernel k2 = nullptr;
#define GPB_PICK2(COVID)                                                                                                              \
    k2 = mode == gpb::MODE_NLL ? gpb::vecchia_nll2_kernel<COVID, gpb::MODE_NLL>                                                      \
         : (mode == gpb::MODE_STORE ? gpb::vecchia_nll2_kernel<COVID, gpb::MODE_STORE> : gpb::vecchia_nll2_kernel<COVID, gpb::MODE_GRAD>)
    switch (cov_type) {
      case gpb::COV_EXPONENTIAL: GPB_PICK2(gpb::COV_EXPONENTIAL); break;
      case gpb::COV_MATERN15: GPB_PICK2(gpb::COV_MATERN15); break;
      case gpb::COV_MATERN25: GPB_PICK2(gpb::COV_MATERN25); break;
      default: GPB_PICK2(gpb::COV_GAUSSIAN); break;
    }
#undef GPB_PICK2
    const size_t smem2 = sizeof(double) * gpb::kWarpsPerBlock * 2 * (gpb::kNll2Half + 64);
    CUDA_TRY(cudaFuncSetAttribute(k2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
    CUDA_TRY(cudaFuncSetAttribute(k2, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    int per_sm2 = 0;
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm2, k2, gpb::kWarpsPerBlock * 32, smem2));
    int grid2 = std::max(per_sm2, 1) * h->num_sms;
    grid2 = std::max(1, std::min(grid2, h->grid_cap / 2));  // two partial rows per warp
    k2<<<grid2, gpb::kWarpsPerBlock * 32, smem2, h->stream>>>(a);
    CUDA_TRY(cudaGetLastError());
    reduce_partials_kernel<<<1, 256, 0, h->stream>>>(h->partials, (int64_t)grid2 * gpb::kWarpsPerBlock * 2, h->sums);
    CUDA_TRY(cudaGetLastError());
    h->launches += 2;
    if (h->allreduce && !latent) {
      if (h->allreduce(h->allreduce_ctx, h->sums, gpb::kNumAcc, (void*)h->stream)) return fail("gpbdev_vecchia_eval: device all-reduce failed");
    }
    if (mode == gpb::MODE_STORE) h->factor_stored = true;
    if (mode == gpb::MODE_GRAD && a.A != nullptr) {  // the pass also wrote A, D^-1, u (vecchia_nll2_kernel<GRAD>)
      h->factor_stored = true;
      h->stored_cov = cov_type; h->stored_latent = false; h->stored_var = var; h->stored_range = range;
    }
    return 0;
  }
  FactorKernel k = pick_kernel(cov_type, mode, h->d, h->m);
  const size_t smem = sizeof(double) * gpb::kWarpsPerBlock * (32 * gpb::kLd + 32 * h->d + 64);
  CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  CUDA_TRY(cudaFuncSetAttribute(k, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  // persistent grid = resident CTAs per SM (registers / shared memory of this instantiation) x SM count
  int per_sm = 0;
  CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k, gpb::kWarpsPerBlock * 32, smem));
  int grid = std::max(per_sm, 1) * h->num_sms;
  if (grid > h->grid_cap) grid = h->grid_cap;
  k<<<grid, gpb::kWarpsPerBlock * 32, smem, h->stream>>>(a);
  CUDA_TRY(cudaGetLastError());
  reduce_partials_kernel<<<1, 256, 0, h->stream>>>(h->partials, (int64_t)grid * gpb::kWarpsPerBlock, h->sums);
  CUDA_TRY(cudaGetLastError());
  h->launches += 2;
  if (h->allreduce && !latent) {  // row shards: the 9 sums are summed over the ranks on this stream (NCCL kernel)
    if (h->allreduce(h->allreduce_ctx, h->sums, gpb::kNumAcc, (void*)h->stream)) return fail("gpbdev_vecchia_eval: device all-reduce failed");
  }
  if (mode == gpb::MODE_STORE || mode == gpb::MODE_STORE_GRAD) h->factor_stored = true;
  return 0;
}

}  // namespace

extern "C" {

const char* gpbdev_last_error(void) { return g_last_error.c_str(); }

int gpbdev_vecchia_set_allreduce(gpbdev_vecchia_t h, gpbdev_allreduce_fn fn, void* ctx) {
  if (!h) return fail("gpbdev_vecchia_set_allreduce: null argument");
  h->allreduce = fn;
  h->allreduce_ctx = ctx;
  return 0;
}

int gpbdev_device_count(void) {
  int c = 0;
  if (cudaGetDeviceCount(&c) != cudaSuccess) { cudaGetLastError(); return 0; }
  return c;
}

int gpbdev_vecchia_create(gpbdev_vecchia_t* out, int device, int64_t n, int d, int m, const double* coords_ordered,
                          const int32_t* perm, const int32_t* nn, int64_t row_begin, int64_t row_end) {
  if (!out || !coords_ordered || !perm) return fail("gpbdev_vecchia_create: null argument");
  if (n <= 0 || d <= 0 || d > 16) return fail("gpbdev_vecchia_create: need n > 0 and 1 <= dim <= 16");
  if (m < 1 || m > gpb::kBigMaxNeighbors)
    return fail("gpbdev_vecchia_create: num_neighbors must be in [1, " + std::to_string(gpb::kBigMaxNeighbors) +
                "] for the B200 Vecchia engine");
  if ((int64_t)n * m >= (int64_t)2147483647) return fail("gpbdev_vecchia_create: n * num_neighbors exceeds int32 positions");
  if (row_begin < 0 || row_end > n || row_begin > row_end) return fail("gpbdev_vecchia_create: bad row shard");
  if (gpbdev_device_count() <= device)
    return fail("gpbdev_vecchia_create: no CUDA device " + std::to_string(device) + " — the B200 engine has no CPU fallback");
  CUDA_TRY(cudaSetDevice(device));
  gpbdev_vecchia* h = new gpbdev_vecchia();
  h->device = device; h->n = n; h->d = d; h->m = m; h->row_begin = row_begin; h->row_end = row_end;
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  h->num_sms = prop.multiProcessorCount;
  CUDA_TRY(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  CUDA_TRY(cudaEventCreate(&h->ev0));
  CUDA_TRY(cudaEventCreate(&h->ev1));
  CUDA_TRY(cudaMalloc(&h->coords, sizeof(double) * n * d));
  CUDA_TRY(cudaMalloc(&h->nn, sizeof(int32_t) * n * m));
  CUDA_TRY(cudaMalloc(&h->perm, sizeof(int32_t) * n));
  CUDA_TRY(cudaMalloc(&h->y_in, sizeof(double) * n));
  CUDA_TRY(cudaMalloc(&h->y, sizeof(double) * n));
  CUDA_TRY(cudaMemset(h->y, 0, sizeof(double) * n));
  // upper bound of the persistent grid (the launch picks resident-CTAs-per-SM x SM count, see launch_eval)
  h->grid_cap = h->num_sms * 8;
  const int64_t rows = row_end - row_begin;
  const int64_t max_blocks = (rows + gpb::kWarpsPerBlock - 1) / gpb::kWarpsPerBlock;
  if (h->grid_cap > max_blocks) h->grid_cap = (int)std::max<int64_t>(max_blocks, 1);
  CUDA_TRY(cudaMalloc(&h->partials, sizeof(double) * h->grid_cap * gpb::kWarpsPerBlock * gpb::kNumAcc));
  CUDA_TRY(cudaMalloc(&h->sums, sizeof(double) * gpb::kNumAcc));
  CUDA_TRY(cudaMallocHost(&h->sums_host, sizeof(double) * gpb::kNumAcc));
  CUDA_TRY(cudaMallocHost(&h->stage_host, sizeof(double) * n));
  CUDA_TRY(cudaMemcpy(h->coords, coords_ordered, sizeof(double) * n * d, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(h->perm, perm, sizeof(int32_t) * n, cudaMemcpyHostToDevice));
  if (nn) {
    CUDA_TRY(cudaMemcpy(h->nn, nn, sizeof(int32_t) * n * m, cudaMemcpyHostToDevice));
    h->nn_host.assign(nn, nn + (size_t)n * m);
  } else {
    // rank of every point in the sorted coordinate sums (Vecchia_utils.cpp:775-786). The permutation of
    // equal sums is whatever std::sort yields, so the same library call is made on the same input.
    std::vector<double> csum((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
      double sacc = 0.;
      for (int k = 0; k < d; ++k) sacc += coords_ordered[i * d + k];
      csum[(size_t)i] = sacc;
    }
    std::vector<int> sort_sum((size_t)n);
    std::iota(sort_sum.begin(), sort_sum.end(), 0);
    std::sort(sort_sum.begin(), sort_sum.end(), [&csum](int i1, int i2) { return csum[i1] < csum[i2]; });
    std::vector<int32_t> pos((size_t)n);
    for (int64_t r = 0; r < n; ++r) pos[(size_t)sort_sum[(size_t)r]] = (int32_t)r;
    int32_t *pos_dev = nullptr, *sort_sum_dev = nullptr;
    double* csum_dev = nullptr;
    CUDA_TRY(cudaMalloc(&pos_dev, sizeof(int32_t) * n));
    CUDA_TRY(cudaMalloc(&sort_sum_dev, sizeof(int32_t) * n));
    CUDA_TRY(cudaMalloc(&csum_dev, sizeof(double) * n));
    CUDA_TRY(cudaMemcpy(pos_dev, pos.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(sort_sum_dev, sort_sum.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice));
    CUDA_TRY(cudaMemcpy(csum_dev, csum.data(), sizeof(double) * n, cudaMemcpyHostToDevice));
    std::string err;
    const int nl = gpb::knn_vecchia_device(h->coords, coords_ordered, n, d, m, pos_dev, sort_sum_dev, csum_dev, h->nn, h->stream,
                                           h->num_sms, &h->knn_replayed, &err);
    cudaFree(pos_dev); cudaFree(sort_sum_dev); cudaFree(csum_dev);
    if (nl < 0) { gpbdev_vecchia_free(h); return fail("gpbdev_vecchia_create: device neighbour search failed: " + err); }
    h->launches += nl;
    CUDA_TRY(cudaStreamSynchronize(h->stream));
  }
  *out = h;
  return 0;
}

int gpbdev_vecchia_free(gpbdev_vecchia_t h) {
  if (!h) return 0;
  cudaSetDevice(h->device);
  laplace_release(h);
  cudaFree(h->coords); cudaFree(h->nn); cudaFree(h->perm); cudaFree(h->y_in); cudaFree(h->y);
  cudaFree(h->dA); cudaFree(h->dD);
  cudaFree(h->A); cudaFree(h->Dinv); cudaFree(h->u); cudaFree(h->yaux); cudaFree(h->colptr); cudaFree(h->csc_pos);
  cudaFree(h->csc_row); cudaFree(h->A_csc);
  cudaFree(h->partials); cudaFree(h->sums); cudaFree(h->flush);
  cudaFreeHost(h->sums_host); cudaFreeHost(h->stage_host);
  if (h->ev0) cudaEventDestroy(h->ev0);
  if (h->ev1) cudaEventDestroy(h->ev1);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return 0;
}

int gpbdev_vecchia_get_nn(gpbdev_vecchia_t h, int32_t* nn_host) {
  if (!h || !nn_host) return fail("gpbdev_vecchia_get_nn: null argument");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaMemcpy(nn_host, h->nn, sizeof(int32_t) * h->n * h->m, cudaMemcpyDeviceToHost));
  return 0;
}

int gpbdev_vecchia_set_y_device(gpbdev_vecchia_t h, const double* y_dev) {
  if (!h || !y_dev) return fail("gpbdev_vecchia_set_y_device: null argument");
  CUDA_TRY(cudaSetDevice(h->device));
  gather_perm_kernel<<<h->num_sms * 8, 256, 0, h->stream>>>(y_dev, h->perm, h->y, h->n);
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  h->factor_stored = false;
  return 0;
}

// zero x outside [b, e)
__global__ void zero_outside_range_kernel(double* __restrict__ x, int64_t n, int64_t b, int64_t e) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    if (i < b || i >= e) x[i] = 0.;
}

int gpbdev_vecchia_set_y(gpbdev_vecchia_t h, const double* y_host) {
  if (!h || !y_host) return fail("gpbdev_vecchia_set_y: null argument");
  CUDA_TRY(cudaSetDevice(h->device));
  // Row-sharded engine with the device collective: every rank uploads only ITS slice of the response (the same index range as its
  // row shard, taken over the original order) and the slices are exchanged over NVLink (zero elsewhere + sum all-reduce) instead
  // of N full host-to-device copies of the same vector.
  const bool sliced = h->allreduce != nullptr && (h->row_begin != 0 || h->row_end != h->n);
  const int64_t b = sliced ? h->row_begin : 0, e = sliced ? h->row_end : h->n;
  cudaPointerAttributes attr;
  const bool pinned = cudaPointerGetAttributes(&attr, y_host) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  cudaGetLastError();
  if (pinned) {  // page-locked caller buffer: DMA straight from it
    CUDA_TRY(cudaMemcpyAsync(h->y_in + b, y_host + b, sizeof(double) * (e - b), cudaMemcpyHostToDevice, h->stream));
  } else {
    // pageable caller memory: stage through the engine's pinned buffer (parallel copy) so the H2D runs at link speed
    CUDA_TRY(cudaStreamSynchronize(h->stream));
    const int64_t len = e - b;
    const int64_t chunk = 1 << 16;
#pragma omp parallel for schedule(static) num_threads(8)
    for (int64_t c = 0; c < (len + chunk - 1) / chunk; ++c) {
      const int64_t lo = b + c * chunk, cl = std::min(chunk, e - lo);
      std::memcpy(h->stage_host + lo, y_host + lo, sizeof(double) * cl);
    }
    CUDA_TRY(cudaMemcpyAsync(h->y_in + b, h->stage_host + b, sizeof(double) * len, cudaMemcpyHostToDevice, h->stream));
  }
  if (sliced) {
    zero_outside_range_kernel<<<h->num_sms * 4, 256, 0, h->stream>>>(h->y_in, h->n, b, e);
    CUDA_TRY(cudaGetLastError());
    if (h->allreduce(h->allreduce_ctx, h->y_in, h->n, (void*)h->stream)) return fail("gpbdev_vecchia_set_y: device all-reduce failed");
    h->launches += 1;
  }
  return gpbdev_vecchia_set_y_device(h, h->y_in);
}

int gpbdev_vecchia_eval_async(gpbdev_vecchia_t h, int cov_type, double var, double range, int mode) {
  if (!h) return fail("gpbdev_vecchia_eval: null handle");
  return launch_eval(h, cov_type, var, range, mode);
}

int gpbdev_vecchia_get_sums(gpbdev_vecchia_t h, double* out) {
  if (!h || !out) return fail("gpbdev_vecchia_get_sums: null argument");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaMemcpyAsync(h->sums_host, h->sums, sizeof(double) * gpb::kNumAcc, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  std::memcpy(out, h->sums_host, sizeof(double) * gpb::kNumAcc);
  return 0;
}

int gpbdev_vecchia_eval(gpbdev_vecchia_t h, int cov_type, double var, double range, int mode, double* out) {
  if (!h || !out) return fail("gpbdev_vecchia_eval: null argument");
  if (launch_eval(h, cov_type, var, range, mode)) return -1;
  return gpbdev_vecchia_get_sums(h, out);
}

int gpbdev_vecchia_yaux(gpbdev_vecchia_t h, double* yaux_host) {
  if (!h || !yaux_host) return fail("gpbdev_vecchia_yaux: null argument");
  if (!h->factor_stored) return fail("gpbdev_vecchia_yaux: call gpbdev_vecchia_eval(mode=STORE) first");
  CUDA_TRY(cudaSetDevice(h->device));
  if (ensure_csc(h)) return -1;
  bt_apply_kernel<<<h->num_sms * 8, 256, 0, h->stream>>>(h->A, h->u, h->colptr, h->csc_pos, h->perm, h->yaux, h->n,
                                                         h->m, h->row_begin, h->row_end, 1.0);
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  if (h->allreduce && h->allreduce(h->allreduce_ctx, h->yaux, h->n, (void*)h->stream)) return fail("gpbdev_vecchia_yaux: device all-reduce failed");
  CUDA_TRY(cudaMemcpyAsync(h->stage_host, h->yaux, sizeof(double) * h->n, cudaMemcpyDeviceToHost, h->stream));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  std::memcpy(yaux_host, h->stage_host, sizeof(double) * h->n);
  return 0;
}

int gpbdev_vecchia_yaux_device(gpbdev_vecchia_t h, double* out_dev, double scale) {
  if (!h || !out_dev) return fail("gpbdev_vecchia_yaux_device: null argument");
  if (!h->factor_stored) return fail("gpbdev_vecchia_yaux_device: call gpbdev_vecchia_eval(mode=STORE) first");
  CUDA_TRY(cudaSetDevice(h->device));
  if (ensure_csc(h)) return -1;
  bt_apply_kernel<<<h->num_sms * 8, 256, 0, h->stream>>>(h->A, h->u, h->colptr, h->csc_pos, h->perm, out_dev, h->n, h->m,
                                                         h->row_begin, h->row_end, scale);
  CUDA_TRY(cudaGetLastError());
  h->launches += 1;
  if (h->allreduce && h->allreduce(h->allreduce_ctx, out_dev, h->n, (void*)h->stream)) return fail("gpbdev_vecchia_yaux_device: device all-reduce failed");
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  return 0;
}

// latent factor (non-Gaussian likelihood: no nugget, jitter on the neighbour blocks) with its range derivative, to host buffers:
// A, dA n x m row-major; Dinv, dD n. Test / diagnostics entry of MODE_STORE_GRAD.
// Vecchia prediction at new locations (SURVEY §8 f1), observed data ordered first, neighbours among the observed points only
// (CalcPredVecchiaObservedFirstOrder, CondObsOnly = true: src/GPBoost/Vecchia_utils.cpp:1701-2100). Uses the responses of the last
// gpbdev_vecchia_set_y*. coords_pred_host: np x d row-major. Outputs (host, np each): mean = A_p y_N(p), var = D_p on the
// transformed scale (the caller multiplies by sigma^2 and adds the nugget when the response is predicted).
int gpbdev_vecchia_predict(gpbdev_vecchia_t h, int cov_type, double var, double range, const double* coords_pred_host, int64_t np,
                           int num_neighbors_pred, double* mean_out_host, double* var_out_host) {
  if (!h || !coords_pred_host || !mean_out_host || !var_out_host) return fail("gpbdev_vecchia_predict: null argument");
  if (np <= 0) return fail("gpbdev_vecchia_predict: no prediction points");
  if (cov_type < 0 || cov_type > 3) return fail("gpbdev_vecchia_predict: unknown covariance id");
  if (!(var > 0.) || !(range > 0.)) return fail("gpbdev_vecchia_predict: covariance parameters must be positive");
  if (h->row_begin != 0 || h->row_end != h->n) return fail("gpbdev_vecchia_predict: prediction needs the whole model on this device (row-sharded engine)");
  const int64_t n = h->n;
  const int d = h->d;
  int mp = (int)std::min<int64_t>(num_neighbors_pred, n);  // Vecchia_utils.cpp:752-755
  if (mp < 1 || mp > gpb::kBigMaxNeighbors)
    return fail("gpbdev_vecchia_predict: num_neighbors_pred must be in [1, " + std::to_string(gpb::kBigMaxNeighbors) + "] for the B200 Vecchia engine");
  if ((n + np) >= (int64_t)2147483647 || np * (int64_t)mp >= (int64_t)2147483647) return fail("gpbdev_vecchia_predict: too many points for int32 indices");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  const int64_t na = n + np;
  // all points = observed (Vecchia order) followed by the prediction points; ranks in the sorted coordinate sums decide distance ties
  std::vector<double> call((size_t)na * d);
  CUDA_TRY(cudaMemcpy(call.data(), h->coords, sizeof(double) * n * d, cudaMemcpyDeviceToHost));
  std::memcpy(call.data() + (size_t)n * d, coords_pred_host, sizeof(double) * np * d);
  std::vector<double> csum((size_t)na);
  for (int64_t i = 0; i < na; ++i) {
    double sacc = 0.;
    for (int k = 0; k < d; ++k) sacc += call[(size_t)i * d + k];
    csum[(size_t)i] = sacc;
  }
  std::vector<int> sort_sum((size_t)na);
  std::iota(sort_sum.begin(), sort_sum.end(), 0);
  std::sort(sort_sum.begin(), sort_sum.end(), [&csum](int i1, int i2) { return csum[i1] < csum[i2]; });
  std::vector<int32_t> pos((size_t)na);
  for (int64_t r = 0; r < na; ++r) pos[(size_t)sort_sum[(size_t)r]] = (int32_t)r;
  double *call_dev = nullptr, *csum_dev = nullptr, *mean_dev = nullptr, *var_dev = nullptr;
  int32_t *pos_dev = nullptr, *sort_dev = nullptr, *nnp = nullptr;
  auto release = [&]() { cudaFree(call_dev); cudaFree(csum_dev); cudaFree(mean_dev); cudaFree(var_dev); cudaFree(pos_dev); cudaFree(sort_dev); cudaFree(nnp); };
  cudaError_t e = cudaMalloc(&call_dev, sizeof(double) * na * d);
  if (e == cudaSuccess) e = cudaMalloc(&csum_dev, sizeof(double) * na);
  if (e == cudaSuccess) e = cudaMalloc(&pos_dev, sizeof(int32_t) * na);
  if (e == cudaSuccess) e = cudaMalloc(&sort_dev, sizeof(int32_t) * na);
  if (e == cudaSuccess) e = cudaMalloc(&nnp, sizeof(int32_t) * np * mp);
  if (e == cudaSuccess) e = cudaMalloc(&mean_dev, sizeof(double) * np);
  if (e == cudaSuccess) e = cudaMalloc(&var_dev, sizeof(double) * np);
  if (e == cudaSuccess) e = cudaMemcpy(call_dev, call.data(), sizeof(double) * na * d, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(csum_dev, csum.data(), sizeof(double) * na, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(pos_dev, pos.data(), sizeof(int32_t) * na, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(sort_dev, sort_sum.data(), sizeof(int32_t) * na, cudaMemcpyHostToDevice);
  if (e != cudaSuccess) { release(); return fail(std::string("gpbdev_vecchia_predict: ") + cudaGetErrorString(e)); }
  std::string err;
  int replayed = 0;
  const int nl = gpb::knn_vecchia_device(call_dev, call.data(), na, d, mp, pos_dev, sort_dev, csum_dev, nnp, h->stream, h->num_sms, &replayed, &err,
                                         /*q_begin=*/n, /*end_search_at=*/n - 1);
  if (nl < 0) { release(); return fail("gpbdev_vecchia_predict: device neighbour search failed: " + err); }
  h->launches += nl;
  gpb::BigArgs b;
  b.coords = h->coords; b.y = h->y; b.nn = nnp; b.qcoords = call_dev + (size_t)n * d;
  b.A = nullptr; b.Dinv = nullptr; b.w = nullptr; b.pred_mean = mean_dev; b.pred_var = var_dev; b.partials = nullptr;
  b.row_begin = 0; b.row_end = np; b.m = mp; b.d = d;
  b.var = var; b.range = range; b.diag_nb = var + 1.; b.diag_obs = var;  // Vecchia_utils.cpp:1940-1952 (nugget on the neighbour block), :1925-1931
  BigKernel bk = pick_big_kernel(cov_type, gpb::BIG_PRED);
  const size_t bsmem = gpb::big_smem_bytes(gpb::BIG_PRED, 4, d);
  e = cudaFuncSetAttribute(bk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bsmem);
  if (e == cudaSuccess) {
    const int grid = (int)std::max<int64_t>(1, std::min<int64_t>(h->num_sms, (np + 3) / 4));
    bk<<<grid, 128, bsmem, h->stream>>>(b);
    e = cudaGetLastError();
    h->launches += 1;
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(mean_out_host, mean_dev, sizeof(double) * np, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaMemcpyAsync(var_out_host, var_dev, sizeof(double) * np, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  release();
  if (e != cudaSuccess) return fail(std::string("gpbdev_vecchia_predict: ") + cudaGetErrorString(e));
  return 0;
}

int gpbdev_vecchia_latent_factor_grad(gpbdev_vecchia_t h, int cov_type, double var, double range, double* A_host, double* Dinv_host,
                                      double* dA_host, double* dD_host) {
  if (!h || !A_host || !Dinv_host || !dA_host || !dD_host) return fail("gpbdev_vecchia_latent_factor_grad: null argument");
  if (launch_eval(h, cov_type, var, range, gpb::MODE_STORE_GRAD, true)) return -1;
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaMemcpy(A_host, h->A, sizeof(double) * h->n * h->m, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(Dinv_host, h->Dinv, sizeof(double) * h->n, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(dA_host, h->dA, sizeof(double) * h->n * h->m, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(dD_host, h->dD, sizeof(double) * h->n, cudaMemcpyDeviceToHost));
  return 0;
}

int gpbdev_vecchia_get_factor(gpbdev_vecchia_t h, double* A_host, double* Dinv_host) {
  if (!h || !A_host || !Dinv_host) return fail("gpbdev_vecchia_get_factor: null argument");
  if (!h->factor_stored) return fail("gpbdev_vecchia_get_factor: call gpbdev_vecchia_eval(mode=STORE) first");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  CUDA_TRY(cudaMemcpy(A_host, h->A, sizeof(double) * h->n * h->m, cudaMemcpyDeviceToHost));
  CUDA_TRY(cudaMemcpy(Dinv_host, h->Dinv, sizeof(double) * h->n, cudaMemcpyDeviceToHost));
  return 0;
}

int gpbdev_vecchia_timer_start(gpbdev_vecchia_t h) {
  if (!h) return fail("null handle");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaEventRecord(h->ev0, h->stream));
  return 0;
}
int gpbdev_vecchia_timer_stop(gpbdev_vecchia_t h, float* ms) {
  if (!h || !ms) return fail("null argument");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaEventRecord(h->ev1, h->stream));
  CUDA_TRY(cudaEventSynchronize(h->ev1));
  CUDA_TRY(cudaEventElapsedTime(ms, h->ev0, h->ev1));
  return 0;
}
int gpbdev_vecchia_sync(gpbdev_vecchia_t h) {
  if (!h) return fail("null handle");
  CUDA_TRY(cudaSetDevice(h->device));
  CUDA_TRY(cudaStreamSynchronize(h->stream));
  return 0;
}
int64_t gpbdev_vecchia_launch_count(gpbdev_vecchia_t h) { return h ? h->launches : 0; }
int gpbdev_vecchia_knn_replayed(gpbdev_vecchia_t h) { return h ? h->knn_replayed : 0; }

int gpbdev_fp64_peak(int device, double* tflops) {
  if (!tflops) return fail("null argument");
  CUDA_TRY(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, device));
  double* out = nullptr;
  CUDA_TRY(cudaMalloc(&out, 8));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 1 << 14;
  fp64_peak_kernel<<<blocks, threads>>>(out, 1 << 10, 1.0000001, 1e-9);
  double best = 0.;
  for (int rep = 0; rep < 5; ++rep) {
    CUDA_TRY(cudaEventRecord(e0));
    fp64_peak_kernel<<<blocks, threads>>>(out, iters, 1.0000001, 1e-9);
    CUDA_TRY(cudaEventRecord(e1));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0.f;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 8 * (double)iters * blocks * threads;
    best = std::max(best, flops / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
  *tflops = best;
  return 0;
}

int gpbdev_vecchia_flush_l2(gpbdev_vecchia_t h) {
  if (!h) return fail("null handle");
  CUDA_TRY(cudaSetDevice(h->device));
  if (!h->flush) {
    h->flush_n = (int64_t)(256 << 20) / sizeof(double);  // 256 MiB > 126 MB L2
    CUDA_TRY(cudaMalloc(&h->flush, sizeof(double) * h->flush_n));
  }
  fill_kernel<<<h->num_sms * 8, 256, 0, h->stream>>>(h->flush, h->flush_n, 1.0);
  CUDA_TRY(cudaGetLastError());
  return 0;
}

}  // extern "C"

#include "newton.cuh"
#include "laplace.cuh"
