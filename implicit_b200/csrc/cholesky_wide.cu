// R1 for 64 < padded factors <= 128: one CTA per row, normal equations accumulated in a
// (F/16 x F/16) register tile per thread with exact fp32 FMAs, then a CTA-wide in-shared-memory
// Cholesky (reference: _least_squares, implicit/cpu/_als.pyx:76-142).
//
// This is the correctness path for wide models (recalculate_user / partial_fit on a factors=128 CG
// model, `use_cg=False` at factors=100); the register-resident tensor-core kernel in cholesky.cu
// covers factors <= 64, where BASELINE.json quotes the Cholesky metric.
#include <limits.h>

#include "common.h"

namespace als {
namespace {

constexpr int kWideThreads = 256;
constexpr int kWideStage = 16;  // nonzeros staged per step

template <int T>
struct WideCfg {
  static constexpr int F = 16 * T;
  static constexpr int LDA = F + 1;
  static constexpr int SMEM_FLOATS = F * LDA + F /*b*/ + kWideStage * F + 2 * kWideStage + 8;
  static constexpr int SLOT_FLOATS = F * F + F;
};

template <int T>
__global__ void __launch_bounds__(kWideThreads)
cholesky_wide_kernel(const int32_t *__restrict__ indices, const float *__restrict__ data, const float *__restrict__ Y,
                     float *__restrict__ X, int64_t row_offset, const float *__restrict__ Greg,
                     const WorkItem *__restrict__ work, int n_work, float *slots, long long *bad_row, int pass,
                     float *const *peers, int n_peers) {
  using C = WideCfg<T>;
  constexpr int F = C::F, LDA = C::LDA;
  extern __shared__ __align__(16) float smem[];
  float *As = smem;                       // [F][LDA]
  float *bs = As + F * LDA;               // [F]
  float *ys = bs + F;                     // [kWideStage][F]
  float *ws = ys + kWideStage * F;        // [kWideStage]
  float *cs = ws + kWideStage;            // [kWideStage]
  int *flag = reinterpret_cast<int *>(cs + kWideStage);
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;

  for (int item = blockIdx.x; item < n_work; item += gridDim.x) {
    const WorkItem wi = work[item];
    const bool whole = wi.slot == -1, chunk = wi.slot >= 0, finish = wi.slot == -2;
    float *xout = X + (row_offset + wi.row) * F;
    __syncthreads();
    if (whole && wi.k0 == wi.k1) {  // empty row -> zeros (_als.pyx:98-100)
      for (int m = tid; m < F; m += kWideThreads) {
        xout[m] = 0.f;
        for (int pi = 0; pi < n_peers; ++pi) peers[pi][(row_offset + wi.row) * F + m] = 0.f;
      }
      continue;
    }
    float acc[T][T], bacc[T];
#pragma unroll
    for (int i = 0; i < T; ++i) {
      bacc[i] = 0.f;
#pragma unroll
      for (int j = 0; j < T; ++j) acc[i][j] = chunk ? 0.f : Greg[(ty + 16 * i) * F + tx + 16 * j];
    }
    if (pass == 0) {
      for (int k0 = wi.k0; k0 < wi.k1; k0 += kWideStage) {
        __syncthreads();
        for (int e = tid; e < kWideStage * (F / 4); e += kWideThreads) {
          const int r = e / (F / 4), c4 = e % (F / 4);
          float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
          if (k0 + r < wi.k1) v = __ldg(reinterpret_cast<const float4 *>(Y + (int64_t)indices[k0 + r] * F) + c4);
          reinterpret_cast<float4 *>(ys + r * F)[c4] = v;
        }
        if (tid < kWideStage) {
          const bool valid = k0 + tid < wi.k1;
          const float c = valid ? data[k0 + tid] : 0.f;
          ws[tid] = valid ? fabsf(c) - 1.f : 0.f;  // _als.pyx:115-124
          cs[tid] = c > 0.f ? c : 0.f;
        }
        __syncthreads();
#pragma unroll 4
        for (int r = 0; r < kWideStage; ++r) {
          const float w = ws[r], cp = cs[r];
          float a[T], b[T];
#pragma unroll
          for (int i = 0; i < T; ++i) {
            a[i] = ys[r * F + ty + 16 * i];
            b[i] = ys[r * F + tx + 16 * i];
          }
#pragma unroll
          for (int i = 0; i < T; ++i) {
            const float wa = w * a[i];
#pragma unroll
            for (int j = 0; j < T; ++j) acc[i][j] = fmaf(wa, b[j], acc[i][j]);
          }
          if (ty == 0) {
#pragma unroll
            for (int j = 0; j < T; ++j) bacc[j] = fmaf(cp, b[j], bacc[j]);
          }
        }
      }
    } else {
      for (int s = 0; s < wi.k1; ++s) {  // finish: add the chunk partials in slot order
        const float *sl = slots + (int64_t)(wi.k0 + s) * C::SLOT_FLOATS;
#pragma unroll
        for (int i = 0; i < T; ++i) {
#pragma unroll
          for (int j = 0; j < T; ++j) acc[i][j] += sl[(ty + 16 * i) * F + tx + 16 * j];
          if (ty == 0) bacc[i] += sl[F * F + tx + 16 * i];
        }
      }
    }
    if (chunk) {
      float *sl = slots + (int64_t)wi.slot * C::SLOT_FLOATS;
#pragma unroll
      for (int i = 0; i < T; ++i) {
#pragma unroll
        for (int j = 0; j < T; ++j) sl[(ty + 16 * i) * F + tx + 16 * j] = acc[i][j];
        if (ty == 0) sl[F * F + tx + 16 * i] = bacc[i];
      }
      continue;
    }
    if (!(whole || finish)) continue;
    // ---- A, b to shared memory; upper Cholesky U^T U = A with the forward solve riding along
    __syncthreads();
#pragma unroll
    for (int i = 0; i < T; ++i) {
#pragma unroll
      for (int j = 0; j < T; ++j) As[(ty + 16 * i) * LDA + tx + 16 * j] = acc[i][j];
      if (ty == 0) bs[tx + 16 * i] = bacc[i];
    }
    if (tid == 0) *flag = 0;
    __syncthreads();
    for (int k = 0; k < F; ++k) {
      const float d = As[k * LDA + k];
      if (!(d > 0.f)) {
        if (tid == 0) *flag = 1;
        break;  // uniform: every thread reads the same d
      }
      float s = rsqrtf(d);
      s = s * fmaf(-0.5f * d * s, s, 1.5f);
      __syncthreads();
      for (int j = k + 1 + tid; j < F; j += kWideThreads) As[k * LDA + j] *= s;
      if (tid == 0) {
        As[k * LDA + k] = s;  // the diagonal keeps the reciprocal pivot
        bs[k] *= s;
      }
      __syncthreads();
      const float zk = bs[k];
      for (int i = k + 1 + ty; i < F; i += 16) {
        const float uki = As[k * LDA + i];
        for (int j = i + ((tx - i) & 15); j < F; j += 16)  // j >= i, j == tx (mod 16)
          As[i * LDA + j] = fmaf(-uki, As[k * LDA + j], As[i * LDA + j]);
        if (tx == 0) bs[i] = fmaf(-uki, zk, bs[i]);
      }
      __syncthreads();
    }
    __syncthreads();
    if (*flag) {
      if (tid == 0) atomicMin(bad_row, (long long)(row_offset + wi.row));
      continue;
    }
    // ---- back substitution U x = z (column oriented)
    for (int k = F - 1; k >= 0; --k) {
      if (tid == 0) bs[k] *= As[k * LDA + k];
      __syncthreads();
      const float xk = bs[k];
      for (int i = tid; i < k; i += kWideThreads) bs[i] = fmaf(-As[i * LDA + k], xk, bs[i]);
      __syncthreads();
    }
    for (int m = tid; m < F; m += kWideThreads) {
      xout[m] = bs[m];
      for (int pi = 0; pi < n_peers; ++pi) peers[pi][(row_offset + wi.row) * F + m] = bs[m];
    }
  }
}

// Like init_solver_scalars (cholesky.cu): [1] keeps the first bad row of every half since the last als_solver_status.
// Resetting [0] alone lost a failed half of 65..128 factors that the asynchronous (multi-GPU) fit had not collected
// yet: the next half erased it and als_solver_status reported nothing (tests/test_gpu_width_sweep.py, f = 80, 128).
__global__ void init_bad_row(long long *bad_row) {
  if (bad_row[0] < bad_row[1]) bad_row[1] = bad_row[0];
  bad_row[0] = LLONG_MAX;
}

template <int T>
int run_wide(als_ctx *ctx, const als_csr *Cm, als_factors *X, const als_factors *Y) {
  using C = WideCfg<T>;
  const int smem = C::SMEM_FLOATS * (int)sizeof(float);
  auto kern = cholesky_wide_kernel<T>;
  ALS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  float *slots = nullptr;
  if (Cm->n_slots) {
    int rc = ensure_scratch(ctx, (int64_t)Cm->n_slots * C::SLOT_FLOATS * (int64_t)sizeof(float));
    if (rc != ALS_OK) return rc;
    slots = (float *)ctx->scratch;
  }
  init_bad_row<<<1, 1, 0, ctx->stream>>>(ctx->bad_row);
  ALS_CUDA(cudaGetLastError());
  ctx->launches++;
  const int per_sm = std::max(1, (227 * 1024) / (smem + 1024));
  if (Cm->n_work) {
    const int grid = (int)std::min<int64_t>(Cm->n_work, (int64_t)ctx->sm_count * per_sm);
    ProfScope prof(ctx, kProfCholesky);
    kern<<<grid, kWideThreads, smem, ctx->stream>>>(Cm->indices, Cm->data, Y->d, X->d, Cm->row_offset, ctx->Greg, Cm->work,
                                                    (int)Cm->n_work, slots, ctx->bad_row, 0, X->peers_dev, X->n_peers);
    ALS_CUDA(cudaGetLastError());
    ctx->launches++;
  }
  if (Cm->n_finish) {
    const int grid = (int)std::min<int64_t>(Cm->n_finish, (int64_t)ctx->sm_count * per_sm);
    ProfScope prof(ctx, kProfCholFinish);
    kern<<<grid, kWideThreads, smem, ctx->stream>>>(Cm->indices, Cm->data, Y->d, X->d, Cm->row_offset, ctx->Greg,
                                                    Cm->finish, (int)Cm->n_finish, slots, ctx->bad_row, 1, X->peers_dev, X->n_peers);
    ALS_CUDA(cudaGetLastError());
    ctx->launches++;
  }
  return ALS_OK;
}

}  // namespace

int launch_cholesky_wide(als_ctx *ctx, const als_csr *C, als_factors *X, const als_factors *Y) {
  switch (Y->ld / 16) {
    case 5: return run_wide<5>(ctx, C, X, Y);
    case 6: return run_wide<6>(ctx, C, X, Y);
    case 7: return run_wide<7>(ctx, C, X, Y);
    case 8: return run_wide<8>(ctx, C, X, Y);
    default:
      set_error("cholesky: factors=%d (padded %d) is not supported: the Cholesky solver covers factors <= 128, wider models use CG", Y->f, Y->ld);
      return ALS_E_UNSUPPORTED;
  }
}

}  // namespace als
