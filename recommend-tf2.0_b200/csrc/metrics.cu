// Keras AUC (ROC curve, trapezoid summation, evenly spaced thresholds) — the one number every
// CTR training script of the reference reports (`metrics=[AUC()]`, `model.evaluate`,
// src/ctr/fm/train.py:50,58,67; semantics SURVEY.md App. A19):
//   bucket(p) = max(ceilf(p * (T-1)) - 1, 0)   (one fp32 multiply, then ceilf)
//   tp[i] = sum_{j>=i} pos[j],  fp[i] = sum_{j>=i} neg[j]
//   AUC = sum_{i<T-1} (fpr[i] - fpr[i+1]) * (tpr[i] + tpr[i+1]) / 2
// rtf_auc_update keeps per-bucket integer counts (order-independent sums: bit-reproducible);
// rtf_auc_result forms the suffix sums and the trapezoid in fp64 in a fixed order.
#include "rtf_common.cuh"

namespace rtf {

constexpr int AUC_MAX_T = 4096;     // 2 * 4096 * 4 B = 32 KB of static shared memory
constexpr int AUC_THREADS = 256, AUC_PER = 4;
// a CTA's 32-bit shared-memory counts must not wrap: it visits at most this many elements
constexpr long long AUC_CTA_MAX = 1LL << 30;

// counts[0][b] += positives in bucket b, counts[1][b] += negatives.  Elements with p outside
// [0, 1], p NaN or a label other than 0 / 1 are not counted and set bit 0 of *err.
__global__ void __launch_bounds__(AUC_THREADS)
auc_update_kernel(const float* __restrict__ pred, const float* __restrict__ label, long long n,
                  int T, unsigned long long* __restrict__ counts, int* __restrict__ err) {
  __shared__ unsigned int hist[2 * AUC_MAX_T];
  for (int i = threadIdx.x; i < 2 * T; i += AUC_THREADS) hist[i] = 0u;
  __syncthreads();
  const float tm1 = (float)(T - 1);
  const int lane = threadIdx.x & 31;
  bool bad = false;
  const long long stride = (long long)gridDim.x * AUC_THREADS * AUC_PER;
  // the loop condition is the warp's first element: all 32 lanes stay in step for the match
  for (long long wbase = (long long)blockIdx.x * AUC_THREADS * AUC_PER + (threadIdx.x & ~31);
       wbase < n; wbase += stride) {
    const long long base = wbase + lane;
    float pv[AUC_PER], yv[AUC_PER];
#pragma unroll
    for (int e = 0; e < AUC_PER; ++e) {       // all loads first: AUC_PER in flight per thread
      const long long i = base + (long long)e * AUC_THREADS;
      pv[e] = i < n ? __ldg(pred + i) : 0.f;
      yv[e] = i < n ? __ldg(label + i) : 0.f;
    }
#pragma unroll
    for (int e = 0; e < AUC_PER; ++e) {
      const long long i = base + (long long)e * AUC_THREADS;
      int key = -1;
      if (i < n) {
        const float p = pv[e], y = yv[e];
        if (p >= 0.f && p <= 1.f && (y == 0.f || y == 1.f)) {     // NaN fails both compares
          const int b = max((int)ceilf(__fmul_rn(p, tm1)) - 1, 0);
          key = (y == 1.f ? 0 : T) + b;
        } else {
          bad = true;
        }
      }
      // warp-aggregated increment: the predictions of a trained model cluster in a few buckets,
      // so lanes sharing a bin elect one leader that adds the group's size (one shared atomic
      // per distinct bin instead of up to 32 serialised on one address)
      const unsigned peers = __match_any_sync(0xffffffffu, key);
      if (key >= 0 && lane == __ffs(peers) - 1) atomicAdd(&hist[key], (unsigned)__popc(peers));
    }
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(err, 1);
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * T; i += AUC_THREADS) {
    const unsigned c = hist[i];
    if (c) atomicAdd(counts + i, (unsigned long long)c);     // hist and counts are both [2][T]
  }
}

// One CTA.  Thread t owns the buckets [t*chunk, (t+1)*chunk): it needs tp / fp at the first
// bucket past its range (the suffix sums of the chunks above it) and walks its range downwards,
// adding its trapezoid terms in descending bucket order; thread 0 then adds the per-thread sums
// in ascending thread order.  The order depends on T only: the result is reproducible.
__global__ void __launch_bounds__(AUC_THREADS)
auc_result_kernel(const unsigned long long* __restrict__ counts, int T, float* __restrict__ auc) {
  __shared__ unsigned long long cpos[AUC_THREADS + 1], cneg[AUC_THREADS + 1];
  __shared__ double part[AUC_THREADS];
  const int t = threadIdx.x;
  const int chunk = (T + AUC_THREADS - 1) / AUC_THREADS;
  const int lo = min(t * chunk, T), hi = min(lo + chunk, T);
  unsigned long long sp = 0, sn = 0;
  for (int i = lo; i < hi; ++i) {
    sp += counts[i];
    sn += counts[T + i];
  }
  cpos[t] = sp;
  cneg[t] = sn;
  __syncthreads();
  if (t == 0) {     // suffix sums over the chunks: cpos[t] = tp at bucket t*chunk
    unsigned long long ap = 0, an = 0;
    cpos[AUC_THREADS] = cneg[AUC_THREADS] = 0;
    for (int k = AUC_THREADS - 1; k >= 0; --k) {
      ap += cpos[k];
      an += cneg[k];
      cpos[k] = ap;
      cneg[k] = an;
    }
  }
  __syncthreads();
  const unsigned long long P = cpos[0], N = cneg[0];
  // divide_no_nan: with no positives (negatives) every tpr (fpr) is 0
  const double ip = P ? 1.0 / (double)P : 0.0, in = N ? 1.0 / (double)N : 0.0;
  unsigned long long tp = cpos[t + 1], fp = cneg[t + 1];     // at bucket hi
  double tpr1 = (double)tp * ip, fpr1 = (double)fp * in;
  double acc = 0.0;
  for (int i = hi - 1; i >= lo; --i) {
    tp += counts[i];
    fp += counts[T + i];
    const double tpr0 = (double)tp * ip, fpr0 = (double)fp * in;
    if (i < T - 1) acc += (fpr0 - fpr1) * (tpr0 + tpr1) * 0.5;
    tpr1 = tpr0;
    fpr1 = fpr0;
  }
  part[t] = acc;
  __syncthreads();
  if (t == 0) {
    double s = 0.0;
    for (int k = 0; k < AUC_THREADS; ++k) s += part[k];
    *auc = (float)s;
  }
}

}  // namespace rtf

using namespace rtf;

extern "C" int rtf_auc_update(const float* d_pred, const float* d_label, int64_t n,
                              int num_thresholds, unsigned long long* d_counts, int* d_err,
                              void* stream) {
  if (!d_pred || !d_label || !d_counts || !d_err || n < 0) return RTF_E_ARG;
  if (num_thresholds < 2 || num_thresholds > AUC_MAX_T) return RTF_E_RANGE;
  if (n == 0) return 0;
  const long long per_cta = (long long)AUC_THREADS * AUC_PER;
  long long grid = (n + per_cta - 1) / per_cta;
  grid = grid < 4LL * kNumSMs ? grid : 4LL * kNumSMs;     // enough to fill HBM, few flushes
  const long long need = (n + AUC_CTA_MAX - 1) / AUC_CTA_MAX;
  grid = grid > need ? grid : need;
  auc_update_kernel<<<(unsigned)grid, AUC_THREADS, 0, (cudaStream_t)stream>>>(
      d_pred, d_label, n, num_thresholds, d_counts, d_err);
  RTF_CHECK_LAUNCH();
  return 0;
}

extern "C" int rtf_auc_result(const unsigned long long* d_counts, int num_thresholds, float* d_auc,
                              void* stream) {
  if (!d_counts || !d_auc) return RTF_E_ARG;
  if (num_thresholds < 2 || num_thresholds > AUC_MAX_T) return RTF_E_RANGE;
  auc_result_kernel<<<1, AUC_THREADS, 0, (cudaStream_t)stream>>>(d_counts, num_thresholds, d_auc);
  RTF_CHECK_LAUNCH();
  return 0;
}
