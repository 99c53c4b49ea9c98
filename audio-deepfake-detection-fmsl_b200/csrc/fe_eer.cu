// On-device ROC / EER / "min_dcf" of the evaluation sweep (SURVEY 8f-2), bit-compatible with what the reference
// computes on the host with scikit-learn (Thesis/02_Evaluation_Scripts/Maze5_eval.py:588-594;
// score_file_processor.py:176-196):
//     fpr, tpr, thr = sklearn.metrics.roc_curve(y, s)        # drop_intermediate=True
//     fnr = 1 - tpr;  eer = fpr[nanargmin |fnr - fpr|];  min_dcf = min(fnr + fpr)
// roc_curve (scikit-learn _ranking.py): stable sort by decreasing score, one point per DISTINCT score (the last index
// of each run of equal scores), tps = cumsum(y)[idx], fps = 1 + idx - tps, points whose second differences of fps and
// tps both vanish are dropped (first and last kept), a leading (0, 0, inf) point, division by the totals in float64.
//
// One launch, one CTA of 1024 threads (the sweep has 71,237 scores; the whole job is a few hundred KB and lives in
// L2): a stable LSD radix sort of (score key, label) records -- 4-bit digits, every thread owns a contiguous chunk,
// per-thread digit counters in shared memory, so no atomics and a fixed order -- then the distinct-score compaction,
// the pruning rule and the argmin / min reductions, all in float64 where the reference is.  Scores stay on the device
// from the classifier to the three numbers; nothing is synchronised until the caller reads them.
#include <cuda_runtime.h>
#include <stdint.h>

#include "fe_common.h"
#include "fe_kernels.h"

namespace {

constexpr int kThreads = 1024;
constexpr int kDigits = 16;   // 4-bit digits: 16 x 1024 counters = 64 KB of shared memory

struct eer_ws {
  unsigned long long* rec[2];   // ping-pong records: key << 32 | label
  unsigned int* d_idx;          // per distinct score: index of the last element of its run
  unsigned int* d_tps;          // per distinct score: positives up to and including that index
};

// descending-score order as an ascending unsigned key
__device__ __forceinline__ unsigned int score_key(float s) {
  const unsigned int u = __float_as_uint(s);
  const unsigned int asc = u ^ ((u >> 31) ? 0xffffffffu : 0x80000000u);
  return ~asc;
}
__device__ __forceinline__ float key_score(unsigned int k) {
  const unsigned int asc = ~k;
  const unsigned int u = (asc >> 31) ? (asc ^ 0x80000000u) : ~asc;
  return __uint_as_float(u);
}

// inclusive block scan of one value per thread (1024 threads); returns the inclusive prefix, *total = block sum
__device__ unsigned int block_scan_incl(unsigned int v, unsigned int* s_warp, unsigned int* total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned int y = __shfl_up_sync(0xffffffffu, x, o);
    if (lane >= o) x += y;
  }
  __syncthreads();   // s_warp may still be read from a previous call
  if (lane == 31) s_warp[warp] = x;
  __syncthreads();
  if (warp == 0) {
    unsigned int w = s_warp[lane];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned int y = __shfl_up_sync(0xffffffffu, w, o);
      if (lane >= o) w += y;
    }
    s_warp[lane] = w;
  }
  __syncthreads();
  if (total) *total = s_warp[31];
  return x + (warp > 0 ? s_warp[warp - 1] : 0u);
}

__global__ void __launch_bounds__(kThreads, 1) fe_eer_kernel(const float* __restrict__ scores, const int32_t* __restrict__ labels,
                                                            int64_t n64, eer_ws ws, double* out) {
  extern __shared__ unsigned int s_hist[];   // [digit][thread]
  __shared__ unsigned int s_warp[32];
  __shared__ double s_best_a[32], s_best_d[32];
  __shared__ unsigned int s_best_i[32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned int n = (unsigned int)n64;
  const unsigned int per = (n + kThreads - 1) / kThreads;
  const unsigned int lo = min(n, tid * per), hi = min(n, lo + per);

  // ---- records ------------------------------------------------------------------------------------
  bool nonfinite_here = false;
  for (unsigned int i = tid; i < n; i += kThreads) {
    const float sc = scores[i];
    nonfinite_here |= !isfinite(sc);
    ws.rec[0][i] = ((unsigned long long)score_key(sc) << 32) | (unsigned long long)(labels[i] == 1 ? 1u : 0u);
  }
  if (__syncthreads_or(nonfinite_here)) {   // scikit-learn's roc_curve raises on NaN and infinite scores; here: status 2
    if (tid == 0) { out[0] = out[1] = out[2] = 0.0; out[3] = 2.0; }
    return;
  }

  // ---- stable LSD radix sort on the 32-bit key, 4 bits per pass ---------------------------------------
  int cur = 0;
  for (int shift = 32; shift < 64; shift += 4) {
    const unsigned long long* src = ws.rec[cur];
    unsigned long long* dst = ws.rec[cur ^ 1];
#pragma unroll
    for (int d = 0; d < kDigits; ++d) s_hist[d * kThreads + tid] = 0;
    for (unsigned int i = lo; i < hi; ++i) s_hist[(unsigned int)((src[i] >> shift) & 15u) * kThreads + tid]++;
    __syncthreads();
    // exclusive scan over the flattened [digit][thread] array: thread t owns entries 16 t .. 16 t + 15
    unsigned int loc[kDigits], sum = 0;
#pragma unroll
    for (int j = 0; j < kDigits; ++j) { loc[j] = s_hist[tid * kDigits + j]; sum += loc[j]; }
    unsigned int run = block_scan_incl(sum, s_warp, nullptr) - sum;
#pragma unroll
    for (int j = 0; j < kDigits; ++j) { const unsigned int c = loc[j]; s_hist[tid * kDigits + j] = run; run += c; }
    __syncthreads();
    for (unsigned int i = lo; i < hi; ++i) {
      const unsigned long long r = src[i];
      dst[s_hist[(unsigned int)((r >> shift) & 15u) * kThreads + tid]++] = r;
    }
    __syncthreads();
    cur ^= 1;
  }
  const unsigned long long* rec = ws.rec[cur];

  // ---- one point per distinct score: tps = cumsum(y)[idx], idx = last index of the run ------------------
  unsigned int pos_local = 0, dis_local = 0;
  for (unsigned int i = lo; i < hi; ++i) {
    const unsigned long long r = rec[i];
    pos_local += (unsigned int)(r & 1ull);
    const bool last = (i + 1 == n) || (key_score((unsigned int)(rec[i + 1] >> 32)) != key_score((unsigned int)(r >> 32)));
    dis_local += last ? 1u : 0u;
  }
  unsigned int n_pos = 0, n_dis = 0;
  unsigned int pos_run = block_scan_incl(pos_local, s_warp, &n_pos) - pos_local;
  unsigned int dis_run = block_scan_incl(dis_local, s_warp, &n_dis) - dis_local;
  for (unsigned int i = lo; i < hi; ++i) {
    const unsigned long long r = rec[i];
    pos_run += (unsigned int)(r & 1ull);
    const bool last = (i + 1 == n) || (key_score((unsigned int)(rec[i + 1] >> 32)) != key_score((unsigned int)(r >> 32)));
    if (last) {
      ws.d_idx[dis_run] = i;
      ws.d_tps[dis_run] = pos_run;
      ++dis_run;
    }
  }
  __syncthreads();
  const unsigned int n_neg = n - n_pos;
  if (n_pos == 0 || n_neg == 0 || n == 0) {   // EER needs both classes (Maze5_eval.py:577-582 returns {} then)
    if (tid == 0) { out[0] = out[1] = out[2] = 0.0; out[3] = 1.0; }
    return;
  }

  // ---- pruning rule + argmin |fnr - fpr| (first minimum) + min (fnr + fpr) over the kept points ----------
  const double P = (double)n_pos, N = (double)n_neg;
  double best_a = 1.0, best_d = 1.0;     // the leading (0, 0, inf) point: fnr = 1, fpr = 0
  unsigned int best_i = 0;               // index into the roc arrays: 0 = the leading point, j + 1 = distinct point j
  for (unsigned int j = tid; j < n_dis; j += kThreads) {
    const long long tps = ws.d_tps[j], fps = (long long)ws.d_idx[j] + 1 - tps;
    bool keep = (j == 0) || (j + 1 == n_dis);
    if (!keep) {
      const long long tp0 = ws.d_tps[j - 1], tp1 = ws.d_tps[j + 1];
      const long long fp0 = (long long)ws.d_idx[j - 1] + 1 - tp0, fp1 = (long long)ws.d_idx[j + 1] + 1 - tp1;
      keep = (fp1 - 2 * fps + fp0 != 0) || (tp1 - 2 * tps + tp0 != 0);
    }
    if (!keep) continue;
    const double fpr = (double)fps / N, tpr = (double)tps / P;
    const double fnr = 1.0 - tpr;
    const double a = fabs(fnr - fpr), d = fnr + fpr;
    if (a < best_a) { best_a = a; best_i = j + 1; }   // j ascends within a thread: a strict < keeps the first minimum
    best_d = fmin(best_d, d);
  }
  // block reduction: smallest a, ties -> smallest roc index
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double a2 = __shfl_xor_sync(0xffffffffu, best_a, o);
    const unsigned int i2 = __shfl_xor_sync(0xffffffffu, best_i, o);
    const double d2 = __shfl_xor_sync(0xffffffffu, best_d, o);
    if (a2 < best_a || (a2 == best_a && i2 < best_i)) { best_a = a2; best_i = i2; }
    best_d = fmin(best_d, d2);
  }
  if (lane == 0) { s_best_a[warp] = best_a; s_best_i[warp] = best_i; s_best_d[warp] = best_d; }
  __syncthreads();
  if (warp == 0) {
    best_a = s_best_a[lane]; best_i = s_best_i[lane]; best_d = s_best_d[lane];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double a2 = __shfl_xor_sync(0xffffffffu, best_a, o);
      const unsigned int i2 = __shfl_xor_sync(0xffffffffu, best_i, o);
      const double d2 = __shfl_xor_sync(0xffffffffu, best_d, o);
      if (a2 < best_a || (a2 == best_a && i2 < best_i)) { best_a = a2; best_i = i2; }
      best_d = fmin(best_d, d2);
    }
    if (lane == 0) {
      double eer = 0.0, thr = __longlong_as_double(0x7ff0000000000000ll);   // leading point: fpr 0, threshold inf
      if (best_i > 0) {
        const unsigned int j = best_i - 1;
        const long long tps = ws.d_tps[j], fps = (long long)ws.d_idx[j] + 1 - tps;
        eer = (double)fps / N;
        thr = (double)key_score((unsigned int)(rec[ws.d_idx[j]] >> 32));
      }
      out[0] = eer; out[1] = best_d; out[2] = thr; out[3] = 0.0;
    }
  }
}

}  // namespace

extern "C" int64_t b200fe_eer_workspace_bytes(int64_t n) {
  if (n < 0 || n > ((int64_t)1 << 30)) return B200FE_ERR_BAD_ARG;
  const int64_t m = (n + 1) & ~(int64_t)1;
  return 2 * m * 8 + 2 * m * 4 + 64;
}

extern "C" int32_t b200fe_eer_min_dcf(const float* scores, const int32_t* labels, int64_t n, double* out4, void* workspace,
                                      size_t workspace_bytes, void* stream) {
  if (!scores || !labels || !out4 || !workspace || n < 1 || n > ((int64_t)1 << 30)) {
    fe_set_error("b200fe_eer_min_dcf: bad arguments (n = %lld)", (long long)n);
    return B200FE_ERR_BAD_ARG;
  }
  if ((int64_t)workspace_bytes < b200fe_eer_workspace_bytes(n)) {
    fe_set_error("b200fe_eer_min_dcf: workspace too small");
    return B200FE_ERR_WORKSPACE;
  }
  if (((uintptr_t)workspace & 15) != 0) {
    fe_set_error("b200fe_eer_min_dcf: workspace must be 16-byte aligned");
    return B200FE_ERR_ALIGNMENT;
  }
  const int64_t m = (n + 1) & ~(int64_t)1;
  eer_ws ws;
  char* w = (char*)workspace;
  ws.rec[0] = (unsigned long long*)w;             w += m * 8;
  ws.rec[1] = (unsigned long long*)w;             w += m * 8;
  ws.d_idx = (unsigned int*)w;                    w += m * 4;
  ws.d_tps = (unsigned int*)w;
  const int smem = kDigits * kThreads * 4;
  cudaError_t e = cudaFuncSetAttribute(fe_eer_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (e == cudaSuccess) {
    fe_eer_kernel<<<1, kThreads, smem, (cudaStream_t)stream>>>(scores, labels, n, ws, out4);
    e = cudaGetLastError();
  }
  if (e != cudaSuccess) {
    fe_set_error("b200fe_eer_min_dcf: %s", cudaGetErrorString(e));
    return B200FE_ERR_CUDA;
  }
  return B200FE_OK;
}
