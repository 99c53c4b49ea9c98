// C-ABI entry points that touch the device (include/b200fe.h).  Host-only entry points live in
// fe_tables.cpp.  Nothing here allocates device memory: tables, workspace, staging and outputs all
// belong to the caller.
#include <cuda_runtime.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>

#include "fe_common.h"
#include "fe_gemm.h"
#include "fe_kernels.h"

namespace {

thread_local int64_t g_launches = 0;

// Energies of one chunk of rows (the workspace between the energies kernel and the tail).  Round 1 kept a chunk inside
// the 126 MB L2 (48 MB); measured on B200 the launch ramps and tails of three small launches cost more than the extra
// 64 KB per utterance of DRAM traffic when the energies spill (the path runs at a quarter of the HBM roofline):
// 48 MB 4.11 M utt/s, 96 MB 4.26 M, >= 140 MB (one chunk for 4096 rows) 4.40 M (profiles/r2_chunk_size_sweep.txt).
// B200FE_WS_MB overrides the target (measurement hook).
int64_t ws_target_bytes() {
  static const int64_t v = [] {
    const char* e = getenv("B200FE_WS_MB");
    const long mb = e ? atol(e) : 0;
    return (int64_t)(mb >= 1 && mb <= 4096 ? mb : 160) << 20;
  }();
  return v;
}

int32_t cuda_fail(cudaError_t e, const char* what) {
  fe_set_error("%s: %s", what, cudaGetErrorString(e));
  return B200FE_ERR_CUDA;
}

int32_t check_device() {
  // per device ordinal: a process may drive several GPUs (0 unknown, 1 ok); a failed check is not cached
  static std::atomic<int> cached[kFeMaxDevices];
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) { fe_set_error("cudaGetDevice: %s", cudaGetErrorString(e)); return B200FE_ERR_NO_DEVICE; }
  if (dev >= 0 && dev < kFeMaxDevices && cached[dev].load(std::memory_order_relaxed) == 1) return B200FE_OK;
  int major = 0;
  e = cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev);
  if (e != cudaSuccess) { fe_set_error("cudaDeviceGetAttribute: %s", cudaGetErrorString(e)); return B200FE_ERR_NO_DEVICE; }
  if (major != 10) {
    fe_set_error("device compute capability %d.x: this library is built for sm_100a only", major);
    return B200FE_ERR_NO_DEVICE;
  }
  if (dev >= 0 && dev < kFeMaxDevices) cached[dev].store(1, std::memory_order_relaxed);
  return B200FE_OK;
}

bool needs_group_max(const b200fe_params* p) { return p->log_mode == B200FE_LOG_DB && p->top_db >= 0.0f; }

int64_t group_count(const b200fe_params* p, int64_t R) { return (R + p->top_db_group - 1) / p->top_db_group; }

int64_t group_max_bytes(const b200fe_params* p, int64_t R) {
  return needs_group_max(p) ? ((group_count(p, R) * 4 + 255) & ~(int64_t)255) : 0;
}

// Rows whose filterbank energies are materialised at once.
int64_t chunk_rows_for(const b200fe_params* p, int64_t R, int64_t n_frames) {
  if (needs_group_max(p) && p->top_db_group > 1) return R;  // maxima span rows: finish all rows first
  const int64_t per_row = (int64_t)p->n_filter * n_frames * 4;
  int64_t c = ws_target_bytes() / (per_row > 0 ? per_row : 1);
  if (c < 148) c = 148;
  return c < R ? c : R;
}

int pick_tt(int n_frames) {
  const int tiles = (n_frames + 127) / 128;
  int tt = (n_frames + tiles - 1) / tiles;
  tt = (tt + 7) & ~7;
  return tt < 8 ? 8 : tt;
}

int32_t common_checks(const b200fe_params* p, const void* wave, int64_t R, int64_t T, const void* tables,
                      const void* out, int wave_align = 4) {
  int32_t st = fe_validate_params(p);
  if (st != B200FE_OK) return st;
  if (!wave || !tables || !out) { fe_set_error("wave / tables / out is NULL"); return B200FE_ERR_BAD_ARG; }
  if (R < 1) { fe_set_error("R=%lld must be >= 1", (long long)R); return B200FE_ERR_BAD_ARG; }
  if (T > 0x7fffffffLL / 2) { fe_set_error("T=%lld too long", (long long)T); return B200FE_ERR_UNSUPPORTED; }
  if (T <= p->n_fft / 2) {
    fe_set_error("T=%lld must exceed n_fft/2=%d for reflect padding", (long long)T, p->n_fft / 2);
    return B200FE_ERR_BAD_ARG;
  }
  if (((uintptr_t)tables & 15) != 0) { fe_set_error("tables must be 16-byte aligned"); return B200FE_ERR_ALIGNMENT; }
  if (((uintptr_t)wave & (wave_align - 1)) != 0 || ((uintptr_t)out & 3) != 0) {
    if (wave_align == 4) fe_set_error("wave / out must be 4-byte aligned");
    else fe_set_error("wave must be %d-byte and out 4-byte aligned", wave_align);
    return B200FE_ERR_ALIGNMENT;
  }
  return check_device();
}

}  // namespace

extern "C" int64_t b200fe_last_launch_count(void) { return g_launches; }

extern "C" int32_t b200fe_has_tcgen05(void) { return fe_gemm_compiled(); }

extern "C" int32_t b200fe_resolve_variant(const b200fe_params* p) {
  int32_t st = fe_validate_params(p);
  if (st != B200FE_OK) return st;
  if (p->variant == B200FE_VARIANT_FFT) return B200FE_VARIANT_FFT;
  const bool ok = fe_gemm_supported(p);
  if (p->variant == B200FE_VARIANT_DFT_GEMM) {
    if (!ok) {
      fe_set_error("variant dft_gemm does not support this configuration");
      return B200FE_ERR_UNSUPPORTED;
    }
    return B200FE_VARIANT_DFT_GEMM;
  }
  return (ok && fe_gemm_preferred(p)) ? B200FE_VARIANT_DFT_GEMM : B200FE_VARIANT_FFT;
}

// The streaming tcgen05 kernel fetches dense rows with TMA boxes: ragged clips and pre-emphasised input are
// first written as dense rows (one chunk at a time) into the workspace.
static bool needs_dense_rows(const b200fe_params* p, bool ragged) {
  return p->variant == B200FE_VARIANT_DFT_GEMM && (ragged || p->preemph != 0.0f);
}

// pcm16: 16-bit PCM input, which both kernel families read only as staged dense float32 rows
static int64_t dense_rows_bytes(const b200fe_params* p, bool ragged, bool pcm16, int64_t chunk, int64_t T) {
  return (pcm16 || needs_dense_rows(p, ragged)) ? ((chunk * T * 4 + 255) & ~(int64_t)255) : 0;
}

static int64_t features_workspace_bytes(const b200fe_params* p, int64_t R, int64_t T, bool ragged, bool pcm16) {
  const int64_t nf = b200fe_n_frames(p, T);
  if (nf < 0) return nf;
  if (R < 1) { fe_set_error("R=%lld must be >= 1", (long long)R); return B200FE_ERR_BAD_ARG; }
  if (p->n_filter < 1) { fe_set_error("n_filter must be >= 1 for the feature path"); return B200FE_ERR_BAD_ARG; }
  const int64_t chunk = chunk_rows_for(p, R, nf);
  return group_max_bytes(p, R) + ((fe_align16(chunk * p->n_filter * nf * 4) + 255) & ~(int64_t)255) +
         dense_rows_bytes(p, ragged, pcm16, chunk, T) + fe_gemm_workspace_bytes(p, chunk, T);
}

extern "C" int64_t b200fe_workspace_bytes_ex(const b200fe_params* p, int64_t R, int64_t T, int32_t ragged) {
  return features_workspace_bytes(p, R, T, ragged != 0, false);
}

extern "C" int64_t b200fe_workspace_bytes_ragged_i16(const b200fe_params* p, int64_t R, int64_t T) {
  return features_workspace_bytes(p, R, T, true, true);
}

extern "C" int64_t b200fe_workspace_bytes(const b200fe_params* p, int64_t R, int64_t T) {
  return b200fe_workspace_bytes_ex(p, R, T, 0);
}

extern "C" int32_t b200fe_spectrogram_forward(const float* wave, int64_t R, int64_t T, const b200fe_params* p,
                                              const void* tables, float* out, void* stream) {
  g_launches = 0;
  int32_t st = common_checks(p, wave, R, T, tables, out);
  if (st != B200FE_OK) return st;
  const int n_freq = p->n_fft / 2 + 1;
  const int ft = fe_fft_pick_ft(p->n_fft, p->hop_length, n_freq, 0);
  if (ft == 0) { fe_set_error("n_fft=%d hop=%d does not fit shared memory", p->n_fft, p->hop_length); return B200FE_ERR_UNSUPPORTED; }
  fe_fft_args a;
  memset(&a, 0, sizeof(a));
  a.wave = wave;
  a.tables = tables;
  a.out = out;
  a.T = T;
  a.n_fft = p->n_fft;
  a.hop = p->hop_length;
  a.n_frames = (int32_t)(1 + T / p->hop_length);
  a.n_filter = 0;
  a.ft = ft;
  a.tiles_per_row = (a.n_frames + ft - 1) / ft;
  a.radix2_first = (__builtin_ctz(p->n_fft / 2) & 1);
  a.top_db_group = 1;
  a.preemph = p->preemph;
  // keep each launch's grid below 2^31 CTAs
  const int64_t max_rows = 0x7fffffffLL / a.tiles_per_row;
  for (int64_t r0 = 0; r0 < R; r0 += max_rows) {
    const int64_t nr = R - r0 < max_rows ? R - r0 : max_rows;
    a.row_base = r0;
    a.out = out + (size_t)r0 * n_freq * a.n_frames;
    cudaError_t e = fe_launch_fft(a, 0, nr, (cudaStream_t)stream);
    if (e != cudaSuccess) return cuda_fail(e, "spectrogram kernel launch");
    ++g_launches;
  }
  return B200FE_OK;
}

// wave: float32 samples, or 16-bit PCM (pcm16: ragged only; every row is staged as dense float32 rows, x / 32768)
static int32_t run_features(const void* wave_, bool pcm16, int64_t R, int64_t T, const int64_t* offsets,
                            const int32_t* lengths, const b200fe_params* p, const void* tables,
                            float* out, void* workspace, size_t workspace_bytes, void* stream_,
                            bool energies_only) {
  g_launches = 0;
  const float* wave = (const float*)wave_;
  int32_t st = common_checks(p, wave_, R, T, tables, out, pcm16 ? 2 : 4);
  if (st != B200FE_OK) return st;
  if ((offsets == nullptr) != (lengths == nullptr) || (pcm16 && offsets == nullptr)) {
    fe_set_error(pcm16 ? "16-bit PCM input needs offsets and lengths"
                       : "offsets and lengths must both be given or both be NULL");
    return B200FE_ERR_BAD_ARG;
  }
  if (p->n_filter < 1) { fe_set_error("n_filter must be >= 1 for the feature path"); return B200FE_ERR_BAD_ARG; }
  const int64_t need = features_workspace_bytes(p, R, T, offsets != nullptr, pcm16);
  if (need < 0) return (int32_t)need;
  if (!workspace || workspace_bytes < (size_t)need) {
    fe_set_error("workspace: %zu bytes given, %lld needed", workspace_bytes, (long long)need);
    return B200FE_ERR_WORKSPACE;
  }
  if (((uintptr_t)workspace & 15) != 0) { fe_set_error("workspace must be 16-byte aligned"); return B200FE_ERR_ALIGNMENT; }
  // AUTO is resolved by the caller against the host copy of the tables (b200fe_tables_variant);
  // a forward call that still says AUTO only sees the device copy and takes the FFT variant.
  int32_t variant = B200FE_VARIANT_FFT;
  if (p->variant == B200FE_VARIANT_DFT_GEMM) {
    if (!fe_gemm_supported(p)) {
      fe_set_error("variant dft_gemm does not support this configuration");
      return B200FE_ERR_UNSUPPORTED;
    }
    if (!fe_stream_supported(p, T, R) ||
        (!pcm16 && !needs_dense_rows(p, offsets != nullptr) && ((uintptr_t)wave & 15) != 0)) {
      fe_set_error("variant dft_gemm needs T %% 4 == 0, T > n_fft/2 and a 16-byte aligned waveform (TMA)");
      return B200FE_ERR_UNSUPPORTED;
    }
    variant = B200FE_VARIANT_DFT_GEMM;
  }

  cudaStream_t stream = (cudaStream_t)stream_;
  const int n_frames = (int)(1 + T / p->hop_length);
  const int n_out = (int)b200fe_n_out_channels(p);
  const int64_t chunk = chunk_rows_for(p, R, n_frames);
  unsigned int* gmax = needs_group_max(p) ? (unsigned int*)workspace : nullptr;
  float* energies = (float*)((char*)workspace + group_max_bytes(p, R));
  float* dense = (float*)((char*)energies + ((fe_align16(chunk * p->n_filter * (int64_t)n_frames * 4) + 255) & ~(int64_t)255));
  const bool staged = pcm16 || (variant == B200FE_VARIANT_DFT_GEMM && needs_dense_rows(p, offsets != nullptr));
  void* gemm_ws = (char*)dense + dense_rows_bytes(p, offsets != nullptr, pcm16, chunk, T);
  const size_t row_energy_floats = (size_t)p->n_filter * n_frames;

  if (gmax) {
    cudaError_t e = cudaMemsetAsync(gmax, 0, (size_t)group_count(p, R) * 4, stream);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(group_max)");
  }

  fe_fft_args fa;
  memset(&fa, 0, sizeof(fa));
  fa.wave = wave;
  fa.offsets = offsets;
  fa.lengths = lengths;
  fa.tables = tables;
  fa.out = energies;
  fa.group_max = gmax;
  fa.T = T;
  fa.n_fft = p->n_fft;
  fa.hop = p->hop_length;
  fa.n_frames = n_frames;
  fa.n_filter = p->n_filter;
  fa.radix2_first = (__builtin_ctz(p->n_fft / 2) & 1);
  fa.top_db_group = p->top_db_group;
  fa.preemph = p->preemph;
  if (variant == B200FE_VARIANT_FFT) {
    fa.ft = fe_fft_pick_ft(p->n_fft, p->hop_length, p->n_filter, 1);
    if (fa.ft == 0) { fe_set_error("n_fft=%d hop=%d does not fit shared memory", p->n_fft, p->hop_length); return B200FE_ERR_UNSUPPORTED; }
    fa.tiles_per_row = (n_frames + fa.ft - 1) / fa.ft;
  }

  fe_tail_args ta;
  memset(&ta, 0, sizeof(ta));
  ta.energies = energies;
  ta.group_max = gmax;
  ta.tables = tables;
  ta.out = out;
  ta.n_frames = n_frames;
  ta.n_filter = p->n_filter;
  ta.n_coef = p->n_coef;
  ta.n_out = n_out;
  ta.log_mode = p->log_mode;
  ta.deltas = p->deltas;
  ta.delta_win = p->deltas > 0 ? p->delta_win : 3;
  ta.top_db_group = p->top_db_group;
  ta.top_db = p->top_db;
  ta.tt = pick_tt(n_frames);
  ta.halo = p->deltas * ((ta.delta_win - 1) / 2);
  {  // test hook: compare the tail kernels (B200FE_GENERIC_TAIL=1: fe_tail_kernel, =fast: fe_tail_fast_kernel)
    const char* g = getenv("B200FE_GENERIC_TAIL");
    ta.force_generic = g ? (g[0] == 'f' ? 2 : 1) : 0;
  }
  if (fe_tail_smem_bytes(ta) > 200 * 1024) {
    fe_set_error("n_filter=%d n_coef=%d does not fit the tail kernel's shared memory", p->n_filter, p->n_coef);
    return B200FE_ERR_UNSUPPORTED;
  }

  for (int64_t r0 = 0; r0 < R; r0 += chunk) {
    const int64_t nr = R - r0 < chunk ? R - r0 : chunk;
    cudaError_t e;
    if (energies_only) fa.out = out + (size_t)r0 * row_energy_floats;
    if (pcm16) {
      // every row staged (pre-emphasis included), then read as dense rows of this chunk by either kernel family
      e = fe_launch_dense_rows((const int16_t*)wave_, offsets, lengths, r0, nr, T, p->preemph, dense, stream);
      if (e != cudaSuccess) return cuda_fail(e, "dense-rows kernel launch");
      g_launches += (nr + 65534) / 65535;
      fe_fft_args fs = fa;
      fs.wave = nullptr;
      fs.wave_chunk = dense;
      fs.offsets = nullptr;
      fs.lengths = nullptr;
      fs.preemph = 0.0f;
      if (variant == B200FE_VARIANT_DFT_GEMM) {
        int launches = 0;
        e = fe_stream_launch(p, fs, r0, nr, gemm_ws, stream, &launches);
        if (e != cudaSuccess) return cuda_fail(e, "dft-gemm kernel launch");
        g_launches += launches;
      } else {
        fs.row_base = r0;
        e = fe_launch_fft(fs, 1, nr, stream);
        if (e != cudaSuccess) return cuda_fail(e, "fft kernel launch");
        ++g_launches;
      }
    } else if (variant == B200FE_VARIANT_DFT_GEMM) {
      int launches = 0;
      if (staged) {
        // Ragged clips that pad() only truncates (len >= T) and that start 16-byte aligned are read where they lie
        // (the tensor maps then count 16-byte units above the lower of the two buffers); only the others -- short
        // clips (repeat-pad), unaligned ones, and everything when pre-emphasis is on -- are staged as dense rows.
        int64_t flat_rel = -1, dense_rel = 0;
        const float* base = dense;
        if (offsets && lengths && p->preemph == 0.0f && ((uintptr_t)wave & 15) == 0 && !getenv("B200FE_STAGE_ALL")) {
          const uintptr_t lo = (uintptr_t)wave < (uintptr_t)dense ? (uintptr_t)wave : (uintptr_t)dense;
          const int64_t fr = (int64_t)(((uintptr_t)wave - lo) / 4), dr = (int64_t)(((uintptr_t)dense - lo) / 4);
          if (((dr + nr * T) >> 2) < kFeInPlaceReach) {
            base = (const float*)lo;
            flat_rel = fr;
            dense_rel = dr;
          }
        }
        e = fe_launch_dense_rows(wave, offsets, lengths, r0, nr, T, p->preemph, dense, stream, flat_rel);
        if (e != cudaSuccess) return cuda_fail(e, "dense-rows kernel launch");
        g_launches += (nr + 65534) / 65535;
        fe_fft_args fs = fa;
        fs.wave_chunk = dense;
        if (flat_rel >= 0) {
          fs.wave = base;
          fs.in_place = 1;
          fs.flat_rel = flat_rel;
          fs.dense_rel = dense_rel;
        } else {
          fs.offsets = nullptr;
          fs.lengths = nullptr;
        }
        e = fe_stream_launch(p, fs, r0, nr, gemm_ws, stream, &launches);
      } else {
        e = fe_stream_launch(p, fa, r0, nr, gemm_ws, stream, &launches);
      }
      if (e != cudaSuccess) return cuda_fail(e, "dft-gemm kernel launch");
      g_launches += launches;
    } else {
      fa.row_base = r0;
      e = fe_launch_fft(fa, 1, nr, stream);
      if (e != cudaSuccess) return cuda_fail(e, "fft kernel launch");
      ++g_launches;
    }
    if (energies_only) continue;
    ta.row_base = r0;
    e = fe_launch_tail(ta, nr, stream);
    if (e != cudaSuccess) return cuda_fail(e, "tail kernel launch");
    g_launches += (nr + 65534) / 65535;
  }
  if (p->cmvn && !energies_only) {
    cudaError_t e = fe_launch_cmvn(out, R * n_out, n_frames, stream);
    if (e != cudaSuccess) return cuda_fail(e, "cmvn kernel launch");
    ++g_launches;
  }
  return B200FE_OK;
}

extern "C" int32_t b200fe_features_forward(const float* wave, int64_t R, int64_t T, const int64_t* offsets,
                                           const int32_t* lengths, const b200fe_params* p, const void* tables,
                                           float* out, void* workspace, size_t workspace_bytes, void* stream) {
  return run_features(wave, false, R, T, offsets, lengths, p, tables, out, workspace, workspace_bytes, stream, false);
}

extern "C" int32_t b200fe_features_forward_ragged_i16(const int16_t* pcm, int64_t R, int64_t T, const int64_t* offsets,
                                                      const int32_t* lengths, const b200fe_params* p, const void* tables,
                                                      float* out, void* workspace, size_t workspace_bytes, void* stream) {
  return run_features(pcm, true, R, T, offsets, lengths, p, tables, out, workspace, workspace_bytes, stream, false);
}

extern "C" int32_t b200fe_fbank_energies_forward(const float* wave, int64_t R, int64_t T, const int64_t* offsets,
                                                 const int32_t* lengths, const b200fe_params* p, const void* tables,
                                                 float* out, void* workspace, size_t workspace_bytes, void* stream) {
  return run_features(wave, false, R, T, offsets, lengths, p, tables, out, workspace, workspace_bytes, stream, true);
}

extern "C" int32_t b200fe_lfcc_forward(const float* wave, int64_t R, int64_t T, const int64_t* offsets,
                                       const int32_t* lengths, const b200fe_params* p, const void* tables,
                                       float* out, void* workspace, size_t workspace_bytes, void* stream) {
  if (p && p->n_coef < 1) { fe_set_error("b200fe_lfcc_forward needs n_coef >= 1"); return B200FE_ERR_BAD_ARG; }
  return b200fe_features_forward(wave, R, T, offsets, lengths, p, tables, out, workspace, workspace_bytes, stream);
}

extern "C" int32_t b200fe_mel_forward(const float* wave, int64_t R, int64_t T, const int64_t* offsets,
                                      const int32_t* lengths, const b200fe_params* p, const void* tables,
                                      float* out, void* workspace, size_t workspace_bytes, void* stream) {
  if (p && p->n_coef != 0) { fe_set_error("b200fe_mel_forward needs n_coef == 0"); return B200FE_ERR_BAD_ARG; }
  return b200fe_features_forward(wave, R, T, offsets, lengths, p, tables, out, workspace, workspace_bytes, stream);
}

extern "C" int32_t b200fe_compute_deltas(const float* in, int64_t rows, int64_t T, int32_t win, float* out,
                                         void* stream) {
  g_launches = 0;
  if (!in || !out) { fe_set_error("in / out is NULL"); return B200FE_ERR_BAD_ARG; }
  if (rows < 1 || T < 1) { fe_set_error("rows=%lld T=%lld must be >= 1", (long long)rows, (long long)T); return B200FE_ERR_BAD_ARG; }
  if (win < 3) { fe_set_error("win_length=%d must be >= 3", win); return B200FE_ERR_BAD_ARG; }
  if ((win & 1) == 0 || win > 9) { fe_set_error("win_length=%d must be odd and <= 9", win); return B200FE_ERR_UNSUPPORTED; }
  int32_t st = check_device();
  if (st != B200FE_OK) return st;
  cudaError_t e = fe_launch_deltas(in, out, rows, T, win, (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_fail(e, "deltas kernel launch");
  g_launches = (rows + 65534) / 65535;
  return B200FE_OK;
}

// ---- host-buffer path ---------------------------------------------------------------------------
namespace {
// What the host loop streams: dense rows [R][T], or ragged clips (offsets != NULL) in a flat buffer of n_samples.
struct host_input {
  const void* data;
  int32_t sample_bytes;      // 2 = 16-bit PCM (converted x / 32768 on the device), 4 = float32
  const int64_t* offsets;    // host clip table (ragged), else NULL
  const int32_t* lengths;
  int64_t n_samples;
};

// Ragged chunks: the copy span of a chunk holds up to chunk_rows * (T + kSpanSlack) samples, so that chunk_rows clips of
// at most T samples packed with up to kSpanSlack samples of alignment slack between them fit one slot.
constexpr int64_t kSpanSlack = 16;

// One slot per stream: [input | clip table | float32 rows | features | workspace of the dense forward call]
struct host_slot_layout {
  int64_t in_bytes, idx_bytes, wave_bytes, out_bytes, ws_bytes, slot_bytes;
};

// params of the dense forward call of a ragged chunk: pre-emphasis is applied while the rows are staged
b200fe_params staged_params(const b200fe_params* p) {
  b200fe_params q = *p;
  q.preemph = 0.0f;
  return q;
}

int32_t host_layout(const b200fe_params* p, int64_t chunk_rows, int64_t T, int32_t sample_bytes, bool ragged,
                    host_slot_layout* L) {
  const int64_t nf = b200fe_n_frames(p, T);
  if (nf < 0) return (int32_t)nf;
  const int64_t n_out = b200fe_n_out_channels(p);
  const b200fe_params q = ragged ? staged_params(p) : *p;
  const int64_t ws = b200fe_workspace_bytes(&q, chunk_rows, T);
  if (ws < 0) return (int32_t)ws;
  if (ragged) {
    L->in_bytes = (chunk_rows * (T + kSpanSlack) * sample_bytes + 255) & ~(int64_t)255;
    L->idx_bytes = ((chunk_rows * 8 + 255) & ~(int64_t)255) + ((chunk_rows * 4 + 255) & ~(int64_t)255);
  } else {
    L->in_bytes = sample_bytes == 2 ? ((chunk_rows * T * 2 + 255) & ~(int64_t)255) : 0;
    L->idx_bytes = 0;
  }
  L->wave_bytes = (chunk_rows * T * 4 + 255) & ~(int64_t)255;
  L->out_bytes = (chunk_rows * n_out * nf * 4 + 255) & ~(int64_t)255;
  L->ws_bytes = (ws + 255) & ~(int64_t)255;
  L->slot_bytes = L->in_bytes + L->idx_bytes + L->wave_bytes + L->out_bytes + L->ws_bytes;
  return B200FE_OK;
}

int64_t host_staging_bytes(const b200fe_params* p, int64_t chunk_rows, int64_t T, int32_t n_streams,
                           int32_t sample_bytes, bool ragged) {
  if (chunk_rows < 1 || n_streams < 1 || n_streams > 4) {
    fe_set_error("chunk_rows=%lld n_streams=%d out of range", (long long)chunk_rows, n_streams);
    return B200FE_ERR_BAD_ARG;
  }
  if (sample_bytes != 2 && sample_bytes != 4) {
    fe_set_error("sample_bytes=%d must be 2 (16-bit PCM) or 4 (float32)", sample_bytes);
    return B200FE_ERR_BAD_ARG;
  }
  host_slot_layout L;
  int32_t st = host_layout(p, chunk_rows, T, sample_bytes, ragged, &L);
  if (st != B200FE_OK) return st;
  return L.slot_bytes * n_streams;
}

// The checks forward_ragged's validation makes on the device, made here on the host copy of the clip table.
int32_t check_clip_table(const host_input& in, int64_t R) {
  for (int64_t r = 0; r < R; ++r) {
    const int64_t off = in.offsets[r], len = in.lengths[r];
    if (len < 1) {
      fe_set_error("ragged input: clip %lld has %lld samples (every clip needs at least one)", (long long)r, (long long)len);
      return B200FE_ERR_BAD_ARG;
    }
    if (off < 0 || off > in.n_samples - len) {
      fe_set_error("ragged input: clip %lld (offset %lld, %lld samples) lies outside the flat buffer of %lld samples",
                   (long long)r, (long long)off, (long long)len, (long long)in.n_samples);
      return B200FE_ERR_BAD_ARG;
    }
  }
  return B200FE_OK;
}

// Rows [r0, r0 + n) of a ragged chunk: at most max_rows rows whose copy span -- from the lowest offset to the highest
// offset + min(length, T): pad() reads no further -- holds at most cap samples.  One row always fits (cap >= T).
int64_t ragged_chunk(const host_input& in, int64_t r0, int64_t max_rows, int64_t T, int64_t cap, int64_t* lo,
                     int64_t* hi) {
  int64_t a = in.offsets[r0], b = a + (in.lengths[r0] < T ? in.lengths[r0] : T);
  int64_t n = 1;
  for (; n < max_rows; ++n) {
    const int64_t o = in.offsets[r0 + n], e = o + (in.lengths[r0 + n] < T ? in.lengths[r0 + n] : T);
    const int64_t a2 = o < a ? o : a, b2 = e > b ? e : b;
    if (b2 - a2 > cap) break;
    a = a2;
    b = b2;
  }
  *lo = a;
  *hi = b;
  return n;
}

// One loop for dense rows and ragged clips; a chunk goes to stream c % n_streams and its slot:
//   dense:  H2D rows -> (16-bit PCM: x / 32768) -> dense forward -> D2H features
//   ragged: H2D copy span, H2D clip table slice -> stage dense rows (pad(), x / 32768, pre-emphasis) -> dense forward
//           without pre-emphasis -> D2H features
int32_t forward_host(const host_input& in, int64_t R, int64_t T, const b200fe_params* p, const void* tables,
                     float* out_host, void* staging, size_t staging_bytes, int64_t chunk_rows, void* const* streams,
                     int32_t n_streams) {
  int64_t launches = 0;
  g_launches = 0;
  const bool ragged = in.offsets != nullptr;
  if (!in.data || !out_host || !staging || !streams || !p) { fe_set_error("NULL argument"); return B200FE_ERR_BAD_ARG; }
  if (R < 1) { fe_set_error("R=%lld must be >= 1", (long long)R); return B200FE_ERR_BAD_ARG; }
  if (p->top_db_group > 1 && p->log_mode == B200FE_LOG_DB && p->top_db >= 0.0f) {
    fe_set_error("the host-buffer path needs top_db_group == 1 (chunks are finished independently)");
    return B200FE_ERR_UNSUPPORTED;
  }
  const int64_t need = host_staging_bytes(p, chunk_rows, T, n_streams, in.sample_bytes, ragged);
  if (need < 0) return (int32_t)need;
  if (staging_bytes < (size_t)need) {
    fe_set_error("staging: %zu bytes given, %lld needed", staging_bytes, (long long)need);
    return B200FE_ERR_WORKSPACE;
  }
  if (((uintptr_t)staging & 255) != 0) { fe_set_error("staging must be 256-byte aligned"); return B200FE_ERR_ALIGNMENT; }
  if (ragged) {
    int32_t st = check_clip_table(in, R);
    if (st != B200FE_OK) return st;
  }
  host_slot_layout L;
  host_layout(p, chunk_rows, T, in.sample_bytes, ragged, &L);
  const b200fe_params q = ragged ? staged_params(p) : *p;
  const int64_t nf = b200fe_n_frames(p, T);
  const int64_t n_out = b200fe_n_out_channels(p);
  const size_t in_elt = (size_t)in.sample_bytes;
  const bool pcm16 = in.sample_bytes == 2;
  const int64_t span_cap = chunk_rows * (T + kSpanSlack);
  int64_t c = 0;
  for (int64_t r0 = 0; r0 < R; ++c) {
    const int64_t max_rows = R - r0 < chunk_rows ? R - r0 : chunk_rows;
    int64_t lo = 0, hi = 0;
    const int64_t nr = ragged ? ragged_chunk(in, r0, max_rows, T, span_cap, &lo, &hi) : max_rows;
    const int s = (int)(c % n_streams);
    cudaStream_t st = (cudaStream_t)streams[s];
    char* slot = (char*)staging + (size_t)s * L.slot_bytes;
    void* d_in = slot;
    char* d_idx = slot + L.in_bytes;
    float* d_wave = (float*)(d_idx + L.idx_bytes);
    float* d_out = (float*)((char*)d_wave + L.wave_bytes);
    void* d_ws = (char*)d_out + L.out_bytes;
    cudaError_t e;
    if (!ragged) {
      // one copy per chunk and direction
      e = cudaMemcpyAsync(pcm16 ? d_in : (void*)d_wave, (const char*)in.data + (size_t)r0 * T * in_elt,
                          (size_t)nr * T * in_elt, cudaMemcpyHostToDevice, st);
      if (e != cudaSuccess) return cuda_fail(e, "H2D copy");
      if (pcm16) {
        e = fe_launch_i16_rows((const int16_t*)d_in, d_wave, nr * T, st);
        if (e != cudaSuccess) return cuda_fail(e, "pcm16 conversion kernel launch");
        ++launches;
      }
    } else {
      int64_t* d_off = (int64_t*)d_idx;
      int32_t* d_len = (int32_t*)(d_idx + ((chunk_rows * 8 + 255) & ~(int64_t)255));
      e = cudaMemcpyAsync(d_in, (const char*)in.data + (size_t)lo * in_elt, (size_t)(hi - lo) * in_elt,
                          cudaMemcpyHostToDevice, st);
      if (e != cudaSuccess) return cuda_fail(e, "H2D copy");
      e = cudaMemcpyAsync(d_off, in.offsets + r0, (size_t)nr * 8, cudaMemcpyHostToDevice, st);
      if (e != cudaSuccess) return cuda_fail(e, "H2D copy (offsets)");
      e = cudaMemcpyAsync(d_len, in.lengths + r0, (size_t)nr * 4, cudaMemcpyHostToDevice, st);
      if (e != cudaSuccess) return cuda_fail(e, "H2D copy (lengths)");
      e = pcm16 ? fe_launch_dense_rows((const int16_t*)d_in, d_off, d_len, 0, nr, T, p->preemph, d_wave, st, lo)
                : fe_launch_dense_rows((const float*)d_in, d_off, d_len, 0, nr, T, p->preemph, d_wave, st, -1, lo);
      if (e != cudaSuccess) return cuda_fail(e, "dense-rows kernel launch");
      launches += (nr + 65534) / 65535;
    }
    int32_t rc = b200fe_features_forward(d_wave, nr, T, nullptr, nullptr, &q, tables, d_out, d_ws, (size_t)L.ws_bytes, st);
    if (rc != B200FE_OK) return rc;
    launches += g_launches;
    e = cudaMemcpyAsync(out_host + (size_t)r0 * n_out * nf, d_out, (size_t)nr * n_out * nf * 4, cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) return cuda_fail(e, "D2H copy");
    r0 += nr;
  }
  for (int s = 0; s < n_streams; ++s) {
    cudaError_t e = cudaStreamSynchronize((cudaStream_t)streams[s]);
    if (e != cudaSuccess) return cuda_fail(e, "cudaStreamSynchronize");
  }
  g_launches = launches;
  return B200FE_OK;
}

host_input dense_input(const void* rows, int32_t sample_bytes) { return host_input{rows, sample_bytes, nullptr, nullptr, 0}; }
}  // namespace

extern "C" int64_t b200fe_host_staging_bytes(const b200fe_params* p, int64_t chunk_rows, int64_t T, int32_t n_streams) {
  return host_staging_bytes(p, chunk_rows, T, n_streams, 4, false);
}

extern "C" int64_t b200fe_host_staging_bytes_i16(const b200fe_params* p, int64_t chunk_rows, int64_t T, int32_t n_streams) {
  return host_staging_bytes(p, chunk_rows, T, n_streams, 2, false);
}

extern "C" int64_t b200fe_host_staging_bytes_ragged(const b200fe_params* p, int64_t chunk_rows, int64_t T,
                                                    int32_t sample_bytes, int32_t n_streams) {
  return host_staging_bytes(p, chunk_rows, T, n_streams, sample_bytes, true);
}

extern "C" int32_t b200fe_features_forward_host(const float* wave_host, int64_t R, int64_t T, const b200fe_params* p,
                                                const void* tables, float* out_host, void* staging,
                                                size_t staging_bytes, int64_t chunk_rows, void* const* streams,
                                                int32_t n_streams) {
  return forward_host(dense_input(wave_host, 4), R, T, p, tables, out_host, staging, staging_bytes, chunk_rows, streams,
                      n_streams);
}

extern "C" int32_t b200fe_features_forward_host_i16(const int16_t* pcm_host, int64_t R, int64_t T, const b200fe_params* p,
                                                    const void* tables, float* out_host, void* staging,
                                                    size_t staging_bytes, int64_t chunk_rows, void* const* streams,
                                                    int32_t n_streams) {
  return forward_host(dense_input(pcm_host, 2), R, T, p, tables, out_host, staging, staging_bytes, chunk_rows, streams,
                      n_streams);
}

extern "C" int32_t b200fe_features_forward_host_ragged(const void* clips_host, int32_t sample_bytes, int64_t n_samples,
                                                       const int64_t* offsets_host, const int32_t* lengths_host,
                                                       int64_t R, int64_t T, const b200fe_params* p, const void* tables,
                                                       float* out_host, void* staging, size_t staging_bytes,
                                                       int64_t chunk_rows, void* const* streams, int32_t n_streams) {
  g_launches = 0;
  if (!offsets_host || !lengths_host) { fe_set_error("offsets / lengths is NULL"); return B200FE_ERR_BAD_ARG; }
  if (n_samples < 1) { fe_set_error("n_samples=%lld must be >= 1", (long long)n_samples); return B200FE_ERR_BAD_ARG; }
  const host_input in{clips_host, sample_bytes, offsets_host, lengths_host, n_samples};
  return forward_host(in, R, T, p, tables, out_host, staging, staging_bytes, chunk_rows, streams, n_streams);
}
