// Launch interface of the CUDA-core kernels (fe_kernels.cu); the tcgen05 streaming kernel (fe_stream.cu) is declared in fe_gemm.h.
#ifndef FE_KERNELS_H_
#define FE_KERNELS_H_
#include <cuda_runtime.h>
#include "fe_common.h"

struct fe_fft_args {
  const float* wave;        // dense [R][T] or flat ragged clips
  const float* wave_chunk;  // dense rows of THIS launch ([rows][T], first row = row_base) when the input was staged by
                            // fe_launch_dense_rows; NULL: rows are read from `wave`
  const int64_t* offsets;   // ragged: start of each row's clip (floats), else NULL
  const int32_t* lengths;   // ragged: clip lengths, else NULL
  // streaming kernel, ragged input read partly in place (in_place != 0): `wave` is then the lower of the two buffers,
  // the flat clip buffer starts flat_rel floats above it and the staged rows of this launch dense_rel floats above it
  int64_t flat_rel, dense_rel;
  int32_t in_place;
  const void* tables;       // device blob
  float* out;               // MODE 0: [rows][n_freq][n_frames]; MODE 1: energies [rows_in_launch][n_filter][n_frames]
  unsigned int* group_max;  // per top_db group maximum energy (float bits), NULL when not needed
  int64_t T;
  int64_t row_base;         // absolute index of the launch's first row
  int64_t n_blocks;         // fe_rfft_kernel: (row, tile) work items of the launch (set by fe_launch_fft)
  int32_t n_fft, hop, n_frames, n_filter;
  int32_t ft;               // frames per CTA
  int32_t tiles_per_row;
  int32_t radix2_first;     // log2(n_fft/2) odd
  int32_t fft_warps;        // warps that own FFT buffers (set by fe_launch_fft)
  int32_t top_db_group;
  float preemph;
  int32_t pad_zero;         // ragged clips read through fe_stage_load: 1 = zero-pad short clips, 0 = repeat-pad
};

struct fe_tail_args {
  const float* energies;    // [rows_in_launch][n_filter][n_frames]
  const unsigned int* group_max;
  const void* tables;
  float* out;               // [R][n_out][n_frames] (absolute rows)
  int64_t row_base;
  int32_t n_frames, n_filter, n_coef, n_out;
  int32_t log_mode, deltas, delta_win, top_db_group;
  int32_t tt, halo;         // frames per CTA, halo frames each side (= deltas * (delta_win-1)/2)
  int32_t force_generic;    // tests: 1 = fe_tail_kernel everywhere, 2 = fe_tail_fast_kernel where fe_tail_quad_kernel applies
  float top_db;
};

// Per-device facts, cached per device ordinal (a process may drive several GPUs; lock-free, idempotent fills).
constexpr int kFeMaxDevices = 64;
int fe_current_device(void);        // cudaGetDevice, -1 on error
int fe_device_sms(int dev);         // multiprocessor count of `dev`
// Opts kernel `fn` in to `bytes` of dynamic shared memory on the current device.  Process-wide and thread-safe: the
// attribute is never set below the largest size granted so far for (fn, device); an already granted size costs one
// uncontended lock and no CUDA call.
cudaError_t fe_ensure_smem(const void* fn, size_t bytes);

// Kernels launched by this thread since the entry point that was called last reset it (b200fe_last_launch_count).
extern thread_local int64_t fe_launch_count;

// After a <<<>>>: the launch's error, counted in fe_launch_count when there is none.
inline cudaError_t fe_launched(void) {
  const cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) ++fe_launch_count;
  return e;
}

// Rows [0, rows) in pieces of at most max_rows: launch(r0, nr) enqueues one kernel over rows [r0, r0 + nr), or returns
// the error that kept it from doing so.  Stops at the first error.
template <typename F>
cudaError_t fe_launch_rows(int64_t rows, int64_t max_rows, F&& launch) {
  for (int64_t r0 = 0; r0 < rows; r0 += max_rows) {
    cudaError_t e = launch(r0, rows - r0 < max_rows ? rows - r0 : max_rows);
    if (e == cudaSuccess) e = fe_launched();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

// A ragged clip the streaming kernel can read where it lies: pad() only truncates it (len >= T), and its first sample
// is 16-byte aligned relative to the tensor map's base and within the map's reach (32 steps of 32 GB above the base).
// fe_dense_rows_kernel skips exactly these rows; fe_stream_kernel reads exactly these rows from the flat buffer.
constexpr int64_t kFeInPlaceReach = ((int64_t)31 << 31);   // 16-byte units: the 32nd 32 GB step is left as headroom
static __host__ __device__ inline bool fe_clip_in_place(int64_t off, int len, int64_t T, int64_t flat_rel) {
  return flat_rel >= 0 && len >= T && ((off | flat_rel) & 3) == 0 && ((flat_rel + off) >> 2) < kFeInPlaceReach;
}

size_t fe_fft_smem_bytes(int n_fft, int hop, int ft, int n_ch, int mode);
int fe_fft_pick_ft(int n_fft, int hop, int n_ch, int mode);   // frames per CTA, 0: does not fit shared memory
cudaError_t fe_launch_fft(const fe_fft_args& a, int mode, int64_t rows, cudaStream_t stream);
size_t fe_tail_smem_bytes(const fe_tail_args& a);
cudaError_t fe_launch_tail(const fe_tail_args& a, int64_t rows, cudaStream_t stream);
cudaError_t fe_launch_cmvn(float* out, int64_t n_series, int n_frames, cudaStream_t stream);
cudaError_t fe_launch_deltas(const float* in, float* out, int64_t rows, int64_t T, int win,
                             cudaStream_t stream);
// Dense [rows][T] copy of rows [row_base, row_base+rows): repeat-pad (pad_zero 0) or zero-pad (pad_zero 1) / truncate
// ragged clips and apply pre-emphasis, so the streaming kernel (TMA boxes over dense rows) serves those inputs too.
// dst 16-byte aligned.  Ragged row r reads its clip at wave + offsets[r] - base (`wave` may hold only a span of the
// flat buffer).
cudaError_t fe_launch_dense_rows(const float* wave, const int64_t* offsets, const int32_t* lengths,
                                 int64_t row_base, int64_t rows, int64_t T, float preemph, float* dst,
                                 cudaStream_t stream, int64_t flat_rel = -1, int64_t base = 0, int pad_zero = 0);
// The same from 16-bit PCM (x / 32768, exact); every row is written (no clip is read in place).
cudaError_t fe_launch_dense_rows(const int16_t* wave, const int64_t* offsets, const int32_t* lengths,
                                 int64_t row_base, int64_t rows, int64_t T, float preemph, float* dst,
                                 cudaStream_t stream, int64_t base = 0, int pad_zero = 0);
#endif
