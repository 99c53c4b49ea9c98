// CUDA-core kernels of the spectral front-end (sm_100a):
//   fe_fft_kernel    staging (reflect / repeat-pad / pre-emphasis) -> framing+window -> real FFT ->
//                    power -> [filterbank] -> tile store (+ per-group maximum for top_db)
//   fe_tail_kernel   log / dB + top_db clamp -> DCT-II -> delta / delta-delta -> one coalesced store
//   fe_cmvn_kernel   optional per-utterance mean / variance normalisation
//   fe_deltas_kernel stand-alone ComputeDeltas
#include <cuda_runtime.h>
#include <math.h>
#include <stdlib.h>
#include <atomic>
#include <map>
#include <mutex>
#include <utility>

#include "fe_fft.cuh"
#include "fe_tail.cuh"
#include "fe_kernels.h"

namespace {

constexpr int kFftWarps = 8;
constexpr int kFftThreads = kFftWarps * 32;

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}


// ------------------------------------------------------------------------------------------------
// Register-resident warp FFT (the fast path of fe_fft_kernel for n_fft = 64*E, E in {4, 8, 16}).
// One warp = one frame; the n_fft/2-point complex transform of the packed sequence is factored as
// N = E x 32 with n = lane + 32*j:  (1) an E-point DFT over j in each lane's registers,  (2) the twiddle
// W_N^(lane*k2),  (3) a 32-point DFT over the lanes (fe_warp_rfft_power).  All DFTs are radix-2
// decimation-in-frequency with compile-time twiddles where the index is a register number.
// ------------------------------------------------------------------------------------------------
__host__ __device__ constexpr float fe_cos16(int k) {  // cos(2*pi*k/16)
  constexpr float c1 = 0.92387953251128674f, c2 = 0.70710678118654752f, c3 = 0.38268343236508977f;
  switch (k & 15) {
    case 0: return 1.0f;
    case 1: case 15: return c1;
    case 2: case 14: return c2;
    case 3: case 13: return c3;
    case 4: case 12: return 0.0f;
    case 5: case 11: return -c3;
    case 6: case 10: return -c2;
    case 7: case 9: return -c1;
    default: return -1.0f;
  }
}
__host__ __device__ constexpr float fe_sin16(int k) { return fe_cos16(k + 12); }  // sin(x) = cos(x - pi/2)
__host__ __device__ constexpr int fe_ilog2(int e) { return e <= 1 ? 0 : 1 + fe_ilog2(e >> 1); }
__host__ __device__ constexpr int fe_bitrev(int i, int bits) {
  int r = 0;
  for (int b = 0; b < bits; ++b) r = (r << 1) | ((i >> b) & 1);
  return r;
}

template <int E>
__device__ __forceinline__ void fe_regs_dft(float2 (&v)[E]) {
#pragma unroll
  for (int half = E / 2; half >= 1; half >>= 1) {
#pragma unroll
    for (int base = 0; base < E; base += 2 * half) {
#pragma unroll
      for (int i = 0; i < half; ++i) {
        const float2 a = v[base + i], b = v[base + i + half];
        v[base + i] = make_float2(a.x + b.x, a.y + b.y);
        const float dx = a.x - b.x, dy = a.y - b.y;
        const int k16 = i * (8 / half);  // W_(2*half)^i = exp(-2*pi*i*k16/16)
        if (k16 == 0) {
          v[base + i + half] = make_float2(dx, dy);
        } else if (k16 == 4) {
          v[base + i + half] = make_float2(dy, -dx);
        } else {
          const float c = fe_cos16(k16), sn = fe_sin16(k16);
          v[base + i + half] = make_float2(fmaf(dy, sn, dx * c), fmaf(-dx, sn, dy * c));
        }
      }
    }
  }
}

// The lane-dimension DFT is done mostly in registers again ("transposed" form): after the E-point
// DFT over j and the twiddle, the warp transposes through its shared buffer (A[k2*33 + n1], conflict-free both
// ways) so that lane (k2, h) holds n1 = r + E*h, r = 0..E-1, of column k2.  The 32-point DFT over n1 is then
// log2(32/E) butterfly-exchange stages over the bits of h (twiddles W_32^x from a 16-entry shared table; lanes on
// the "sum" side read W^0 = 1) followed by a second E-point register DFT.  Register i of lane (k2, h) ends up with
// Z[E*(bitrev(h) + (32/E)*bitrevE(i)) + k2], which for every i is a permutation of 32 consecutive Z indices over
// the lanes: Z is stored in natural order.  (A first version ran all five stages of the 32-point DFT as lane
// exchanges: 0.845 ms per 1184 mel utterances against 0.760 ms for this form.)
template <int E>
__device__ __forceinline__ void fe_warp_rfft_power(int lane, const float* __restrict__ frame,
                                                     const float* __restrict__ s_win, const float2 (&tw2)[E],
                                                     const float2* __restrict__ s_w32,
                                                     const fe_c2* __restrict__ s_rtw, float2* zbuf, float* pw,
                                                     int pw_stride) {
  constexpr int NH = 32 * E, L = fe_ilog2(E), S = 5 - L;
  float2 v[E];
  const float2* f2 = reinterpret_cast<const float2*>(frame);
  const float2* w2 = reinterpret_cast<const float2*>(s_win);
#pragma unroll
  for (int j = 0; j < E; ++j) {
    const float2 x = f2[lane + 32 * j], w = w2[lane + 32 * j];
    v[j] = make_float2(x.x * w.x, x.y * w.y);
  }
  fe_regs_dft<E>(v);
  zbuf[lane] = v[0];                                   // k2 = 0: twiddle 1
#pragma unroll
  for (int i = 1; i < E; ++i) {
    const float2 t = tw2[i], a = v[i];
    zbuf[fe_bitrev(i, L) * 33 + lane] = make_float2(fmaf(-a.y, t.y, a.x * t.x), fmaf(a.x, t.y, a.y * t.x));
  }
  __syncwarp();
  const int k2 = lane & (E - 1), h = lane >> L;
  {
    const float2* col = zbuf + k2 * 33 + E * h;
#pragma unroll
    for (int r = 0; r < E; ++r) v[r] = col[r];
  }
#pragma unroll
  for (int s = 0; s < S; ++s) {
    const int H = 16 >> s, c = 16 / H;
    const bool lower = (lane & H) != 0;
    const float sgn = lower ? -1.0f : 1.0f;
    const int hl = (lane & (H - 1)) & ~(E - 1);
    const float2* tw = s_w32 + (lower ? hl * c : 0);
    const int step = lower ? c : 0;
#pragma unroll
    for (int r = 0; r < E; ++r) {
      const float px = __shfl_xor_sync(0xffffffffu, v[r].x, H);
      const float py = __shfl_xor_sync(0xffffffffu, v[r].y, H);
      const float tx = fmaf(sgn, v[r].x, px), ty = fmaf(sgn, v[r].y, py);   // upper: v + p, lower: p - v
      const float2 t = tw[r * step];
      v[r] = make_float2(fmaf(-ty, t.y, tx * t.x), fmaf(tx, t.y, ty * t.x));
    }
  }
  fe_regs_dft<E>(v);
  __syncwarp();                                          // every lane has read its column before Z overwrites it
  static_assert(S >= 1, "E <= 16");
  const int kb = E * (int)(__brev((unsigned)h) >> (32 - S)) + k2;   // E * bitrev_S(h) + k2
#pragma unroll
  for (int i = 0; i < E; ++i) zbuf[kb + 32 * fe_bitrev(i, L)] = v[i];
  __syncwarp();
#pragma unroll
  for (int i = 0; i <= NH / 64; ++i) {
    const int k = lane + 32 * i;
    if (i == NH / 64 && lane != 0) break;
    const float2 a = zbuf[k];
    const float2 b = zbuf[(NH - k) & (NH - 1)];
    const float ex = a.x + b.x, ey = a.y - b.y;   // 2*Fe
    const float ox = a.y + b.y, oy = b.x - a.x;   // 2*Fo
    const fe_c2 r = s_rtw[k];
    const float tx = r.x * ox - r.y * oy, ty = r.x * oy + r.y * ox;
    const float px = ex + tx, py = ey + ty, mx = ex - tx, my = ey - ty;
    pw[k * pw_stride] = px * px + py * py;                 // s_win carries the factor 1/2: no 1/4 here
    pw[(NH - k) * pw_stride] = mx * mx + my * my;
  }
}

// ------------------------------------------------------------------------------------------------
// fe_fft_kernel
//   grid.x = rows * tiles_per_row ; one CTA = `ft` consecutive frames of one row
//   MODE 0: write the power spectrum  out[row][k][t]
//   MODE 1: write filterbank energies ws[row_local][f][t] and atomicMax the group maximum
// ------------------------------------------------------------------------------------------------
template <int MODE>
__global__ void __launch_bounds__(kFftThreads) fe_fft_kernel(fe_fft_args a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n_fft = a.n_fft, nh = n_fft >> 1, n_freq = nh + 1, hop = a.hop;
  const int ft = a.ft;
  const int seg = (ft - 1) * hop + n_fft;  // staged samples

  // carve shared memory
  float* s_stage = reinterpret_cast<float*>(smem_raw);
  size_t off = ((size_t)seg * 4 + 15) & ~(size_t)15;
  float* s_win = reinterpret_cast<float*>(smem_raw + off);
  off += (size_t)n_fft * 4;
  fe_c2* s_tw = reinterpret_cast<fe_c2*>(smem_raw + off);
  off += (size_t)nh * 8;
  fe_c2* s_rtw = reinterpret_cast<fe_c2*>(smem_raw + off);
  off += (((size_t)(nh / 2 + 1) * 8) + 15) & ~(size_t)15;
  fe_c2* s_buf = reinterpret_cast<fe_c2*>(smem_raw + off);  // [fft_warps][2][nh+1]
  off += (size_t)a.fft_warps * 2 * (nh + 1) * 8;
  float* s_tile = reinterpret_cast<float*>(smem_raw + off);  // MODE0: [n_freq][ft+1]; MODE1: [n_filter][ft+1]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t row_local = blockIdx.x / a.tiles_per_row;
  const int tile = blockIdx.x - (int)(row_local * a.tiles_per_row);
  const int64_t row = a.row_base + row_local;
  const int t0 = tile * ft;
  const int nf_here = min(ft, a.n_frames - t0);

  const unsigned char* blob = reinterpret_cast<const unsigned char*>(a.tables);
  const fe_blob_header* h = reinterpret_cast<const fe_blob_header*>(blob);

  // ---- constants -> shared --------------------------------------------------------------------
  {
    const float* gw = reinterpret_cast<const float*>(blob + h->off_window);
    for (int i = tid; i < n_fft; i += kFftThreads) s_win[i] = gw[i];
    const fe_c2* gt = reinterpret_cast<const fe_c2*>(blob + h->off_twiddle);
    for (int i = tid; i < nh; i += kFftThreads) s_tw[i] = gt[i];
    const fe_c2* gr = reinterpret_cast<const fe_c2*>(blob + h->off_rtwiddle);
    for (int i = tid; i <= nh / 2; i += kFftThreads) s_rtw[i] = gr[i];
  }

  // ---- stage the waveform segment -------------------------------------------------------------
  // Padded position pp = t0*hop + i  (reflect padding by n_fft/2, torch.stft center=True); the
  // T-sample signal itself is the clip repeat-padded (pad(), maze5.py:280-285) or zero-padded (a.pad_zero) /
  // truncated to T.
  {
    const float* src;
    int clip_len;  // T < 2^31 is checked on the host
    if (a.offsets) {
      src = a.wave + a.offsets[row];
      clip_len = a.lengths[row];
    } else {
      src = a.wave_chunk ? a.wave_chunk + row_local * a.T : a.wave + row * a.T;
      clip_len = (int)a.T;
    }
    const int seg_here = (nf_here - 1) * hop + n_fft;
    fe_stage_load(tid, kFftThreads, src, clip_len, (int)a.T, n_fft, t0 * hop, seg_here, a.preemph, s_stage, a.pad_zero);
  }
  __syncthreads();

  // ---- per-warp FFTs --------------------------------------------------------------------------
  fe_c2* buf0 = s_buf + (size_t)warp * 2 * (nh + 1);
  fe_c2* buf1 = buf0 + (nh + 1);
  const int tile_stride = ft + 1;
  const int32_t* bstart = reinterpret_cast<const int32_t*>(blob + h->off_band_start);
  const int32_t* blen = reinterpret_cast<const int32_t*>(blob + h->off_band_len);
  const int32_t* bwoff = reinterpret_cast<const int32_t*>(blob + h->off_band_woff);
  const float* bw = reinterpret_cast<const float*>(blob + h->off_band_w);

  // only the first fft_warps warps own FFT buffers (all 8 unless n_fft is too large for shared memory)
  for (int fl = warp; fl < nf_here && warp < a.fft_warps; fl += a.fft_warps) {
    const float* frame = s_stage + (size_t)fl * hop;
    fe_c2* in = buf0;
    fe_c2* out = buf1;
    fe_fft_stage_first(lane, frame, s_win, out, nh, a.radix2_first != 0);
    __syncwarp();
    int ns = a.radix2_first ? 2 : 4;
    while (ns < nh) {
      fe_c2* t = in; in = out; out = t;
      fe_fft_stage4(lane, in, out, s_tw, nh, ns);
      __syncwarp();
      ns <<= 2;
    }
    // `out` holds Z; write the power into the other buffer (nh+1 floats fit in nh+1 complex slots)
    float* pw = reinterpret_cast<float*>(in);
    fe_fft_power(lane, out, s_rtw, pw, nh);
    __syncwarp();
    if (MODE == 0) {
      for (int k = lane; k < n_freq; k += 32) s_tile[(size_t)k * tile_stride + fl] = pw[k];
    } else {
      fe_fbank_apply(lane, pw, bstart, blen, bwoff, bw, a.n_filter, s_tile + fl, tile_stride);
    }
    __syncwarp();
  }
  __syncthreads();

  // ---- coalesced tile store -------------------------------------------------------------------
  const int n_ch = (MODE == 0) ? n_freq : a.n_filter;
  float* dst = a.out + ((size_t)row_local * n_ch) * a.n_frames + t0;
  float vmax = 0.0f;
  // thread -> (channel, frame) with frame fastest so that consecutive lanes write consecutive t
  const int per_ch = nf_here;
  const int total = n_ch * per_ch;
  for (int i = tid; i < total; i += kFftThreads) {
    const int c = i / per_ch, t = i - c * per_ch;
    const float v = s_tile[(size_t)c * tile_stride + t];
    dst[(size_t)c * a.n_frames + t] = v;
    vmax = fmaxf(vmax, v);
  }
  if (MODE == 1 && a.group_max) {
    vmax = warp_max(vmax);
    __shared__ float s_red[kFftWarps];
    if (lane == 0) s_red[warp] = vmax;
    __syncthreads();
    if (tid == 0) {
      float m = s_red[0];
#pragma unroll
      for (int w = 1; w < kFftWarps; ++w) m = fmaxf(m, s_red[w]);
      // energies are >= 0, so the unsigned ordering of the bit patterns is the float ordering
      atomicMax(a.group_max + row / a.top_db_group, __float_as_uint(m));
    }
  }
}

// ------------------------------------------------------------------------------------------------
// fe_rfft_kernel : the FFT variant's fast path (n_fft = 64*E, even hop).  Same grid, arguments and results
// as fe_fft_kernel; differences: register-resident warp FFT, powers of the CTA's frames collected in one
// transposed [bin][frame] tile, and the filterbank applied by the whole CTA afterwards with
// lane = frame (every warp walks a band of warp-uniform length: no imbalance between narrow and wide filters).
//   FT = frames per CTA (16 or 32): a warp covers 32/FT filters x FT frames per step of the filterbank phase.
// ------------------------------------------------------------------------------------------------
template <int E>
__host__ __device__ constexpr int fe_rfft_zunits() { return 33 * E; }   // transpose buffer A[k2*33 + n1]; Z (32*E) reuses it

// Filterbank phase of fe_rfft_kernel for FT frames per CTA (stride FT + 1 is a compile-time constant: the band
// loop's shared-memory loads take immediate offsets).  lane -> (filter slot sub, frame tl); weights in shared memory.
template <int FT>
__device__ __forceinline__ void fe_rfft_fbank(int warp, int lane, int n_filter, const int4* __restrict__ s_band,
                                              const float* __restrict__ s_bw, const float* __restrict__ s_pw,
                                              float* __restrict__ s_tile) {
  constexpr int ST = FT + 1, FPW = 32 / FT;
  const int tl = lane & (FT - 1), sub = lane / FT;
  for (int f = warp * FPW + sub; f < n_filter; f += kFftWarps * FPW) {
    const int4 band = s_band[f];
    const int len = band.y;
    const float* pcol = s_pw + band.x * ST + tl;
    const float* w = s_bw + band.z;
    float acc = 0.0f;                                               // same summation order as fe_fbank_apply
    int i = 0;
#pragma unroll 1
    for (; i + 4 <= len; i += 4, pcol += 4 * ST, w += 4) {
      const float p0 = pcol[0], p1 = pcol[ST], p2 = pcol[2 * ST], p3 = pcol[3 * ST];
      const float w0 = w[0], w1 = w[1], w2 = w[2], w3 = w[3];
      acc = fmaf(p0, w0, acc);
      acc = fmaf(p1, w1, acc);
      acc = fmaf(p2, w2, acc);
      acc = fmaf(p3, w3, acc);
    }
    const int rem = len - i;                                        // 0..3, all loads before the FMAs
    const float p0 = rem > 0 ? pcol[0] : 0.0f, p1 = rem > 1 ? pcol[ST] : 0.0f, p2 = rem > 2 ? pcol[2 * ST] : 0.0f;
    const float w0 = rem > 0 ? w[0] : 0.0f, w1 = rem > 1 ? w[1] : 0.0f, w2 = rem > 2 ? w[2] : 0.0f;
    if (rem > 0) acc = fmaf(p0, w0, acc);
    if (rem > 1) acc = fmaf(p1, w1, acc);
    if (rem > 2) acc = fmaf(p2, w2, acc);
    s_tile[f * ST + tl] = acc;
  }
}

template <int MODE, int E>
__global__ void __launch_bounds__(kFftThreads, E == 16 ? 2 : 4) fe_rfft_kernel(fe_fft_args a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int NH = 32 * E, NFFT = 2 * NH, NFREQ = NH + 1;
  const int hop = a.hop, ft = a.ft, stride = ft + 1;
  const int seg = (ft - 1) * hop + NFFT;

  float* s_stage = reinterpret_cast<float*>(smem_raw);
  size_t off = ((size_t)seg * 4 + 15) & ~(size_t)15;
  float* s_win = reinterpret_cast<float*>(smem_raw + off);
  off += (size_t)NFFT * 4;
  fe_c2* s_rtw = reinterpret_cast<fe_c2*>(smem_raw + off);
  off += (((size_t)(NH / 2 + 1) * 8) + 15) & ~(size_t)15;
  float2* s_z = reinterpret_cast<float2*>(smem_raw + off);   // [warps][zunits]
  off += (size_t)kFftWarps * fe_rfft_zunits<E>() * 8;
  float* s_pw = reinterpret_cast<float*>(smem_raw + off);    // [NFREQ][ft+1]
  off += (((size_t)NFREQ * stride * 4) + 15) & ~(size_t)15;
  float* s_tile = reinterpret_cast<float*>(smem_raw + off);  // MODE 1: [n_filter][ft+1]
  off += (MODE == 1) ? ((((size_t)a.n_filter * stride * 4) + 15) & ~(size_t)15) : 0;
  float* s_bw = reinterpret_cast<float*>(smem_raw + off);    // MODE 1: band weights
  off += (MODE == 1) ? (size_t)(2 * NFREQ + 2 * a.n_filter) * 4 : 0;
  int4* s_band = reinterpret_cast<int4*>(smem_raw + ((off + 15) & ~(size_t)15));   // MODE 1: {start, len, weight offset}

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  const unsigned char* blob = reinterpret_cast<const unsigned char*>(a.tables);
  const fe_blob_header* h = reinterpret_cast<const fe_blob_header*>(blob);
  const fe_c2* gt = reinterpret_cast<const fe_c2*>(blob + h->off_twiddle);

  // ---- constants -> shared, frame-independent twiddles -> registers ------------------------------
  {
    const float4* gw = reinterpret_cast<const float4*>(blob + h->off_window);
    // the window is stored halved: Z comes out halved and the split's 1/4 on |X|^2 disappears (exact: power of two)
    for (int i = tid; i < NFFT / 4; i += kFftThreads) {
      const float4 w = gw[i];
      reinterpret_cast<float4*>(s_win)[i] = make_float4(0.5f * w.x, 0.5f * w.y, 0.5f * w.z, 0.5f * w.w);
    }
    const fe_c2* gr = reinterpret_cast<const fe_c2*>(blob + h->off_rtwiddle);
    for (int i = tid; i <= NH / 2; i += kFftThreads) s_rtw[i] = gr[i];
  }
  const float* gbw = reinterpret_cast<const float*>(blob + h->off_band_w);
  const bool bw_shared = MODE == 1 && h->total_w <= 2 * NFREQ + 2 * a.n_filter;   // fe_rfft_bw_cap
  if (bw_shared)
    for (int i = tid; i < h->total_w; i += kFftThreads) s_bw[i] = gbw[i];
  if (MODE == 1) {
    const int32_t* bstart = reinterpret_cast<const int32_t*>(blob + h->off_band_start);
    const int32_t* blen = reinterpret_cast<const int32_t*>(blob + h->off_band_len);
    const int32_t* bwoff = reinterpret_cast<const int32_t*>(blob + h->off_band_woff);
    for (int f = tid; f < a.n_filter; f += kFftThreads) s_band[f] = make_int4(bstart[f], blen[f], bwoff[f], 0);
  }
  float2 tw2[E];
#pragma unroll
  for (int i = 0; i < E; ++i) {
    const fe_c2 t = gt[lane * fe_bitrev(i, fe_ilog2(E))];             // W_NH^(lane * k2)
    tw2[i] = make_float2(t.x, t.y);
  }

  float2* zbuf = s_z + (size_t)warp * fe_rfft_zunits<E>();
  const int tl = lane & (ft - 1), sub = lane / ft, fpw = 32 / ft;     // ft is 16 or 32
  __shared__ float s_red[kFftWarps];
  __shared__ float2 s_w32[16];                                         // W_32^j, j < 16 (transposed warp FFT)
  if (tid < 16) {
    const fe_c2 t = gt[tid * E];
    s_w32[tid] = make_float2(t.x, t.y);
  }

  // Staging of work item `b` into s_stage.  Interior tiles of plain dense rows (no reflection, no repeat, no
  // pre-emphasis, 16-byte aligned) are 128-bit copies, asynchronous (cp.async) on request; everything else goes
  // through fe_stage_load.  Returns true when the copy was issued (or done); async_only: false = nothing was done.
  auto stage_tile = [&](int64_t b, bool async_only) -> bool {
    const int64_t rl = b / a.tiles_per_row;
    const int tile_b = (int)(b - rl * a.tiles_per_row);
    const int64_t row_b = a.row_base + rl;
    const int t0_b = tile_b * ft;
    const int nf_b = min(ft, a.n_frames - t0_b);
    const float* src;
    int clip_len;
    if (a.offsets) {
      src = a.wave + a.offsets[row_b];
      clip_len = a.lengths[row_b];
    } else {
      src = a.wave_chunk ? a.wave_chunk + rl * a.T : a.wave + row_b * a.T;
      clip_len = (int)a.T;
    }
    const int seg_here = (nf_b - 1) * hop + NFFT;
    const int r0 = t0_b * hop - NH;
    const float* p0 = src + r0;
    if (r0 >= 0 && r0 + seg_here <= (int)a.T && clip_len >= (int)a.T && a.preemph == 0.0f &&
        (reinterpret_cast<uintptr_t>(p0) & 15) == 0 && (seg_here & 3) == 0) {
      const uint32_t dst = (uint32_t)__cvta_generic_to_shared(s_stage);
      for (int i = tid; i < seg_here / 4; i += kFftThreads)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * (uint32_t)i), "l"(p0 + 4 * i) : "memory");
      return true;
    }
    if (async_only) return false;
    fe_stage_load(tid, kFftThreads, src, clip_len, (int)a.T, NFFT, t0_b * hop, seg_here, a.preemph, s_stage,
                  a.pad_zero);
    return true;
  };
  bool prefetched = false;

  // ---- persistent CTA: tiles blockIdx.x, blockIdx.x + gridDim.x, ... (constants above are loaded once) ----
  for (int64_t blk = blockIdx.x; blk < a.n_blocks; blk += gridDim.x) {
  const int64_t row_local = blk / a.tiles_per_row;
  const int tile = (int)(blk - row_local * a.tiles_per_row);
  const int64_t row = a.row_base + row_local;
  const int t0 = tile * ft;
  const int nf_here = min(ft, a.n_frames - t0);

  // ---- the waveform segment: staged here unless the previous iteration prefetched it (cp.async) ------
  if (!prefetched) stage_tile(blk, false);
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncthreads();

  // ---- one warp = one frame: FFT in registers, powers into the [bin][frame] tile -------------------
  for (int fl = warp; fl < nf_here; fl += kFftWarps) {
    fe_warp_rfft_power<E>(lane, s_stage + (size_t)fl * hop, s_win, tw2, s_w32, s_rtw, zbuf, s_pw + fl, stride);
    __syncwarp();
  }
  __syncthreads();
  // the staging buffer is free: fetch the next work item's samples behind the filterbank and store phases
  prefetched = (blk + gridDim.x < a.n_blocks) && stage_tile(blk + gridDim.x, true);

  // ---- filterbank: lane -> (filter slot, frame); the band loop has the same length for a whole warp step ----
  const float* tile_src = s_pw;
  int n_ch = NFREQ;
  if (MODE == 1) {
    if (bw_shared) {
      if (ft == 16) fe_rfft_fbank<16>(warp, lane, a.n_filter, s_band, s_bw, s_pw, s_tile);
      else fe_rfft_fbank<32>(warp, lane, a.n_filter, s_band, s_bw, s_pw, s_tile);
    } else {   // a bank denser than any triangular one: weights stay in global memory
      for (int f = warp * fpw + sub; f < a.n_filter; f += kFftWarps * fpw) {
        const int4 band = s_band[f];
        const float* pcol = s_pw + band.x * stride + tl;
        const float* w = gbw + band.z;
        float acc = 0.0f;
        for (int i = 0; i < band.y; ++i) acc = fmaf(pcol[i * stride], __ldg(w + i), acc);
        s_tile[f * stride + tl] = acc;
      }
    }
    __syncthreads();
    tile_src = s_tile;
    n_ch = a.n_filter;
  }

  // ---- coalesced tile store (+ group maximum) --------------------------------------------------
  float* dst = a.out + ((size_t)row_local * n_ch) * a.n_frames + t0;
  float vmax = 0.0f;
  if (tl < nf_here) {
    for (int c = warp * fpw + sub; c < n_ch; c += kFftWarps * fpw) {
      const float v = tile_src[(size_t)c * stride + tl];
      dst[(size_t)c * a.n_frames + tl] = v;
      vmax = fmaxf(vmax, v);
    }
  }
  if (MODE == 1 && a.group_max) {
    vmax = warp_max(vmax);
    if (lane == 0) s_red[warp] = vmax;
    __syncthreads();
    if (tid == 0) {
      float m = s_red[0];
#pragma unroll
      for (int w = 1; w < kFftWarps; ++w) m = fmaxf(m, s_red[w]);
      atomicMax(a.group_max + row / a.top_db_group, __float_as_uint(m));
    }
  }
  __syncthreads();   // the next tile reuses the staging buffer, the tiles and s_red
  }
}

// ------------------------------------------------------------------------------------------------
// fe_tail_kernel : grid (tiles, rows_in_chunk), block kTailThreads
// ------------------------------------------------------------------------------------------------
constexpr int kTailThreads = 128;

__global__ void __launch_bounds__(kTailThreads) fe_tail_kernel(fe_tail_args a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tt = a.tt, halo = a.halo, w = tt + 2 * halo;
  const int nfil = a.n_filter, ncoef = a.n_coef;
  const int nc = ncoef > 0 ? ncoef : nfil;  // channels per block of the output
  float* s_e = reinterpret_cast<float*>(smem_raw);  // [nfil][w]   (log) energies
  float* s_c = s_e + (size_t)nfil * w;              // [nc][w]     coefficients (aliases s_e when no DCT)
  if (ncoef == 0) s_c = s_e;
  float* s_d = s_c + (size_t)nc * w;                // [nc][w]     deltas
  float* s_dct = s_d + (a.deltas > 0 ? (size_t)nc * w : 0);  // [nfil][ncoef]

  const int tid = threadIdx.x;
  const int64_t row_local = blockIdx.y;
  const int64_t row = a.row_base + row_local;
  const int t0 = blockIdx.x * tt;
  const int nF = a.n_frames;
  const int tv0 = t0 - halo;  // virtual frame index of tile position 0

  const unsigned char* blob = reinterpret_cast<const unsigned char*>(a.tables);
  const fe_blob_header* h = reinterpret_cast<const fe_blob_header*>(blob);
  if (ncoef > 0) {
    const float* gd = reinterpret_cast<const float*>(blob + h->off_dct);
    for (int i = tid; i < nfil * ncoef; i += kTailThreads) s_dct[i] = gd[i];
  }

  float floor_db = -INFINITY;
  if (a.log_mode == B200FE_LOG_DB && a.top_db >= 0.0f) {
    const float gmax = __uint_as_float(a.group_max[row / a.top_db_group]);
    floor_db = 10.0f * log10f(fmaxf(gmax, 1e-10f)) - a.top_db;
  }
  const float* src = a.energies + (size_t)row_local * nfil * nF;
  fe_tail_load(tid, kTailThreads, src, nfil, nF, w, tv0, a.log_mode, floor_db, s_e);
  __syncthreads();
  if (ncoef > 0) {
    fe_tail_dct(tid, kTailThreads, s_e, s_dct, nfil, ncoef, w, s_c);
    __syncthreads();
  }
  const int n = (a.delta_win - 1) / 2;
  float* out_row = a.out + (size_t)row * a.n_out * nF;
  const int nt_here = min(tt, nF - t0);
  if (a.deltas >= 1) {
    fe_tail_delta(tid, kTailThreads, s_c, nc, w, n, tv0, nF, s_d);
    __syncthreads();
  }
  fe_tail_store(tid, kTailThreads, s_c, s_d, nc, w, n, halo, t0, nt_here, nF, a.deltas, out_row);
}

// ------------------------------------------------------------------------------------------------
// fe_tail_fast_kernel : the arithmetic of fe_tail_kernel for n_filter, n_coef <= 32 with everything that can be
// resolved at compile time resolved there: one thread per tile position, the frame's (log) energies and cepstral
// coefficients in registers (KQ = ceil(channels / 4) float4 groups), delta stencils of half-width N unrolled
// (N = 0: run-time loop), MUFU-based logarithms (absolute error ~1e-6 dB, far inside the 1e-4 feature tolerance).
// Only the delta stencils go through shared memory.  grid (tiles, rows), block = tt + 2*halo rounded up to a warp.
// ------------------------------------------------------------------------------------------------
constexpr int kFastMax = 32;

__device__ __forceinline__ float fast_log_energy(float v, int log_mode, float floor_db) {
  if (log_mode == B200FE_LOG_DB) {
    v = 3.0102999566398120f * __log2f(fmaxf(v, 1e-10f));   // 10 log10(x) = 10 log10(2) log2(x)
    v = fmaxf(v, floor_db);
  } else if (log_mode == B200FE_LOG_LN) {
    v = 0.6931471805599453f * __log2f(v + 1e-6f);
  }
  return v;
}

// sum_m m * c[m], m = -n .. n, around p
template <int N>
__device__ __forceinline__ float delta_taps(const float* p, int n) {
  if (N > 0) {
    float acc = p[1] - p[-1];
#pragma unroll
    for (int m = 2; m <= N; ++m) acc = fmaf((float)m, p[m] - p[-m], acc);
    return acc;
  }
  float acc = 0.0f;
  for (int m = 1; m <= n; ++m) acc = fmaf((float)m, p[m] - p[-m], acc);
  return acc;
}

template <int KQ, int N, bool EXACT>   // EXACT: the channel count is exactly 4*KQ (no per-channel bound checks)
__global__ void __launch_bounds__(256) fe_tail_fast_kernel(fe_tail_args a) {
  constexpr int kRegs = 4 * KQ;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tt = a.tt, halo = a.halo, w = tt + 2 * halo;
  const int nfil = a.n_filter, ncoef = a.n_coef;
  const int nc = EXACT ? kRegs : (ncoef > 0 ? ncoef : nfil);
  float* s_dct = reinterpret_cast<float*>(smem_raw);    // [nfil][4*KQ] (zero padded rows), read as float4: kept first so
                                                        // that it is 16-byte aligned whatever nc * w is (odd n_coef x odd w)
  float* s_c = s_dct + nfil * kRegs;                    // [nc][w]
  float* s_d = s_c + nc * w;                            // [nc][w]
  float* s_e = s_d + nc * w;                            // [nfil][w] energies, fetched asynchronously

  const int j = threadIdx.x;
  const int64_t row_local = blockIdx.y;
  const int64_t row = a.row_base + row_local;
  const int t0 = blockIdx.x * tt;
  const int nF = a.n_frames;
  const int tv0 = t0 - halo;
  const int tcl = fe_clampi(tv0 + j, 0, nF - 1) - tv0;   // tile position of this position's (clamped) frame
  // the frame's energies come from L2 (several hundred cycles): start all the fetches now (cp.async, no registers
  // held), behind the table and group-maximum loads below; each thread later reads only what it fetched itself
  if (j < w) {
    const float* src = a.energies + (size_t)row_local * nfil * nF + (tv0 + tcl);
    const uint32_t dst = (uint32_t)__cvta_generic_to_shared(s_e + j);
    for (int f = 0; f < nfil; ++f)
      asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + (uint32_t)(f * w) * 4u), "l"(src + (size_t)f * nF) : "memory");
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
  const unsigned char* blob = reinterpret_cast<const unsigned char*>(a.tables);
  const fe_blob_header* h = reinterpret_cast<const fe_blob_header*>(blob);
  if (ncoef > 0) {
    const float* gd = reinterpret_cast<const float*>(blob + h->off_dct);
    for (int i = j; i < nfil * kRegs; i += blockDim.x) {
      const int f = i / kRegs, k = i - f * kRegs;
      s_dct[i] = k < ncoef ? gd[f * ncoef + k] : 0.0f;
    }
  }
  float floor_db = -INFINITY;
  if (a.log_mode == B200FE_LOG_DB && a.top_db >= 0.0f) {
    const float gmax = __uint_as_float(a.group_max[row / a.top_db_group]);
    floor_db = 3.0102999566398120f * __log2f(fmaxf(gmax, 1e-10f)) - a.top_db;
  }
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncthreads();

  const bool owner = j >= halo && j < halo + tt && (t0 + j - halo) < nF;   // this thread stores frame t0 + j - halo
  float* out_p = a.out + (size_t)row * a.n_out * nF + (t0 + j - halo);    // walks down the channels
  float c[kRegs];
#pragma unroll
  for (int k = 0; k < kRegs; ++k) c[k] = 0.0f;
  if (j < w) {
    const float* ej = s_e + j;
    if (ncoef > 0) {
      const float4* dr = reinterpret_cast<const float4*>(s_dct);
#pragma unroll 4
      for (int f = 0; f < nfil; ++f, dr += KQ) {
        const float v = fast_log_energy(ej[f * w], a.log_mode, floor_db);
#pragma unroll
        for (int k4 = 0; k4 < KQ; ++k4) {
          const float4 d = dr[k4];
          c[4 * k4 + 0] = fmaf(v, d.x, c[4 * k4 + 0]);
          c[4 * k4 + 1] = fmaf(v, d.y, c[4 * k4 + 1]);
          c[4 * k4 + 2] = fmaf(v, d.z, c[4 * k4 + 2]);
          c[4 * k4 + 3] = fmaf(v, d.w, c[4 * k4 + 3]);
        }
      }
    } else {
      // no DCT: channel k is the (log) energy of filter k
#pragma unroll
      for (int k = 0; k < kRegs; ++k)
        if (EXACT || k < nc) c[k] = fast_log_energy(ej[k * w], a.log_mode, floor_db);
    }
    if (a.deltas >= 1) {
      float* sc = s_c + j;
#pragma unroll
      for (int k = 0; k < kRegs; ++k)
        if (EXACT || k < nc) sc[k * w] = c[k];
    }
  }
  if (owner) {
    float* o = out_p;
#pragma unroll
    for (int k = 0; k < kRegs; ++k, o += nF)
      if (EXACT || k < nc) *o = c[k];
  }
  if (a.deltas >= 1) {
    const int n = (a.delta_win - 1) / 2;
    const float inv_denom = 3.0f / (float)(n * (n + 1) * (2 * n + 1));
    __syncthreads();
    if (j >= n && j < w - n) {
      const float* cc = s_c + tcl;
      float* dd = s_d + j;
      float* o = out_p + (size_t)nc * nF;
#pragma unroll
      for (int k = 0; k < kRegs; ++k, cc += w, dd += w, o += nF) {
        if (EXACT || k < nc) {
          const float d = delta_taps<N>(cc, n) * inv_denom;
          *dd = d;
          if (owner) *o = d;
        }
      }
    }
    if (a.deltas >= 2) {
      __syncthreads();
      if (owner) {
        // delta of the delta at the clamped frame: s_d position tcl (interior: j itself)
        const float* dd = s_d + tcl;
        float* o = out_p + (size_t)2 * nc * nF;
#pragma unroll
        for (int k = 0; k < kRegs; ++k, dd += w, o += nF)
          if (EXACT || k < nc) *o = delta_taps<N>(dd, n) * inv_denom;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// fe_tail_quad_kernel : fe_tail_fast_kernel's arithmetic for the shape the LFCC front-end runs at (DCT present, channel
// count a multiple of 4, delta half-width 2 or no deltas, n_frames % 4 == 0) with the instruction count cut to what
// the feature write-out (three quarters of the step's HBM bytes) can hide:
//   phase 1  one thread per tile position: the frame's energies fetched with cp.async into the rows the deltas use
//            later (no staging buffer of their own: 5 CTAs per SM instead of 4), one MUFU per logarithm, the DCT against the table in shared memory (torchaudio's float32 table is not symmetric
//            under f -> n_filter-1-f to better than 4e-6, so folding the filter pairs would cost parity),
//            coefficients to shared memory;
//   phase 2/3  one thread per (channel, four consecutive positions): three 16-byte shared loads give the 8-wide
//            window of the two-tap-pair stencil, the four results leave as one 16-byte store (coefficients and
//            deltas in phase 2, delta-deltas in phase 3).
// Positions outside the utterance hold the clamped frame's values (replicate padding, torchaudio ComputeDeltas).
// Shared rows are [4 pad | w | 4 pad] floats so that the window loads of the first and last quad stay in bounds.
// grid (tiles, rows); tt % 4 == 0, halo in {0, 4}.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float lg2_normal(float x) {   // x is never subnormal here: plain MUFU.LG2
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float quad_log_energy(float v, int log_mode, float floor_db) {
  if (log_mode == B200FE_LOG_DB) {
    v = fmaxf(3.0102999566398120f * lg2_normal(fmaxf(v, 1e-10f)), floor_db);
  } else if (log_mode == B200FE_LOG_LN) {
    v = 0.6931471805599453f * lg2_normal(v + 1e-6f);
  }
  return v;
}
// the stencil sum_m m x[m] / 10 (m = -2 .. 2) at four consecutive positions; a, b, c = x[-4..-1], x[0..3], x[4..7]
__device__ __forceinline__ float4 quad_delta(const float4 a, const float4 b, const float4 c, float inv_denom) {
  float4 d;
  d.x = fmaf(2.0f, b.z - a.z, b.y - a.w) * inv_denom;
  d.y = fmaf(2.0f, b.w - a.w, b.z - b.x) * inv_denom;
  d.z = fmaf(2.0f, c.x - b.x, b.w - b.y) * inv_denom;
  d.w = fmaf(2.0f, c.y - b.y, c.x - b.z) * inv_denom;
  return d;
}

#ifndef FE_QUAD_UNROLL
#define FE_QUAD_UNROLL 2
#define FE_QUAD_QUAL __maxnreg__(KQ <= 6 ? 56 : 80)   // 56: 5 CTAs of 224 threads per SM
#endif
#define FE_PRAGMA(x) _Pragma(#x)
#define FE_UNROLL(n) FE_PRAGMA(unroll n)
template <int KQ, int NFT>   // NFT: n_filter when it equals the coefficient count 4*KQ (every loop unrolls), else 0
__global__ void FE_QUAD_QUAL fe_tail_quad_kernel(fe_tail_args a, int tiles_per_row, int n_tiles) {
  constexpr int kRegs = 4 * KQ;   // = n_coef
  constexpr int kUnrollF = NFT ? NFT : FE_QUAD_UNROLL, kUnrollQ = NFT ? (NFT + 3) / 4 : 1;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int tt = a.tt, halo = a.halo, w = tt + 2 * halo, ws = w + 8;
  const int nfil = NFT ? NFT : a.n_filter;
  const int nF = a.n_frames;
  float* s_dct = reinterpret_cast<float*>(smem_raw);   // [nfil][kRegs]
  float* s_c = s_dct + nfil * kRegs + 4;               // [kRegs][ws], position 0 at +4
  float* s_d = s_c + kRegs * ws;                       // [max(kRegs, nfil)][ws]
  float* s_e = s_d;                                    // [nfil][ws] the tile's energies land in the delta rows (free until phase 2)

  const int j = threadIdx.x;
  // (filter | channel, quad) items: quad q of the tile = positions 4q .. 4q+3, rows kl, kl+4, ...
  const int nqt = blockDim.x >> 2;
  const int q = j % nqt, kl = j / nqt;
  const int p0 = 4 * q;
  const bool in_tile = p0 < w;
  const float inv_denom = 0.1f;   // 3 / (n (n+1) (2n+1)), n = 2

  // A tile's energies come from L2 / HBM (a microsecond under load).  They are fetched with cp.async (no registers
  // held), 16 bytes = four frames of one filter each, all issued before anything else.  Quads outside the utterance
  // take the clamped frame four times (replicate padding).  One tile per CTA: a persistent form of this kernel (CTAs
  // walking tiles, the next tile's fetch issued under the delta phases, 54 KB -> 4 CTAs per SM) measured 0.139 ms
  // against 0.125 ms per 4096 utterances: the kernel is bound by the shared-memory pipe and instruction issue
  // (both ~65 % busy), not by the exposed fetch latency, and the fifth resident CTA is worth more than the overlap.
  auto fetch = [&](int g) {
    if (g < n_tiles && in_tile) {
      const int rl = g / tiles_per_row;
      const int fr = (g - rl * tiles_per_row) * tt - halo + p0;   // multiple of 4, like n_frames: inside or outside
      const bool inside = fr >= 0 && fr < nF;
      const float* src = a.energies + ((size_t)rl * nfil + kl) * nF + (inside ? fr : (fr < 0 ? 0 : nF - 1));
      uint32_t dst = (uint32_t)__cvta_generic_to_shared(s_e + kl * ws + p0);
      const size_t src_step = (size_t)4 * nF;
      const uint32_t dst_step = (uint32_t)ws * 16u;
      if (inside) {
#pragma unroll kUnrollQ
        for (int f = kl; f < nfil; f += 4, src += src_step, dst += dst_step)
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
      } else {
        for (int f = kl; f < nfil; f += 4, src += src_step, dst += dst_step)
#pragma unroll
          for (int i = 0; i < 4; ++i)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 4u * i), "l"(src) : "memory");
      }
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  fetch(blockIdx.x);
  const unsigned char* blob = reinterpret_cast<const unsigned char*>(a.tables);
  const fe_blob_header* h = reinterpret_cast<const fe_blob_header*>(blob);
  {
    const float4* gd = reinterpret_cast<const float4*>(blob + h->off_dct);   // [nfil][kRegs] floats, 16-byte aligned
    const int n4 = nfil * KQ;
    for (int i = j; i < n4; i += blockDim.x) reinterpret_cast<float4*>(s_dct)[i] = gd[i];
  }

  {
    const int g = blockIdx.x;
    const int row_local = g / tiles_per_row;
    const int64_t row = a.row_base + row_local;
    const int t0 = (g - row_local * tiles_per_row) * tt;
    const int tv0 = t0 - halo;
    const int tcl = fe_clampi(tv0 + j, 0, nF - 1) - tv0;
    float floor_db = -INFINITY;
    if (a.log_mode == B200FE_LOG_DB && a.top_db >= 0.0f) {
      // (a 64-bit division costs ~80 instructions; the row index of any real batch fits 32 bits)
      const int64_t grp = a.top_db_group == 1 ? row
                          : (row >> 32) == 0 ? (int64_t)((uint32_t)row / (uint32_t)a.top_db_group) : row / a.top_db_group;
      const float gmax = __uint_as_float(a.group_max[grp]);
      floor_db = 3.0102999566398120f * lg2_normal(fmaxf(gmax, 1e-10f)) - a.top_db;
    }
    asm volatile("cp.async.wait_all;" ::: "memory");
    __syncthreads();   // the tile's energies and the table are in

    if (j < w) {
      float c[kRegs];
#pragma unroll
      for (int k = 0; k < kRegs; ++k) c[k] = 0.0f;
      const float* ej = s_e + j;
      const float4* dr = reinterpret_cast<const float4*>(s_dct);
#pragma unroll kUnrollF
      for (int f = 0; f < nfil; ++f, dr += KQ, ej += ws) {
        const float v = quad_log_energy(*ej, a.log_mode, floor_db);
#pragma unroll
        for (int k4 = 0; k4 < KQ; ++k4) {
          const float4 d = dr[k4];
          c[4 * k4 + 0] = fmaf(v, d.x, c[4 * k4 + 0]);
          c[4 * k4 + 1] = fmaf(v, d.y, c[4 * k4 + 1]);
          c[4 * k4 + 2] = fmaf(v, d.z, c[4 * k4 + 2]);
          c[4 * k4 + 3] = fmaf(v, d.w, c[4 * k4 + 3]);
        }
      }
      float* sc = s_c + j;
#pragma unroll
      for (int k = 0; k < kRegs; ++k) sc[k * ws] = c[k];
    }
    __syncthreads();

    const bool owner = p0 >= halo && p0 < halo + tt && tv0 + p0 < nF;   // whole quads: tt, halo, nF are multiples of 4
    float* out_q = a.out + (size_t)row * a.n_out * nF + (tv0 + p0);
    if (a.deltas == 0) {
      if (owner)
        for (int k = kl; k < kRegs; k += 4)
          *reinterpret_cast<float4*>(out_q + (size_t)k * nF) = *reinterpret_cast<const float4*>(s_c + k * ws + p0);
      return;
    }
    if (in_tile) {
      for (int k = kl; k < kRegs; k += 4) {
        const float4* p = reinterpret_cast<const float4*>(s_c + k * ws + p0);
        const float4 b = p[0];
        const float4 d = quad_delta(p[-1], b, p[1], inv_denom);
        *reinterpret_cast<float4*>(s_d + k * ws + p0) = d;
        if (owner) {
          *reinterpret_cast<float4*>(out_q + (size_t)k * nF) = b;
          *reinterpret_cast<float4*>(out_q + (size_t)(kRegs + k) * nF) = d;
        }
      }
    }
    if (a.deltas < 2) return;
    __syncthreads();
    if (tv0 < 0 || tv0 + w > nF) {   // block-uniform: the tile reaches over an end of the utterance
      // replicate padding of the delta series: positions outside the utterance take the delta at the clamped frame
      if (j < w && tcl != j) {
        const float* from = s_d + tcl;
        float* to = s_d + j;
#pragma unroll 4
        for (int k = 0; k < kRegs; ++k) to[k * ws] = from[k * ws];
      }
      __syncthreads();
    }
    if (owner) {
      for (int k = kl; k < kRegs; k += 4) {
        const float4* p = reinterpret_cast<const float4*>(s_d + k * ws + p0);
        *reinterpret_cast<float4*>(out_q + (size_t)(2 * kRegs + k) * nF) = quad_delta(p[-1], p[0], p[1], inv_denom);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// fe_cmvn_kernel : one warp per (row, channel); in place
// ------------------------------------------------------------------------------------------------
__global__ void fe_cmvn_kernel(float* out, int64_t n_series, int n_frames, float eps) {
  const int64_t s = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (s >= n_series) return;
  const int lane = threadIdx.x & 31;
  float* p = out + s * n_frames;
  float sum = 0.0f;
  for (int t = lane; t < n_frames; t += 32) sum += p[t];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum / (float)n_frames;
  float var = 0.0f;
  for (int t = lane; t < n_frames; t += 32) {
    const float d = p[t] - mean;
    var = fmaf(d, d, var);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) var += __shfl_xor_sync(0xffffffffu, var, o);
  const float inv = 1.0f / (sqrtf(var / (float)n_frames) + eps);
  for (int t = lane; t < n_frames; t += 32) p[t] = (p[t] - mean) * inv;
}

// ------------------------------------------------------------------------------------------------
// fe_deltas_kernel : stand-alone ComputeDeltas on [rows][T]
// ------------------------------------------------------------------------------------------------
__global__ void fe_deltas_kernel(const float* __restrict__ in, float* __restrict__ out, int64_t rows,
                                 int64_t T, int n, float denom) {
  const int64_t row = blockIdx.y;
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= rows || t >= T) return;
  const float* p = in + row * T;
  float acc = 0.0f;
  for (int m = -n; m <= n; ++m) {
    int64_t u = t + m;
    u = u < 0 ? 0 : (u >= T ? T - 1 : u);
    acc += (float)m * __ldg(p + u);
  }
  out[row * T + t] = acc / denom;
}

// ------------------------------------------------------------------------------------------------
// fe_dense_rows_kernel : clips (ragged, repeat-padded / truncated to T as pad() does, maze5.py:280-285, or zero-padded /
// truncated with pad_zero) and / or pre-emphasis -> dense rows [rows][T] the streaming tcgen05 kernel can fetch with
// TMA boxes.
// One thread = four consecutive samples of one row, one 16-byte store (VEC4: T % 4 == 0; otherwise four scalar stores,
// for the FFT variant, which reads dense rows of any T).  Samples are float32 or 16-bit PCM converted as x / 32768
// (exact in fp32: what a FLAC / WAV decoder's float conversion yields), read one at a time: an int16 clip may start on
// any 2-byte boundary.  Row r's clip starts offsets[r] - base samples into `wave`, which then holds only the span of
// the flat clip buffer from sample `base` on; without offsets, `wave` holds dense rows [rows][T].
// ------------------------------------------------------------------------------------------------
FE_HD float fe_sample_f32(float x) { return x; }
FE_HD float fe_sample_f32(int16_t x) { return (1.0f / 32768.0f) * (float)x; }

template <typename S, bool VEC4>
__global__ void __launch_bounds__(256) fe_dense_rows_kernel(const S* __restrict__ wave,
                                                           const int64_t* __restrict__ offsets,
                                                           const int32_t* __restrict__ lengths, int64_t row_base,
                                                           int T, float preemph, float* __restrict__ dst,
                                                           int64_t flat_rel, int64_t base, int pad_zero) {
  const int64_t row = row_base + blockIdx.y;
  const S* src;
  int clip_len;
  if (offsets) {
    src = wave + (offsets[row] - base);
    clip_len = lengths[row];
    if (fe_clip_in_place(offsets[row], clip_len, T, flat_rel)) return;   // the streaming kernel reads this clip in place
  } else {
    src = wave + row * (int64_t)T;
    clip_len = T;
  }
  float* d = dst + (int64_t)blockIdx.y * T;
  // same values as fe_padded_sample(), with the clip index carried instead of recomputed per sample
  const bool wrap = clip_len < T && !pad_zero;
  const bool zero_tail = clip_len < T && pad_zero;
  for (int r = (blockIdx.x * blockDim.x + threadIdx.x) * 4; r < T; r += gridDim.x * blockDim.x * 4) {
    if (zero_tail && r > clip_len) {   // past the clip and its pre-emphasis boundary y[len]: zeros, nothing to read
      if (VEC4) {
        *reinterpret_cast<float4*>(d + r) = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
          if (r + i < T) d[r + i] = 0.0f;
      }
      continue;
    }
    // wrap: c < clip_len.  Otherwise c = r + i, which reaches clip_len only in a zero tail (samples 0, and `prev`
    // carries clip[len-1] into y[len])
    int c = wrap ? r % clip_len : r;
    float prev = 0.0f;
    if (preemph != 0.0f && r > 0) prev = fe_sample_f32(src[c == 0 ? clip_len - 1 : c - 1]);
    float v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float x = ((VEC4 || r + i < T) && c < clip_len) ? fe_sample_f32(src[c]) : 0.0f;
      v[i] = (preemph != 0.0f && r + i > 0) ? fmaf(-preemph, prev, x) : x;
      prev = x;
      c = (c + 1 == clip_len && wrap) ? 0 : c + 1;
    }
    if (VEC4) {
      *reinterpret_cast<float4*>(d + r) = make_float4(v[0], v[1], v[2], v[3]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (r + i < T) d[r + i] = v[i];
    }
  }
}

// ------------------------------------------------------------------------------------------------
// fe_tail_pointwise_kernel : the tail when there is no DCT and no deltas (mel features): out = log/dB(energies)
// element by element with the arithmetic of fe_tail_load; a row's [n_filter][n_frames] block is contiguous on
// both sides.  grid (blocks per row, rows), 4 elements per thread, coalesced.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fe_tail_pointwise_kernel(fe_tail_args a) {
  const int64_t row_local = blockIdx.y, row = a.row_base + row_local;
  const int64_t per_row = (int64_t)a.n_filter * a.n_frames;
  float floor_db = -INFINITY;
  if (a.log_mode == B200FE_LOG_DB && a.top_db >= 0.0f) {
    const float gmax = __uint_as_float(a.group_max[row / a.top_db_group]);
    floor_db = 10.0f * log10f(fmaxf(gmax, 1e-10f)) - a.top_db;
  }
  const float* src = a.energies + (size_t)row_local * per_row;
  float* dst = a.out + (size_t)row * per_row;
  const int64_t i0 = (int64_t)blockIdx.x * 1024 + threadIdx.x;
  float v[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) v[u] = (i0 + 256 * u < per_row) ? src[i0 + 256 * u] : 1.0f;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    float x = v[u];
    if (a.log_mode == B200FE_LOG_DB) {
      x = fmaxf(10.0f * log10f(fmaxf(x, 1e-10f)), floor_db);
    } else if (a.log_mode == B200FE_LOG_LN) {
      x = logf(x + 1e-6f);
    }
    if (i0 + 256 * u < per_row) dst[i0 + 256 * u] = x;
  }
}

cudaError_t set_smem(const void* fn, size_t bytes) {
  if (bytes <= 32 * 1024) return cudaSuccess;   // the 48 KB default covers static + dynamic: opt in well below it
  return fe_ensure_smem(fn, bytes);
}

}  // namespace

thread_local int64_t fe_launch_count = 0;

cudaError_t fe_ensure_smem(const void* fn, size_t bytes) {
  // The opt-in is process-wide per (function, device), and it costs a microsecond or two per call, which a small-batch
  // launch notices.  The largest size granted so far is kept per (function, device) under one lock: two host threads
  // launching the same kernel with different sizes must not lower the attribute below what the other was granted
  // (its launch would then be rejected), so a smaller request never calls cudaFuncSetAttribute.
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> granted;
  const int dev = fe_current_device();
  if (dev < 0) return cudaErrorInvalidDevice;
  std::lock_guard<std::mutex> lock(mu);
  size_t& have = granted[{fn, dev}];
  if (have >= bytes) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) have = bytes;
  return e;
}

int fe_current_device(void) {
  int dev = -1;
  return cudaGetDevice(&dev) == cudaSuccess ? dev : -1;
}

int fe_device_sms(int dev) {
  static std::atomic<int> cache[kFeMaxDevices];   // 0: not queried yet
  if (dev >= 0 && dev < kFeMaxDevices) {
    const int c = cache[dev].load(std::memory_order_relaxed);
    if (c > 0) return c;
  }
  int sms = 0;
  if (dev < 0 || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms < 1) return 1;
  if (dev < kFeMaxDevices) cache[dev].store(sms, std::memory_order_relaxed);
  return sms;
}

int fe_fft_warps_for(int n_fft) {
  // per-warp ping-pong buffers: 2 * (n_fft/2 + 1) complex; keep them within ~96 KB
  int w = (96 * 1024) / (2 * (n_fft / 2 + 1) * 8);
  return w > kFftWarps ? kFftWarps : (w < 1 ? 1 : w);
}

int fe_fft_fast_e(int n_fft, int hop) {
  // register-resident warp FFT where the geometry allows it (B200FE_SMEM_FFT: test hook for the Stockham path)
  if ((hop & 1) != 0 || getenv("B200FE_SMEM_FFT") != nullptr) return 0;
  return n_fft == 256 ? 4 : n_fft == 512 ? 8 : n_fft == 1024 ? 16 : 0;
}

// Band weights are copied to shared memory when they fit this many floats (any triangular bank does).
static int fe_rfft_bw_cap(int n_fft, int n_filter) { return 2 * (n_fft / 2 + 1) + 2 * n_filter; }

size_t fe_fft_smem_bytes(int n_fft, int hop, int ft, int n_ch, int mode) {
  const int nh = n_fft / 2;
  size_t seg = (size_t)(ft - 1) * hop + n_fft;
  size_t b = (seg * 4 + 15) & ~(size_t)15;
  const int E = fe_fft_fast_e(n_fft, hop);
  if (E > 0) {
    const int zunits = E == 4 ? fe_rfft_zunits<4>() : E == 8 ? fe_rfft_zunits<8>() : fe_rfft_zunits<16>();
    b += (size_t)n_fft * 4 + ((((size_t)(nh / 2 + 1)) * 8 + 15) & ~(size_t)15);
    b += (size_t)kFftWarps * zunits * 8;
    b += (((size_t)(nh + 1) * (ft + 1) * 4) + 15) & ~(size_t)15;
    if (mode == 1)
      b += ((((size_t)n_ch * (ft + 1) * 4) + 15) & ~(size_t)15) + (size_t)fe_rfft_bw_cap(n_fft, n_ch) * 4 + 16 +
           (size_t)n_ch * 16;
    return b;
  }
  b += (size_t)n_fft * 4 + (size_t)nh * 8 + ((((size_t)(nh / 2 + 1)) * 8 + 15) & ~(size_t)15);
  b += (size_t)fe_fft_warps_for(n_fft) * 2 * (nh + 1) * 8;
  b += (size_t)n_ch * (ft + 1) * 4;
  return b;
}

// Frames per CTA: the fast path wants several CTAs per SM (phases of different CTAs overlap) and 16 or 32
// frames, the shared-memory Stockham path the largest tile that fits.  0: does not fit.
int fe_fft_pick_ft(int n_fft, int hop, int n_ch, int mode) {
  const int E = fe_fft_fast_e(n_fft, hop);
  if (E > 0) {
    const size_t want = (E == 16 ? 113 : 56) * 1024;   // 2 CTAs / SM at 128 registers, 4 at 64
    for (int ft = 32; ft >= 16; ft >>= 1)
      if (fe_fft_smem_bytes(n_fft, hop, ft, n_ch, mode) <= want) return ft;
    return fe_fft_smem_bytes(n_fft, hop, 16, n_ch, mode) <= 200 * 1024 ? 16 : 0;
  }
  for (int ft = 32; ft >= 4; ft >>= 1)
    if (fe_fft_smem_bytes(n_fft, hop, ft, n_ch, mode) <= 200 * 1024) return ft;
  return 0;
}

cudaError_t fe_launch_fft(const fe_fft_args& a_in, int mode, int64_t rows, cudaStream_t stream) {
  fe_fft_args a = a_in;
  a.fft_warps = fe_fft_warps_for(a.n_fft);
  const int n_ch = mode == 0 ? a.n_fft / 2 + 1 : a.n_filter;
  const size_t smem = fe_fft_smem_bytes(a.n_fft, a.hop, a.ft, n_ch, mode);
  const int E = fe_fft_fast_e(a.n_fft, a.hop);
  void (*kern)(fe_fft_args);
  switch (E * 2 + (mode != 0)) {
    case 8: kern = fe_rfft_kernel<0, 4>; break;
    case 9: kern = fe_rfft_kernel<1, 4>; break;
    case 16: kern = fe_rfft_kernel<0, 8>; break;
    case 17: kern = fe_rfft_kernel<1, 8>; break;
    case 32: kern = fe_rfft_kernel<0, 16>; break;
    case 33: kern = fe_rfft_kernel<1, 16>; break;
    case 0: kern = fe_fft_kernel<0>; break;
    default: kern = fe_fft_kernel<1>; break;
  }
  cudaError_t e = set_smem((const void*)kern, smem);
  if (e != cudaSuccess) return e;
  int64_t resident = 0x7fffffffLL;
  if (E > 0) {   // persistent CTAs: as many as are resident at once
    const int sms = fe_device_sms(fe_current_device());
    int per_sm = 1;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kFftThreads, smem);
    if (e != cudaSuccess) return e;
    resident = (int64_t)sms * (per_sm > 0 ? per_sm : 1);
  }
  // one CTA per (row, tile): keep each launch's grid below 2^31 CTAs; `out` and `wave_chunk` hold the launch's rows
  return fe_launch_rows(rows, 0x7fffffffLL / a.tiles_per_row, [&](int64_t r0, int64_t nr) {
    fe_fft_args b = a;
    b.row_base = a.row_base + r0;
    b.out = a.out + (size_t)r0 * n_ch * a.n_frames;
    if (a.wave_chunk) b.wave_chunk = a.wave_chunk + r0 * a.T;
    b.n_blocks = nr * a.tiles_per_row;
    kern<<<(unsigned)(b.n_blocks < resident ? b.n_blocks : resident), kFftThreads, smem, stream>>>(b);
    return cudaSuccess;
  });
}

size_t fe_tail_smem_bytes(const fe_tail_args& a) {
  const int w = a.tt + 2 * a.halo;
  const int nc = a.n_coef > 0 ? a.n_coef : a.n_filter;
  size_t fl = (size_t)a.n_filter * w;
  if (a.n_coef > 0) fl += (size_t)nc * w;
  if (a.deltas > 0) fl += (size_t)nc * w;
  fl += (size_t)a.n_filter * a.n_coef;
  return fl * 4;
}

// The tail arguments of a launch over rows [r0, ...) of a's rows (energies hold a's rows from a.row_base on).
static fe_tail_args tail_rows_from(const fe_tail_args& a, int64_t r0) {
  fe_tail_args b = a;
  b.row_base = a.row_base + r0;
  b.energies = a.energies + (size_t)r0 * a.n_filter * a.n_frames;
  return b;
}

template <int N, bool EXACT>
static void (*pick_tail_fast(int kq))(fe_tail_args) {
  switch (kq) {
    case 1: return fe_tail_fast_kernel<1, N, EXACT>;
    case 2: return fe_tail_fast_kernel<2, N, EXACT>;
    case 3: return fe_tail_fast_kernel<3, N, EXACT>;
    case 4: return fe_tail_fast_kernel<4, N, EXACT>;
    case 5: return fe_tail_fast_kernel<5, N, EXACT>;
    case 6: return fe_tail_fast_kernel<6, N, EXACT>;
    case 7: return fe_tail_fast_kernel<7, N, EXACT>;
    default: return fe_tail_fast_kernel<8, N, EXACT>;
  }
}

// fe_tail_quad_kernel where its shape conditions hold (the LFCC configurations of SURVEY.md 8: 20 coefficients,
// win_length 5 deltas, 404 frames); false: not applicable, the caller goes on to fe_tail_fast_kernel
static bool launch_tail_quad(const fe_tail_args& a_in, int64_t rows, cudaStream_t stream, cudaError_t* err) {
  fe_tail_args a = a_in;
  const int nc = a.n_coef;
  if (nc < 4 || (nc & 3) || (a.n_frames & 3) || ((reinterpret_cast<uintptr_t>(a.out) | reinterpret_cast<uintptr_t>(a.tables) | reinterpret_cast<uintptr_t>(a.energies)) & 15)) return false;
  if (a.deltas > 0 && a.delta_win != 5) return false;
  a.halo = a.deltas > 0 ? 4 : 0;   // deltas = 1 needs 2: rounded up to whole quads
  const int max_tt = 256 - 2 * a.halo;
  const int tiles = (a.n_frames + max_tt - 1) / max_tt;
  a.tt = (((a.n_frames + tiles - 1) / tiles) + 3) & ~3;
  const int w = a.tt + 2 * a.halo;
  const int threads = (w + 31) & ~31;
  // table, coefficient rows, delta rows (which first receive the n_filter energy rows)
  const size_t smem = ((size_t)a.n_filter * nc + 4 + (size_t)(nc + (nc > a.n_filter ? nc : a.n_filter)) * (w + 8) + 4) * 4;
  typedef void (*kern_t)(fe_tail_args, int, int);
  kern_t kern;
  const bool sq = a.n_filter == nc;   // the square DCT (20 x 20 for the LFCC front-end): n_filter at compile time
  switch (nc >> 2) {
    case 1: kern = sq ? fe_tail_quad_kernel<1, 4> : fe_tail_quad_kernel<1, 0>; break;
    case 2: kern = sq ? fe_tail_quad_kernel<2, 8> : fe_tail_quad_kernel<2, 0>; break;
    case 3: kern = sq ? fe_tail_quad_kernel<3, 12> : fe_tail_quad_kernel<3, 0>; break;
    case 4: kern = sq ? fe_tail_quad_kernel<4, 16> : fe_tail_quad_kernel<4, 0>; break;
    case 5: kern = sq ? fe_tail_quad_kernel<5, 20> : fe_tail_quad_kernel<5, 0>; break;
    case 6: kern = sq ? fe_tail_quad_kernel<6, 24> : fe_tail_quad_kernel<6, 0>; break;
    case 7: kern = sq ? fe_tail_quad_kernel<7, 28> : fe_tail_quad_kernel<7, 0>; break;
    default: kern = fe_tail_quad_kernel<8, 0>; break;   // (32 x 32 fully unrolled spills)
  }
  *err = set_smem((const void*)kern, smem);
  if (*err != cudaSuccess) return true;
  // one CTA per (row, tile), a 1-D grid (no 65535-row limit); tile indices (and index + grid) are 32-bit in the kernel
  *err = fe_launch_rows(rows, (int64_t)0x3fffffff / tiles, [&](int64_t r0, int64_t nr) {
    const int n_tiles = (int)(nr * tiles);
    kern<<<(unsigned)n_tiles, threads, smem, stream>>>(tail_rows_from(a, r0), tiles, n_tiles);
    return cudaSuccess;
  });
  return true;
}

static cudaError_t launch_tail_fast(const fe_tail_args& a_in, int64_t rows, cudaStream_t stream) {
  fe_tail_args a = a_in;
  if (a.force_generic != 2) {   // 2: test hook, fe_tail_fast_kernel where fe_tail_quad_kernel applies
    cudaError_t e = cudaSuccess;
    if (launch_tail_quad(a_in, rows, stream, &e)) return e;
  }
  // tile so that tt + 2*halo fills (almost) a whole number of warps, at most 256 threads
  const int max_tt = 256 - 2 * a.halo;
  const int tiles = (a.n_frames + max_tt - 1) / max_tt;
  a.tt = (a.n_frames + tiles - 1) / tiles;
  const int w = a.tt + 2 * a.halo;
  const int threads = (w + 31) & ~31;
  const int nc = a.n_coef > 0 ? a.n_coef : a.n_filter;
  const int kq = (nc + 3) / 4;
  const size_t smem = ((size_t)2 * nc * w + (size_t)a.n_filter * 4 * kq + (size_t)a.n_filter * w) * 4;
  typedef void (*kern_t)(fe_tail_args);
  const int n = a.deltas > 0 ? (a.delta_win - 1) / 2 : 0;
  const bool exact = nc == 4 * kq;
  // delta half-width 2 (torchaudio's win_length = 5) is unrolled; every other width runs the loop form
  const kern_t kern = exact ? (n == 2 ? pick_tail_fast<2, true>(kq) : pick_tail_fast<0, true>(kq))
                            : (n == 2 ? pick_tail_fast<2, false>(kq) : pick_tail_fast<0, false>(kq));
  cudaError_t e = set_smem((const void*)kern, smem);
  if (e != cudaSuccess) return e;
  return fe_launch_rows(rows, 65535, [&](int64_t r0, int64_t nr) {
    kern<<<dim3((unsigned)tiles, (unsigned)nr), threads, smem, stream>>>(tail_rows_from(a, r0));
    return cudaSuccess;
  });
}

cudaError_t fe_launch_tail(const fe_tail_args& a, int64_t rows, cudaStream_t stream) {
  if (a.n_coef == 0 && a.deltas == 0 && a.force_generic != 1) {
    const int64_t per_row = (int64_t)a.n_filter * a.n_frames;
    return fe_launch_rows(rows, 65535, [&](int64_t r0, int64_t nr) {
      fe_tail_pointwise_kernel<<<dim3((unsigned)((per_row + 1023) / 1024), (unsigned)nr), 256, 0, stream>>>(
          tail_rows_from(a, r0));
      return cudaSuccess;
    });
  }
  if (a.n_filter <= kFastMax && a.n_coef <= kFastMax && a.force_generic != 1) return launch_tail_fast(a, rows, stream);
  const size_t smem = fe_tail_smem_bytes(a);
  cudaError_t e = set_smem((const void*)fe_tail_kernel, smem);
  if (e != cudaSuccess) return e;
  const int tiles = (a.n_frames + a.tt - 1) / a.tt;
  // grid.y is limited to 65535 rows per launch
  return fe_launch_rows(rows, 65535, [&](int64_t r0, int64_t nr) {
    fe_tail_kernel<<<dim3((unsigned)tiles, (unsigned)nr), kTailThreads, smem, stream>>>(tail_rows_from(a, r0));
    return cudaSuccess;
  });
}

cudaError_t fe_launch_cmvn(float* out, int64_t n_series, int n_frames, cudaStream_t stream) {
  const int warps = 8;
  const int64_t grid = (n_series + warps - 1) / warps;
  fe_cmvn_kernel<<<(unsigned)grid, warps * 32, 0, stream>>>(out, n_series, n_frames, 1e-5f);
  return fe_launched();
}

cudaError_t fe_launch_deltas(const float* in, float* out, int64_t rows, int64_t T, int win,
                             cudaStream_t stream) {
  const int n = (win - 1) / 2;
  const float denom = (float)(n * (n + 1) * (2 * n + 1)) / 3.0f;
  return fe_launch_rows(rows, 65535, [&](int64_t r0, int64_t nr) {
    fe_deltas_kernel<<<dim3((unsigned)((T + 255) / 256), (unsigned)nr), 256, 0, stream>>>(in + r0 * T, out + r0 * T,
                                                                                         nr, T, n, denom);
    return cudaSuccess;
  });
}

template <typename S>
static cudaError_t launch_dense_rows(const S* wave, const int64_t* offsets, const int32_t* lengths, int64_t row_base,
                                     int64_t rows, int64_t T, float preemph, float* dst, cudaStream_t stream,
                                     int64_t flat_rel, int64_t base, int pad_zero) {
  // CTAs per row: each thread walks its row in T / (1024 bx) steps.  One CTA per 1024 samples (64 per LFCC row) was
  // measured slowest; 16 per row is best when every row is copied (all-staged ragged step 1.30 -> 1.24 ms per 4096
  // clips, profiles/r2_ragged_inplace.txt), 8 when rows the streaming kernel reads in place are in the batch: those
  // leave at once, and a skipped row should cost few empty CTAs.
  unsigned bx = (unsigned)((T / 4 + 255) / 256);
  const unsigned cap = flat_rel >= 0 ? 8 : 16;
  if (bx > cap) bx = cap;
  const bool vec4 = (T & 3) == 0;
  return fe_launch_rows(rows, 65535, [&](int64_t r0, int64_t nr) {
    dim3 grid(bx, (unsigned)nr);
    if (vec4)
      fe_dense_rows_kernel<S, true><<<grid, 256, 0, stream>>>(wave, offsets, lengths, row_base + r0, (int)T, preemph,
                                                              dst + r0 * T, flat_rel, base, pad_zero);
    else
      fe_dense_rows_kernel<S, false><<<grid, 256, 0, stream>>>(wave, offsets, lengths, row_base + r0, (int)T, preemph,
                                                               dst + r0 * T, flat_rel, base, pad_zero);
    return cudaSuccess;
  });
}

cudaError_t fe_launch_dense_rows(const float* wave, const int64_t* offsets, const int32_t* lengths,
                                 int64_t row_base, int64_t rows, int64_t T, float preemph, float* dst,
                                 cudaStream_t stream, int64_t flat_rel, int64_t base, int pad_zero) {
  return launch_dense_rows(wave, offsets, lengths, row_base, rows, T, preemph, dst, stream, flat_rel, base, pad_zero);
}

cudaError_t fe_launch_dense_rows(const int16_t* wave, const int64_t* offsets, const int32_t* lengths,
                                 int64_t row_base, int64_t rows, int64_t T, float preemph, float* dst,
                                 cudaStream_t stream, int64_t base, int pad_zero) {
  return launch_dense_rows(wave, offsets, lengths, row_base, rows, T, preemph, dst, stream, (int64_t)-1, base,
                           pad_zero);
}
