// Warp-level phases of the shared-memory real FFT (variant B200FE_VARIANT_FFT).
//
// One warp transforms one frame.  A real n_fft-point transform is done as an n_fft/2-point complex
// Stockham autosort FFT (radix-4 stages, plus one radix-2 stage when log2(n_fft/2) is odd) on the
// packed sequence z[n] = x[2n] + i*x[2n+1], followed by the real-FFT split that yields the power of
// bins 0..n_fft/2 directly.  Every function here is the share of ONE lane of ONE phase; phases are
// separated by __syncwarp() in the kernel.  The same functions compile as plain C++ so the index
// logic is exercised on the CPU (tests/emu) where lanes are a loop.
//
// What this computes is |rfft(frame * window)|^2, i.e. torch.stft(...).abs().pow(2) as called by
// torchaudio functional/functional.py:123-145.
#ifndef FE_FFT_CUH_
#define FE_FFT_CUH_

#include <math.h>
#include "fe_common.h"

FE_HD fe_c2 fe_cmul(fe_c2 a, fe_c2 b) {
  fe_c2 r;
  r.x = a.x * b.x - a.y * b.y;
  r.y = a.x * b.y + a.y * b.x;
  return r;
}

// Forward radix-4 butterfly (DFT_4 with exp(-2*pi*i/4) = -i), in place on v0..v3.
FE_HD void fe_bfly4(fe_c2& v0, fe_c2& v1, fe_c2& v2, fe_c2& v3) {
  fe_c2 a0 = {v0.x + v2.x, v0.y + v2.y};
  fe_c2 a1 = {v0.x - v2.x, v0.y - v2.y};
  fe_c2 a2 = {v1.x + v3.x, v1.y + v3.y};
  fe_c2 a3 = {v1.y - v3.y, v3.x - v1.x};  // (v1 - v3) * (-i)
  v0.x = a0.x + a2.x; v0.y = a0.y + a2.y;
  v1.x = a1.x + a3.x; v1.y = a1.y + a3.y;
  v2.x = a0.x - a2.x; v2.y = a0.y - a2.y;
  v3.x = a1.x - a3.x; v3.y = a1.y - a3.y;
}

// First stage (Ns = 1, no twiddles) fused with framing and windowing: reads the frame's samples
// straight from the staged waveform and multiplies by the centred window.  nh = n_fft / 2.
// `radix2_first` selects a radix-2 first stage (used when log2(nh) is odd).
FE_HD void fe_fft_stage_first(int lane, const float* frame, const float* win, fe_c2* out, int nh,
                              bool radix2_first) {
  if (!radix2_first) {
    const int q = nh >> 2;
    for (int j = lane; j < q; j += 32) {
      fe_c2 v[4];
#pragma unroll
      for (int r = 0; r < 4; ++r) {
        const int n = 2 * (j + r * q);
        v[r].x = frame[n] * win[n];
        v[r].y = frame[n + 1] * win[n + 1];
      }
      fe_bfly4(v[0], v[1], v[2], v[3]);
      fe_c2* o = out + 4 * j;
      o[0] = v[0]; o[1] = v[1]; o[2] = v[2]; o[3] = v[3];
    }
  } else {
    const int q = nh >> 1;
    for (int j = lane; j < q; j += 32) {
      const int n0 = 2 * j, n1 = 2 * (j + q);
      fe_c2 a = {frame[n0] * win[n0], frame[n0 + 1] * win[n0 + 1]};
      fe_c2 b = {frame[n1] * win[n1], frame[n1 + 1] * win[n1 + 1]};
      fe_c2 s = {a.x + b.x, a.y + b.y}, d = {a.x - b.x, a.y - b.y};
      out[2 * j] = s;
      out[2 * j + 1] = d;
    }
  }
}

// Generic radix-4 Stockham stage: sub-transform length so far `ns` (>= 1), tw = nh-th roots.
FE_HD void fe_fft_stage4(int lane, const fe_c2* in, fe_c2* out, const fe_c2* tw, int nh, int ns) {
  const int q = nh >> 2;
  const int tstride = nh / (4 * ns);
  for (int j = lane; j < q; j += 32) {
    const int k = j & (ns - 1);
    fe_c2 v0 = in[j], v1 = in[j + q], v2 = in[j + 2 * q], v3 = in[j + 3 * q];
    const int t = k * tstride;
    v1 = fe_cmul(v1, tw[t]);
    v2 = fe_cmul(v2, tw[2 * t]);
    v3 = fe_cmul(v3, tw[3 * t]);
    fe_bfly4(v0, v1, v2, v3);
    const int j0 = ((j - k) << 2) + k;
    out[j0] = v0;
    out[j0 + ns] = v1;
    out[j0 + 2 * ns] = v2;
    out[j0 + 3 * ns] = v3;
  }
}

// Real-FFT split + power: from Z = FFT_nh(z) to P[k] = |X[k]|^2 for k = 0..nh.
//   Fe = (Z[k] + conj Z[nh-k]) / 2,  Fo = (Z[k] - conj Z[nh-k]) / (2i),  W = exp(-2*pi*i*k/n_fft)
//   X[k] = Fe + W*Fo,  X[nh-k] = conj(Fe - W*Fo)
FE_HD void fe_fft_power(int lane, const fe_c2* z, const fe_c2* rtw, float* pw, int nh) {
  for (int k = lane; k <= (nh >> 1); k += 32) {
    const fe_c2 a = z[k];
    const fe_c2 b = z[(nh - k) & (nh - 1)];
    const fe_c2 fe2 = {a.x + b.x, a.y - b.y};  // 2*Fe
    const fe_c2 fo2 = {a.y + b.y, b.x - a.x};  // 2*Fo
    const fe_c2 t = fe_cmul(rtw[k], fo2);
    const float px = fe2.x + t.x, py = fe2.y + t.y;
    const float mx = fe2.x - t.x, my = fe2.y - t.y;
    pw[k] = 0.25f * (px * px + py * py);
    pw[nh - k] = 0.25f * (mx * mx + my * my);
  }
}

// Sparse triangular filterbank: each lane owns filters lane, lane+32, ...; a filter is a contiguous
// band of bins [start, start+len) with its own weights (torchaudio transforms/_transforms.py:818).
FE_HD void fe_fbank_apply(int lane, const float* pw, const int32_t* bstart, const int32_t* blen,
                          const int32_t* bwoff, const float* bw, int n_filter, float* e_out,
                          int e_stride) {
  for (int f = lane; f < n_filter; f += 32) {
    const int s = bstart[f], len = blen[f];
    const float* w = bw + bwoff[f];
    float acc = 0.0f;
    for (int i = 0; i < len; ++i) acc = fmaf(pw[s + i], w[i], acc);
    e_out[(size_t)f * e_stride] = acc;
  }
}

// Index of padded position `pp` (0 .. T + n_fft - 1, reflect padding by `half`) in the T-sample signal.
FE_HD int fe_reflect_index(int pp, int half, int T) {
  int r = pp - half;
  if (r < 0) r = -r;
  if (r >= T) r = 2 * (T - 1) - r;
  return r;
}

// Staging phase: thread `tid` of `nthreads` fills s_stage[i] for padded positions pp0 + i, i < seg.
// Padding is torch.stft's reflect padding by n_fft/2; the T-sample signal is the clip repeat-padded
// or truncated to T (pad(), Thesis/01_Models/01_Baseline_Models/maze5.py:280-285: sample r =
// clip[r mod len]), or with pad_zero != 0 zero-padded or truncated to T (the evaluation script's
// dataset: sample r = clip[r] for r < len, 0 after); optional pre-emphasis y[r] = x[r] - a*x[r-1],
// y[0] = x[0] (torchaudio functional/functional.py:2426-2448) is applied to the T-sample signal
// before the reflect padding, as torchaudio would.
// Sample r (0 <= r < T) of the T-sample signal a clip stands for: pad / truncate, then pre-emphasis.
// Without wrap-around every index c < T, so c >= clip_len happens only past the end of a zero-padded clip.
FE_HD float fe_padded_sample(const float* src, int clip_len, int T, int r, float preemph, int pad_zero = 0) {
  const bool wrap = clip_len < T && !pad_zero;
  const int c = wrap ? (r % clip_len) : r;
  float v = c < clip_len ? src[c] : 0.0f;
  if (preemph != 0.0f && r > 0) {
    const int c1 = wrap ? ((r - 1) % clip_len) : (r - 1);
    v = fmaf(-preemph, c1 < clip_len ? src[c1] : 0.0f, v);
  }
  return v;
}

FE_HD void fe_stage_load(int tid, int nthreads, const float* src, int clip_len, int T, int n_fft, int pp0,
                         int seg, float preemph, float* s_stage, int pad_zero = 0) {
  const int half = n_fft >> 1;
#pragma unroll 4
  for (int i = tid; i < seg; i += nthreads) {
    const int r = fe_reflect_index(pp0 + i, half, T);
    s_stage[i] = fe_padded_sample(src, clip_len, T, r, preemph, pad_zero);
  }
}

#endif  // FE_FFT_CUH_
