/*
 * b200fe.h — C-ABI of the B200 (sm_100a) spectral front-end.
 *
 * Drop-in boundary for the feature path of Ansh4121/audio-deepfake-detection-fmsl.  The reference is
 * pure Python and has no FFI of its own; the interface this library replaces is
 *   (i)  the nn.Module feature slot `out = self.sinc_conv(x)` — (B,1,T) float32 -> (B,C,T') float32
 *        Thesis/01_Models/01_Baseline_Models/maze5.py:241 (also maze4.py:228,
 *        02_FMSL_Enhanced_Models/maze5_fmsl_standardized.py:302, maze4_fmsl_standardized.py:287), and
 *   (ii) the arithmetic of the torchaudio transforms the reference depends on (maze5.py:32):
 *        torchaudio/transforms/_transforms.py:721-828 (LFCC), :25 (Spectrogram), :515 (MelSpectrogram),
 *        :300 (AmplitudeToDB), :992 (ComputeDeltas); torchaudio/functional/functional.py:119-145,
 *        :356, :961, :2426.
 * Each entry point below cites the piece it replaces.  Python binds these with ctypes
 * (audio-deepfake-detection-fmsl_b200/_lib.py); INTEGRATION.md shows the reference-side stub.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross the boundary;
 *   - the caller owns every buffer (waveforms, tables blob, workspace, output); the library allocates
 *     no device memory, frees nothing, and keeps no mutable global state besides a thread-local
 *     last-error string and cached per-kernel attributes;
 *   - all device work is enqueued on the `stream` argument (a cudaStream_t passed as void*); no
 *     implicit synchronisation; CUDA-graph capturable;
 *   - return value 0 = success, negative = b200fe_status error; nothing throws or exits.
 */
#ifndef B200FE_H_
#define B200FE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200FE_ABI_VERSION 1

typedef enum b200fe_status {
  B200FE_OK = 0,
  B200FE_ERR_BAD_ARG = -1,       /* null pointer, non-positive size, inconsistent params            */
  B200FE_ERR_UNSUPPORTED = -2,   /* legal in torchaudio but not implemented here (no CPU fallback)  */
  B200FE_ERR_WORKSPACE = -3,     /* workspace / tables buffer too small                             */
  B200FE_ERR_ALIGNMENT = -4,     /* pointer not aligned as documented                               */
  B200FE_ERR_CUDA = -5,          /* a CUDA runtime call failed; see b200fe_last_error_string()      */
  B200FE_ERR_NO_DEVICE = -6      /* no sm_100 device / kernels cannot run here                      */
} b200fe_status;

typedef enum b200fe_log_mode {
  B200FE_LOG_NONE = 0,           /* filterbank energies as they are (MelSpectrogram)                */
  B200FE_LOG_DB = 1,             /* 10*log10(clamp(x,1e-10)), then top_db clamp  (functional.py:356) */
  B200FE_LOG_LN = 2              /* log(x + 1e-6)  (LFCC log_lf=True, _transforms.py:820-822)        */
} b200fe_log_mode;

typedef enum b200fe_variant {
  B200FE_VARIANT_AUTO = 0,       /* fastest measured variant that supports the configuration        */
  B200FE_VARIANT_FFT = 1,        /* real FFT on the CUDA cores (register-resident warp FFT; Stockham fallback) */
  B200FE_VARIANT_DFT_GEMM = 2    /* folded DFT as a split-fp16 GEMM on tcgen05 tensor cores / TMEM   */
} b200fe_variant;

/* How a ragged clip shorter than T becomes a T-sample row (the pad_mode argument of the *_pad entry points).
 * A clip of at least T samples keeps its first T samples in both modes.  Pre-emphasis, when set, runs over the
 * T-sample row, then torch.stft's reflect padding. */
typedef enum b200fe_pad_mode {
  B200FE_PAD_REPEAT = 0,         /* sample i = clip[i mod len]: the training loader's pad() (maze5.py:280-285)       */
  B200FE_PAD_ZERO = 1            /* sample i = clip[i] for i < len, then 0.0f: the evaluation script's dataset
                                    (Maze5_eval.py:203-221); with pre-emphasis y[len] = -a*clip[len-1], later 0     */
} b200fe_pad_mode;

/* Everything that fixes the transform.  Mirrors the constructor arguments of torchaudio's
 * Spectrogram / LFCC / MelSpectrogram / ComputeDeltas (transforms/_transforms.py:25,721,515,992). */
typedef struct b200fe_params {
  int32_t abi_version;   /* B200FE_ABI_VERSION                                                     */
  int32_t n_fft;         /* power of two, 64..4096                                                  */
  int32_t win_length;    /* 1..n_fft; window is zero-padded centred to n_fft like torch.stft        */
  int32_t hop_length;    /* >= 1                                                                    */
  int32_t n_filter;      /* filterbank columns (n_filter of LFCC, n_mels of MelSpectrogram), 1..256 */
  int32_t n_coef;        /* DCT outputs (n_lfcc); 0 = no DCT, output the (log) filterbank energies  */
  int32_t log_mode;      /* b200fe_log_mode                                                         */
  float   top_db;        /* clamp range for B200FE_LOG_DB; < 0 disables the clamp (top_db=None)     */
  int32_t top_db_group;  /* consecutive rows that share one top_db maximum: 1 = per utterance (the   */
                         /* (B,1,T) semantics the maze models use, maze5.py:235-241); B = torchaudio's */
                         /* packing of a 2-D (B,T) input (functional.py:394-399)                    */
  int32_t deltas;        /* 0,1,2: rounds of ComputeDeltas concatenated on the coefficient axis     */
  int32_t delta_win;     /* ComputeDeltas win_length (odd, 3..9); mode is always 'replicate'        */
  float   preemph;       /* pre-emphasis coefficient, 0 = off (functional.py:2426)                  */
  int32_t cmvn;          /* 1 = per-utterance mean/variance normalisation over time (extension)     */
  int32_t variant;       /* b200fe_variant                                                          */
} b200fe_params;

/* ---- introspection ------------------------------------------------------------------------- */
int32_t     b200fe_version(void);                    /* B200FE_ABI_VERSION of the built library     */
const char* b200fe_last_error_string(void);          /* thread-local; never NULL                    */
const char* b200fe_status_string(int32_t status);
int32_t     b200fe_has_tcgen05(void);                /* 1 when the DFT-GEMM variant was compiled in */

/* 1 + T / hop  (torch.stft center=True framing, functional.py:123-134). <0 on bad args. */
int64_t b200fe_n_frames(const b200fe_params* p, int64_t T);
/* n_out = (n_coef ? n_coef : n_filter) * (1 + deltas) */
int64_t b200fe_n_out_channels(const b200fe_params* p);
/* variant AUTO resolves to for these params (B200FE_VARIANT_FFT or _DFT_GEMM); <0 on bad args */
int32_t b200fe_resolve_variant(const b200fe_params* p);

/* ---- constant tables ------------------------------------------------------------------------
 * The caller computes window / filterbank / DCT on the host with the same torch functions torchaudio
 * uses (torch.hann_window, F.linear_fbanks / F.melscale_fbanks, F.create_dct) so the table bits are
 * identical, and hands them to b200fe_tables_pack, a pure host function that lays them out (plus FFT
 * twiddles, the sparse band form of the filterbank and the fp16 hi/lo DFT operand tiles of the GEMM
 * variant) into one blob.  The caller uploads the blob once (16-byte aligned) and passes the device
 * copy as `tables` to the forward calls.
 *   window  float32[win_length]
 *   fbank   float32[n_fft/2+1][n_filter]  row-major (torchaudio layout), may be NULL for spectrogram-only
 *   dct     float32[n_filter][n_coef]     row-major (F.create_dct layout), NULL when n_coef == 0   */
int64_t b200fe_tables_bytes(const b200fe_params* p);
int32_t b200fe_tables_pack(const b200fe_params* p, const float* window, const float* fbank,
                           const float* dct, void* blob_host, size_t blob_bytes);

/* Which kernel family the forward calls should use with THIS packed blob: resolves
 * B200FE_VARIANT_AUTO (and validates an explicit request) against what the tables support — the
 * DFT-GEMM variant needs win_length == 2*hop_length, n_fft in {128..512}, a window symmetric about
 * the frame centre with window[0] == 0 (periodic Hann) and a triangular filterbank whose bins feed
 * at most two adjacent filters.  Returns B200FE_VARIANT_FFT / _DFT_GEMM, or an error when an
 * explicitly requested variant is not available.  Callers store the answer in params.variant;
 * forward calls given B200FE_VARIANT_AUTO use the FFT variant (they only see the device copy).
 * A forward call that says B200FE_VARIANT_DFT_GEMM with a blob this function would have refused
 * cannot be detected on the host (no synchronisation): the kernel traps and the stream reports a
 * CUDA error (B200FE_ERR_CUDA from the next call), it never returns garbage silently. */
int32_t b200fe_tables_variant(const b200fe_params* p, const void* blob_host);

/* ---- device entry points -------------------------------------------------------------------- */
/* Scratch needed by b200fe_features_forward for R rows of T samples (filterbank energies of one
 * chunk of rows + per-group maxima).  <0 on bad args. */
int64_t b200fe_workspace_bytes(const b200fe_params* p, int64_t R, int64_t T);
/* The same for a call that passes offsets / lengths (ragged != 0): with params.variant ==
 * B200FE_VARIANT_DFT_GEMM ragged clips (and pre-emphasised input, ragged or not) are first written as
 * dense repeat-padded rows, one chunk of rows at a time, into the workspace, which grows by chunk*T*4 bytes
 * (ragged clips of at least T samples whose first sample is 16-byte aligned are read in place instead; the
 * workspace size does not depend on how many there are). */
int64_t b200fe_workspace_bytes_ex(const b200fe_params* p, int64_t R, int64_t T, int32_t ragged);
/* The sizers of ragged calls (b200fe_workspace_bytes_ex with ragged != 0, b200fe_workspace_bytes_ragged_i16,
 * b200fe_host_staging_bytes_ragged) serve both pad modes: zero-padding stages exactly the rows repeat-padding stages. */

/* The ragged call of b200fe_features_forward with 16-bit PCM clips, what the reference's loader decodes before it turns
 * them into float32 and pad()s them (maze5.py:297-351, :280-285): every row is staged as a dense float32 row in the
 * workspace -- repeat-padded / truncated to T, converted x / 32768 (exact), pre-emphasis applied -- for either kernel
 * family, so the features are bit-identical to the float32 ragged call on the converted samples.
 *   pcm  int16 device flat clips, 2-byte aligned (a clip may start on any sample);  offsets / lengths as above (required)
 *   workspace  >= b200fe_workspace_bytes_ragged_i16(p, R, T): the ragged workspace plus one chunk of dense rows for
 *   either variant */
int64_t b200fe_workspace_bytes_ragged_i16(const b200fe_params* p, int64_t R, int64_t T);
int32_t b200fe_features_forward_ragged_i16(const int16_t* pcm, int64_t R, int64_t T, const int64_t* offsets,
                                           const int32_t* lengths, const b200fe_params* p, const void* tables,
                                           float* out, void* workspace, size_t workspace_bytes, void* stream);

/* Replaces Spectrogram.forward (transforms/_transforms.py:25; functional.py:119-145, power=2):
 *   wave  float32 device [R][T] contiguous           out  float32 device [R][n_fft/2+1][n_frames]   */
int32_t b200fe_spectrogram_forward(const float* wave, int64_t R, int64_t T, const b200fe_params* p,
                                   const void* tables, float* out, void* stream);

/* Replaces LFCC.forward (+ ComputeDeltas x deltas + cat) and MelSpectrogram.forward (+AmplitudeToDB)
 * — the call behind the feature slot maze5.py:241.
 *   wave     float32 device.  Dense mode (offsets == NULL): [R][T] contiguous.
 *            Ragged mode: flat clips; row r is samples wave[offsets[r] .. offsets[r]+lengths[r]) and is
 *            repeat-padded / truncated to T on the fly exactly like pad() at maze5.py:280-285
 *            (sample i = clip[i mod len]; clips longer than T keep their first T samples).
 *   offsets  int64 device [R] or NULL;   lengths  int32 device [R] or NULL (both or neither)
 *   out      float32 device [R][n_out_channels][n_frames] contiguous
 *   workspace  device scratch of at least b200fe_workspace_bytes_ex(p,R,T,offsets != NULL), 16-byte aligned */
int32_t b200fe_features_forward(const float* wave, int64_t R, int64_t T, const int64_t* offsets,
                                const int32_t* lengths, const b200fe_params* p, const void* tables,
                                float* out, void* workspace, size_t workspace_bytes, void* stream);

/* The ragged calls with a choice of padding: b200fe_features_forward (offsets and lengths required here) and
 * b200fe_features_forward_ragged_i16 with pad_mode (b200fe_pad_mode) after the clip table.  B200FE_PAD_REPEAT is the
 * call without the suffix; B200FE_PAD_ZERO zero-pads clips shorter than T.  The same kernels are launched and the same
 * rows staged in both modes, so the workspace sizes are those of the calls without the suffix.  A pad_mode outside
 * {0, 1} returns B200FE_ERR_BAD_ARG before any CUDA call. */
int32_t b200fe_features_forward_ragged_pad(const float* wave, int64_t R, int64_t T, const int64_t* offsets,
                                           const int32_t* lengths, int32_t pad_mode, const b200fe_params* p,
                                           const void* tables, float* out, void* workspace, size_t workspace_bytes,
                                           void* stream);
int32_t b200fe_features_forward_ragged_i16_pad(const int16_t* pcm, int64_t R, int64_t T, const int64_t* offsets,
                                               const int32_t* lengths, int32_t pad_mode, const b200fe_params* p,
                                               const void* tables, float* out, void* workspace, size_t workspace_bytes,
                                               void* stream);

/* Stage output of the same path: the filterbank energies (spec^T @ fb)^T of
 * transforms/_transforms.py:818, before log / DCT / deltas:  out float32 device [R][n_filter][n_frames].
 * This is exactly the first (dominant) kernel of b200fe_features_forward, launched alone — used by the
 * stage-wise parity tests and by bench.py to time that kernel with CUDA events. */
int32_t b200fe_fbank_energies_forward(const float* wave, int64_t R, int64_t T, const int64_t* offsets,
                                      const int32_t* lengths, const b200fe_params* p, const void* tables,
                                      float* out, void* workspace, size_t workspace_bytes, void* stream);

/* Thin aliases with the names SURVEY.md 8(b) gives (LFCC: n_coef > 0; mel: n_coef == 0). */
int32_t b200fe_lfcc_forward(const float* wave, int64_t R, int64_t T, const int64_t* offsets,
                            const int32_t* lengths, const b200fe_params* p, const void* tables,
                            float* out, void* workspace, size_t workspace_bytes, void* stream);
int32_t b200fe_mel_forward(const float* wave, int64_t R, int64_t T, const int64_t* offsets,
                           const int32_t* lengths, const b200fe_params* p, const void* tables,
                           float* out, void* workspace, size_t workspace_bytes, void* stream);

/* Replaces ComputeDeltas.forward (transforms/_transforms.py:992; functional.py:961-1008):
 *   in / out  float32 device [rows][T]; replicate padding; win odd 3..9                             */
int32_t b200fe_compute_deltas(const float* in, int64_t rows, int64_t T, int32_t win, float* out,
                              void* stream);

/* ---- host-buffer entry point (end-to-end path) ------------------------------------------------
 * Same transform with HOST waveforms and a HOST output: the library streams chunks of rows
 * host -> device -> kernels -> host through caller-provided device staging, overlapping the copies
 * of one chunk with the kernels of another on `n_streams` internal-use streams supplied by the
 * caller.  wave_host / out_host should be pinned (cudaHostAlloc / torch pin_memory) for the copies
 * to be asynchronous.  Blocks until the last chunk has landed in out_host.
 *   staging        device scratch, >= b200fe_host_staging_bytes(p, chunk_rows, T, n_streams)
 *   streams        array of n_streams cudaStream_t (as void*), 1..4                                */
int64_t b200fe_host_staging_bytes(const b200fe_params* p, int64_t chunk_rows, int64_t T, int32_t n_streams);
int32_t b200fe_features_forward_host(const float* wave_host, int64_t R, int64_t T, const b200fe_params* p,
                                     const void* tables, float* out_host, void* staging,
                                     size_t staging_bytes, int64_t chunk_rows, void* const* streams,
                                     int32_t n_streams);

/* The same with 16-bit PCM rows on the host (what ASVspoof's FLAC files decode to before the reference's loader
 * turns them into float32, maze5.py:297-351): the PCM crosses PCIe (half the bytes), a device kernel converts
 * x / 32768 — exact in float32, so the features are bit-identical to the float32 call on the converted samples.
 *   pcm_host  int16 [R][T];  staging >= b200fe_host_staging_bytes_i16(p, chunk_rows, T, n_streams)            */
int64_t b200fe_host_staging_bytes_i16(const b200fe_params* p, int64_t chunk_rows, int64_t T, int32_t n_streams);
int32_t b200fe_features_forward_host_i16(const int16_t* pcm_host, int64_t R, int64_t T, const b200fe_params* p,
                                         const void* tables, float* out_host, void* staging,
                                         size_t staging_bytes, int64_t chunk_rows, void* const* streams,
                                         int32_t n_streams);

/* Variable-length clips in HOST memory: replaces the reference's loader + pad() + batching (maze5.py:297-351,
 * :280-285) in front of the feature slot of its scoring loop (maze5.py:415-430).  Clip r is
 * clips_host[offsets_host[r] .. + lengths_host[r]) of a flat buffer of n_samples samples, int16 PCM (sample_bytes 2,
 * x / 32768) or float32 (sample_bytes 4); out_host float32 [R][n_out_channels][n_frames] as above.
 * Chunks of at most chunk_rows consecutive rows are pipelined as in b200fe_features_forward_host.  A chunk copies one
 * span of the flat buffer, from its lowest offset to its highest offset + min(length, T) (pad() reads no further), and
 * closes early when the next row would take the span past chunk_rows * (T + 16) samples; then the chunk's slice of
 * the clip table is copied, a kernel stages the rows dense (pad(), x / 32768, pre-emphasis) and the dense forward call
 * runs.  Features are bit-identical to b200fe_features_forward(_ragged_i16) on the same clips.  The clip table is
 * checked on the host before any CUDA call (every length >= 1, offset >= 0, offset + length <= n_samples:
 * B200FE_ERR_BAD_ARG naming the first bad row).  Needs top_db_group == 1.
 *   staging  >= b200fe_host_staging_bytes_ragged(p, chunk_rows, T, sample_bytes, n_streams), 256-byte aligned
 *   streams  array of n_streams cudaStream_t (as void*), 1..4                                                      */
int64_t b200fe_host_staging_bytes_ragged(const b200fe_params* p, int64_t chunk_rows, int64_t T,
                                         int32_t sample_bytes, int32_t n_streams);
int32_t b200fe_features_forward_host_ragged(const void* clips_host, int32_t sample_bytes, int64_t n_samples,
                                            const int64_t* offsets_host, const int32_t* lengths_host, int64_t R,
                                            int64_t T, const b200fe_params* p, const void* tables, float* out_host,
                                            void* staging, size_t staging_bytes, int64_t chunk_rows,
                                            void* const* streams, int32_t n_streams);
/* The same with pad_mode (b200fe_pad_mode) after the clip table; B200FE_PAD_REPEAT is the call above.  The chunks,
 * copies, launches and staging size are the same in both modes. */
int32_t b200fe_features_forward_host_ragged_pad(const void* clips_host, int32_t sample_bytes, int64_t n_samples,
                                                const int64_t* offsets_host, const int32_t* lengths_host,
                                                int32_t pad_mode, int64_t R, int64_t T, const b200fe_params* p,
                                                const void* tables, float* out_host, void* staging,
                                                size_t staging_bytes, int64_t chunk_rows, void* const* streams,
                                                int32_t n_streams);

/* ---- scoring tail on the device (SURVEY 8f-2) ---------------------------------------------------
 * Replaces the host-side  fpr, tpr, thr = sklearn.metrics.roc_curve(y, s); fnr = 1 - tpr;
 * eer = fpr[nanargmin |fnr - fpr|]; min_dcf = min(fnr + fpr)  of Thesis/02_Evaluation_Scripts/Maze5_eval.py:588-594
 * (also score_file_processor.py:176-196), with roc_curve's default drop_intermediate=True: the same three numbers,
 * digit for digit, computed in float64 from scores that never left the device.
 *   scores  float32 device [n]   per-utterance scores (maze5.py:425: log-softmax column 1)
 *   labels  int32 device [n]     1 = bonafide (positive class), anything else = spoof
 *   out4    float64 device [4]   eer, min_dcf, eer threshold, status (0 ok, 1 = only one class present: the
 *                                reference returns no metrics then, Maze5_eval.py:577-582; 2 = a score is NaN or
 *                                infinite: scikit-learn's roc_curve raises on such input)
 *   workspace  device scratch >= b200fe_eer_workspace_bytes(n), 16-byte aligned
 * One kernel on `stream`; no synchronisation (the caller reads out4 when it needs the numbers). */
int64_t b200fe_eer_workspace_bytes(int64_t n);
int32_t b200fe_eer_min_dcf(const float* scores, const int32_t* labels, int64_t n, double* out4, void* workspace,
                           size_t workspace_bytes, void* stream);

/* Number of kernel launches the last b200fe_*_forward call on this thread enqueued (bench.py's
 * gpu_launches figure is counted from this). */
int64_t b200fe_last_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* B200FE_H_ */
