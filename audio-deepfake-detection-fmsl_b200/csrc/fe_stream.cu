// Streaming tcgen05 kernel of the DFT-GEMM variant (sm_100a): waveform -> filterbank energies.
//
// The launch's rows are one stream of frames (row-major: utterance, frame); a tile = 128 consecutive stream
// frames = the 128 TMEM lanes of one M=128 MMA, whatever utterances they belong to, so every tile is full.
// One persistent CTA per SM walks tiles  blockIdx.x, blockIdx.x + gridDim.x, ...
//
// Warp roles (27 warps):
//    0-15  drain      warp = (TMEM lane quarter, run, column half): tcgen05.ld of the four accumulators, packed fp32x2
//                     powers of the run's bins (run 0: bin k, run 1: bin n_fft/2 - k) and sliding even/odd
//                     triangular-filter sums over column pairs (fe_gemm_layout.h).  A finished filter segment is the
//                     filter's final energy for the frame and goes straight to the workspace [row][filter][frame]; the
//                     four walkers of a frame meet once per tile for the segments that straddle the column halves and
//                     bin n_fft/4.  TMEM is released after the last tcgen05.ld.  (A drain warp issues about one
//                     instruction per five cycles -- dependent packed-FMA chains -- so the drain time is set by how
//                     many warps share the walk, not by the issue slots: profiles/r2_stream_v3_*.)  Behind the drain,
//                     while the tensor pipe runs the next tile, these warps scout the tile after that: max|x| per
//                     hop block straight from global memory -> s_gmax[tile parity] (which also pulls the tile's hop
//                     blocks into L2 ahead of the loader's TMA boxes).
//   16-23  producers  two groups of four warps (lane = frame).  Per tile: per-frame power-of-two scale from the
//                     scouted block maxima, then production units (stage, K half): 16 sample pairs of every frame,
//                     fold (FMUL2 / FFMA2) + scale + fp16 hi/lo split (cvt.rn.f16x2 + FHFMA residuals) into the UMMA
//                     A tiles; group = K half.  The A slots are not aliased by anything, so the first two stages of
//                     tile i+1 are produced while tile i is drained.
//   24-25  MMA        one issuing thread per sub-GEMM pair (ce, co / se, so): per stage 3 x 2 tcgen05.mma (M=128,
//                     N=n_fft/4, K=16: hi*hi + lo*hi + hi*lo) into the 4 TMEM accumulators, tcgen05.commit -> mbarriers
//   26     loader     per tile: the hop blocks the tile's frames need, once each, as a handful of TMA tensor boxes
//                     {32 floats, hop/32, 2^k hop blocks} with the 128-byte swizzle: hop blocks sit densely in shared
//                     memory and lane <-> frame reads are still conflict-free.  A small 1-D bulk copy costs the TMA
//                     unit ~90 cycles whatever its size, hence boxes.  Reflect-padded edge blocks are synthesised
//                     with plain loads; cp.async.bulk.prefetch.tensor of the next tile's boxes into L2.  Per stage:
//                     the 32 KB of DFT operand tiles.
// TMEM holds exactly the four accumulators (4 x 128 columns), so the MMAs of a tile and its drain cannot overlap;
// the tile period is MMA phase + drain, everything else (sample loads, scout, production, stores) runs beside them.
#include <atomic>
#include <stdio.h>
#include <unistd.h>

#include "fe_tc.cuh"

#include "fe_gemm.cuh"
#include "fe_gemm.h"
#include "fe_gemm_tables.h"

namespace {

constexpr int kDrainWarps = 16;       // warps 0..15: quarter = warp & 3, run = (warp >> 2) & 1, column half = warp >> 3
constexpr int kProducerWarp0 = kDrainWarps;
constexpr int kProducerGroups = 2;    // group = K half of the stage (tests/emu/fe_emu.cpp mirrors the unit -> group mapping)
constexpr int kProducerWarps = 4 * kProducerGroups;
constexpr int kProducerThreads = kProducerWarps * 32;
constexpr int kMmaWarp0 = kProducerWarp0 + kProducerWarps;   // warps 20, 21: MMA issuers, two sub-GEMMs each (ce, co / se, so)
constexpr int kNumMmaWarps = 2;
constexpr int kLoaderWarp = kMmaWarp0 + kNumMmaWarps;
constexpr int kThreads = (kLoaderWarp + 1) * 32;
constexpr int kTileM = FE_GEMM_TILE_M;
constexpr int kMaxSlots = 131;                    // hop blocks of a tile: 128 + 1 + one more per utterance boundary (at most two: fe_tile_frames)
constexpr int kAStageBytes = 8 * 2 * kTileM * 16; // 32 KB: [sub 4][hi, lo] tiles of 128 rows x 16 K
constexpr int kGmaxStride = (((kMaxSlots + 1) * 4 + 15) & ~15) / 4;   // floats per tile parity of the block maxima

struct stream_args {
  const float* wave;        // first row of the launch
  const void* tables;
  float* energies;          // [rows][n_filter][n_frames]
  unsigned int* group_max;  // or NULL
  int* error_flag;
  int64_t T;
  int64_t row_base;         // absolute index of the launch's first row (group_max indexing)
  int32_t rows, n_frames, n_filter, hop, nhalf, nstages, kpairs;
  int32_t total_frames, tile_frames, n_tiles, top_db_group;
  // ragged input read partly in place (offsets != NULL): `wave` is the tensor maps' base, clips that qualify
  // (fe_clip_in_place) are read from the flat buffer flat_rel floats above it, the others from their staged dense rows
  // dense_rel floats above it; the maps' last dimension then counts 16-byte units from the base instead of rows
  const int64_t* offsets;
  const int32_t* lengths;
  int64_t flat_rel, dense_rel;
};

// first sample of launch row `row`, in floats above a.wave
__device__ __forceinline__ int64_t row_src(const stream_args& a, int row) {
  if (!a.offsets) return (int64_t)row * a.T;
  const int64_t arow = a.row_base + row;
  const int64_t off = __ldg(a.offsets + arow);
  return fe_clip_in_place(off, __ldg(a.lengths + arow), a.T, a.flat_rel) ? a.flat_rel + off : a.dense_rel + (int64_t)row * a.T;
}

constexpr int kNumBars = 14;   // BAR_COUNT below

struct smem_layout {
  int samp, a_stage, b_stage, dw, dwn, dctl, dhdr, mid, gmax, us2, midp, exl0, exch, bars, tmem_slot, total;
};

__host__ __device__ inline smem_layout make_layout(int hop, int nhalf, int kpairs) {
  smem_layout L;
  int off = 0;
  L.samp = off;      off += kMaxSlots * hop * 4;            // dense hop-block rows, 128-byte swizzled (base 1024-aligned)
  off = (off + 127) & ~127;
  L.a_stage = off;   off += 2 * kAStageBytes;
  L.b_stage = off;   off += 2 * fe_gemm_b_stage_bytes(nhalf);
  L.dw = off;        off += 2 * (nhalf / 2) * (int)sizeof(fe_drain_w);
  L.dwn = off;       off += 2 * (nhalf / FE_DRAIN_BATCH) * 16 * 4;
  L.dctl = off;      off += (2 * (nhalf / FE_DRAIN_BATCH) * 4 + 15) & ~15;
  L.dhdr = off;      off += (int)sizeof(fe_drain_hdr);
  L.mid = off;       off += kpairs * 4;          // interleaved weights of bin n_fft/4: even j -> Re, odd j -> Im
  L.gmax = off;      off += 2 * (((kMaxSlots + 1) * 4 + 15) & ~15);   // [tile parity] max |x| per hop block of the tile
  L.us2 = off;       off += 2 * kTileM * 4;                       // [tile parity][frame] unscale^2
  L.midp = off;      off += 2 * kProducerGroups * kTileM * 8;     // [tile parity][producer group][frame] (Re, Im) partials of bin n_fft/4
  L.exl0 = off;      off += 2 * 2 * 2 * kTileM * 4;               // [tile parity][run][class][frame] half 0 -> half 1 leftovers
  L.exch = off;      off += 2 * 2 * kTileM * 4;                   // [tile parity][class][frame] run 1 -> run 0 straddler partials
  L.bars = off;      off += kNumBars * 8;
  L.tmem_slot = off; off += 16;
  L.total = off;
  return L;
}

enum { BAR_SAMP_FULL = 0, BAR_SAMP_EMPTY = 1, BAR_A_FULL = 2, BAR_B_FULL = 4, BAR_STAGE_FREE = 6, BAR_ACC_FULL = 8,
       BAR_ACC_EMPTY = 9, BAR_PROD_DONE = 10, BAR_SCOUT_FULL = 12, BAR_COUNT = 14 };
static_assert(BAR_COUNT == kNumBars, "barrier count");

#ifdef FE_GEMM_TRACE
#ifndef FE_TRACE_CTA
#define FE_TRACE_CTA 0
#endif
#ifndef FE_TRACE_IT0
#define FE_TRACE_IT0 0
#endif
#define ST_TRACE(ev, it, q) do { if (blockIdx.x == FE_TRACE_CTA && (int)(it) >= FE_TRACE_IT0 && (int)(it) < FE_TRACE_IT0 + 8) { ((long long*)(a.error_flag + 64))[(((int)(it) - FE_TRACE_IT0) * 8 + (q)) * 16 + (ev)] = clock64(); } } while (0)
#else
#define ST_TRACE(ev, it, q) do { } while (0)
#endif

// 128-byte swizzle of the sample buffer (what TMA SWIZZLE_128B does): 16-byte chunk index ^= 128-byte line index mod 8
__device__ __forceinline__ uint32_t swz(uint32_t o) { return o ^ (((o >> 7) & 7u) << 4); }

struct tmaps8 {
  CUtensorMap m[8];   // box heights 1, 2, 4, ..., 128 hop blocks
};

__device__ __forceinline__ void tma_box_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

__device__ __forceinline__ void tma_box_5d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}

__device__ __forceinline__ void tma_prefetch_5d(const CUtensorMap* map, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.prefetch.tensor.5d.L2.global [%0, {%1, %2, %3, %4, %5}];" ::"l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3),
               "r"(c4)
               : "memory");
}

__device__ __forceinline__ void tma_prefetch_4d(const CUtensorMap* map, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global [%0, {%1, %2, %3, %4}];" ::"l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}

// boxes of 2^k hop blocks starting at block `blk` of launch row `row`.  Dense rows: 4-D maps, last coordinate = row.
// Ragged input: 5-D maps whose last two dimensions count 16-byte units (2^31 of them = 32 GB) and 32 GB steps above
// the base, so that the flat clip buffer and the staged rows may lie anywhere in the device's address space.
__device__ __forceinline__ void row_box(const stream_args& a, uint32_t dst, const CUtensorMap* map, uint32_t bar, int blk, int row) {
  if (a.offsets) {
    const int64_t u = row_src(a, row) >> 2;
    tma_box_5d(dst, map, bar, 0, 0, blk, (int)(u & 0x7fffffff), (int)(u >> 31));
  } else {
    tma_box_4d(dst, map, bar, 0, 0, blk, row);
  }
}
__device__ __forceinline__ void row_prefetch(const stream_args& a, const CUtensorMap* map, int blk, int row) {
  if (a.offsets) {
    const int64_t u = row_src(a, row) >> 2;
    tma_prefetch_5d(map, 0, 0, blk, (int)(u & 0x7fffffff), (int)(u >> 31));
  } else {
    tma_prefetch_4d(map, 0, 0, blk, row);
  }
}

// max |x| of every hop block of a tile, straight from global memory, by `nwarps` warps (this one is `w`): 8 lanes per
// hop block, 4 blocks per pass, every lane's loads of a pass in flight together.  The drain warps run this one tile
// AHEAD of the sample loads, in the time they would otherwise idle behind the tile's MMAs: the per-frame scales are
// known before the samples land in shared memory (nothing of it is on the producers' path), and the tile's hop blocks
// are in L2 when the loader's TMA boxes ask for them.  Edge blocks (v = 0, v = nF: reflect padding) take the same
// element-wise path the loader uses, so the maxima are those of exactly the samples the producers will see.
__device__ __forceinline__ void scout_tile_global(const stream_args& a, int nF, int hop, const fe_tile_geo& g,
                                                  float* s_gmax, int w, int nwarps, int lane) {
  const int T = (int)a.T;
  const int r_in = lane >> 3, l8 = lane & 7;
  const int c4 = hop >> 2;                // 16-byte chunks per hop block (hop % 32 == 0: at most 64, 8 per lane)
  for (int r0 = 4 * w; r0 < g.nv; r0 += 4 * nwarps) {
    const int r = r0 + r_in;
    float mx = 0.0f;
    if (r < g.nv) {
      const int sv = g.sv0 + r;
      const int row = sv / (nF + 1), v = sv - row * (nF + 1);
      const float* x = a.wave + row_src(a, row);
      if (v > 0 && v < nF) {
        const float4* p = reinterpret_cast<const float4*>(x + (int64_t)(v - 1) * hop);
        float4 q[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          const int i = l8 + 8 * u;
          q[u] = i < c4 ? __ldg(p + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u)
          mx = fmaxf(mx, fmaxf(fmaxf(fabsf(q[u].x), fabsf(q[u].y)), fmaxf(fabsf(q[u].z), fabsf(q[u].w))));
      } else {
        for (int e = l8; e < hop; e += 8) {
          int idx = (v - 1) * hop + e;
          idx = idx < 0 ? -idx : idx;
          idx = idx >= T ? 2 * (T - 1) - idx : idx;
          mx = fmaxf(mx, fabsf(__ldg(x + idx)));
        }
      }
    }
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 1));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 2));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, 4));
    if (l8 == 0 && r < g.nv) s_gmax[r] = mx;
  }
}

__device__ __forceinline__ void quarter_bar(int quarter) { asm volatile("bar.sync %0, 128;" ::"r"(2 + quarter) : "memory"); }   // the frame quarter's four walkers
__device__ __forceinline__ void runs_bar(int quarter) { asm volatile("bar.sync %0, 64;" ::"r"(6 + quarter) : "memory"); }      // its two half-1 walkers

// a finished filter segment of the drain: final energy of (frame, filter) -> workspace (32-bit element offsets: a
// launch's energies are < 2^31 bytes, fe_stream_supported)
struct emit_store {
  float* base;        // energies of the launch
  uint32_t off;       // (row * n_filter) * n_frames + t
  uint32_t n_frames;
  int n_filter;
  bool valid;
  float us2, vmax;
  __device__ __forceinline__ void operator()(int f, float v) {
    if (valid && f < n_filter) {
      const float e = v * us2;
      base[off + (uint32_t)f * n_frames] = e;
      vmax = fmaxf(vmax, e);
    }
  }
};

// The walk of one drain thread over its columns [k_begin, k_end) (fe_gemm_layout.h).  The last batch releases the
// thread's share of TMEM right after its tcgen05.ld has landed.
template <int RUN>
__device__ __forceinline__ void drain_walk(uint32_t taddr, int nhalf, int k_begin, int k_end, const fe_drain_w* w_run,
                                           const uint32_t* ctl_run, const float* wn_run, fe_drain_state& st, emit_store& emit,
                                           uint32_t acc_empty_bar, int lane) {
  // running addresses (registers): four accumulator columns in tensor memory, the batch's tables in shared memory
  uint32_t t0 = taddr + (uint32_t)k_begin;
  const uint32_t tn = (uint32_t)nhalf;
  uint32_t w_addr = smem_u32(w_run + (k_begin >> 1));
  uint32_t ctl_addr = smem_u32(ctl_run + (k_begin >> 3));
  uint32_t wn_addr = smem_u32(wn_run + (k_begin >> 3) * 16);
  int left = (k_end - k_begin) >> 3;
#pragma unroll 1
  for (; left > 0; --left, t0 += 8, w_addr += 64, ctl_addr += 4, wn_addr += 64) {
    float ce[8], co[8], se[8], so[8];
#ifdef FE_EXP_NO_LDTM   // timing experiment: arithmetic without the tensor-memory loads
#pragma unroll
    for (int i = 0; i < 8; ++i) { ce[i] = emit.us2 + i; co[i] = emit.us2 * i; se[i] = emit.us2 - i; so[i] = emit.us2 * 0.5f * i; }
#else
    tmem_ld8(t0, ce);
    tmem_ld8(t0 + tn, co);
    tmem_ld8(t0 + 2 * tn, se);
    tmem_ld8(t0 + 3 * tn, so);
#endif
    tmem_ld_wait();
    tmem_ld_tie8(ce); tmem_ld_tie8(co); tmem_ld_tie8(se); tmem_ld_tie8(so);
    // the tables are fetched behind the wait (volatile: not hoisted above it): 16 fewer registers live across the
    // tensor-memory loads, and the other walkers of the scheduler cover the shared-memory latency
    unsigned ctl;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(ctl) : "r"(ctl_addr));
    fe_drain_w w[4];
#pragma unroll
    for (int p = 0; p < 4; ++p)
      asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(w[p].w[0][0]), "=f"(w[p].w[0][1]), "=f"(w[p].w[1][0]), "=f"(w[p].w[1][1])
                   : "r"(w_addr + 16u * p));
    if (left == 1) {
      // this walker's share of the accumulators is in registers: TMEM is free for the next tile's MMAs once all 16 say so
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(acc_empty_bar);
    }
    fe_f2 pw[4];
#ifdef FE_EXP_NO_MATH   // timing experiment: the tensor-memory loads without the arithmetic
    st.acc[0].x += ce[0] + co[1] + se[2] + so[3];
    continue;
#endif
#pragma unroll
    for (int p = 0; p < 4; ++p)
      pw[p] = fe_drain_power<RUN>(fe_f2{ce[2 * p], ce[2 * p + 1]}, fe_f2{co[2 * p], co[2 * p + 1]}, fe_f2{se[2 * p], se[2 * p + 1]},
                                  fe_f2{so[2 * p], so[2 * p + 1]});
    fe_drain_batch(pw, w, reinterpret_cast<const float*>(__cvta_shared_to_generic(wn_addr)), ctl, st, emit);
  }
}

// One production unit (stage q, K half): 16 sample pairs of frame m from the sample buffer (brow / frow: byte offsets of
// the frame's backward / forward hop block), folded, scaled and split into the UMMA A tiles of slot `a_slot` (shared
// address of the slot), then the slot's A_FULL arrival.

__device__ __forceinline__ void produce_unit(const unsigned char* s_samp, uint32_t brow, uint32_t frow, int hop, int q, int khalf,
                                             int m, float scale, const float* s_mid, float& mid_re, float& mid_im,
                                             unsigned char* a_slot, uint32_t bar_stage_free, uint32_t free_parity,
                                             uint32_t bar_a_full, int* error_flag, int lane) {
  const int j0 = 32 * q + 16 * khalf;
  float fwd[16], bwd[16], buf[16];
#pragma unroll
  for (int ch = 0; ch < 4; ++ch) {
    const float4 f = *reinterpret_cast<const float4*>(s_samp + swz(frow + j0 * 4 + ch * 16));
    fwd[4 * ch + 0] = f.x; fwd[4 * ch + 1] = f.y; fwd[4 * ch + 2] = f.z; fwd[4 * ch + 3] = f.w;
    float4 b;   // asm: keeps the 16-byte load whole even where only three of its elements are used
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
                 : "r"(smem_u32(s_samp) + swz(brow + (hop - j0 - 16) * 4 + ch * 16)));
    buf[4 * ch + 0] = b.x; buf[4 * ch + 1] = b.y; buf[4 * ch + 2] = b.z; buf[4 * ch + 3] = b.w;
  }
  // bwd[i] = x[c - j0 - i] = backward-row element hop - j0 - i; element hop (i = 0, j0 = 0) is the centre sample
  bwd[0] = (j0 == 0) ? fwd[0] : *reinterpret_cast<const float*>(s_samp + swz(brow + (hop - j0) * 4));
#pragma unroll
  for (int i = 1; i < 16; ++i) bwd[i] = buf[16 - i];
  fe_u4 chunk[8];
  fe_stream_produce_unit(fwd, bwd, scale, s_mid + j0, mid_re, mid_im, chunk);
  mbar_wait(bar_stage_free, free_parity, error_flag, 7);   // MMAs of this slot's previous use retired
  unsigned char* a_row = a_slot + khalf * kTileM * 16 + m * 16;
#pragma unroll
  for (int sf = 0; sf < 8; ++sf) *reinterpret_cast<fe_u4*>(a_row + sf * fe_gemm_tile_bytes(kTileM)) = chunk[sf];
  fence_proxy_async();
  __syncwarp();
  if (lane == 0) mbar_arrive(bar_a_full);
}

// ------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 1) fe_stream_kernel(const __grid_constant__ tmaps8 maps, const stream_args a) {
  extern __shared__ __align__(1024) unsigned char smem[];
  const smem_layout L = make_layout(a.hop, a.nhalf, a.kpairs);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const unsigned char* blob = reinterpret_cast<const unsigned char*>(a.tables);
  const fe_blob_header* h = reinterpret_cast<const fe_blob_header*>(blob);
  const int nF = a.n_frames, hop = a.hop, nfil = a.n_filter;
  const int rs = hop * 4;        // bytes per hop-block row (dense; the 128-byte swizzle keeps lane <-> frame reads conflict-free)
  const int npairs = a.nhalf / 2, nbatch = a.nhalf / FE_DRAIN_BATCH;

  if (!h->gemm_ok) {
    // tables without the variant's tiles (a C-ABI caller that set variant = DFT_GEMM without asking
    // b200fe_tables_variant): the launch must not look successful -> error flag + trap, surfaced to the caller as
    // B200FE_ERR_CUDA by the next CUDA call, like a protocol timeout
    if (tid == 0) mbar_timeout(a.error_flag, 98);
    return;
  }
  unsigned char* s_samp = smem + L.samp;
  fe_drain_w* s_dw = reinterpret_cast<fe_drain_w*>(smem + L.dw);
  uint32_t* s_dctl = reinterpret_cast<uint32_t*>(smem + L.dctl);
  float* s_dwn = reinterpret_cast<float*>(smem + L.dwn);
  fe_drain_hdr* s_dhdr = reinterpret_cast<fe_drain_hdr*>(smem + L.dhdr);
  float* s_mid = reinterpret_cast<float*>(smem + L.mid);
  float* s_gmax = reinterpret_cast<float*>(smem + L.gmax);
  float* s_us2 = reinterpret_cast<float*>(smem + L.us2);
  float2* s_midp = reinterpret_cast<float2*>(smem + L.midp);
  float* s_exl0 = reinterpret_cast<float*>(smem + L.exl0);
  float* s_exch = reinterpret_cast<float*>(smem + L.exch);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(smem + L.tmem_slot);
  const uint32_t bars = smem_u32(smem + L.bars);
  auto bar = [&](int i) { return bars + 8u * (uint32_t)i; };

  // ---- one-time setup -----------------------------------------------------------------------------
  {
    const fe_drain_w* gdw = reinterpret_cast<const fe_drain_w*>(blob + h->off_gemm_dw);
    for (int i = tid; i < 2 * npairs; i += kThreads) s_dw[i] = gdw[i];
    const uint32_t* gctl = reinterpret_cast<const uint32_t*>(blob + h->off_gemm_dctl);
    for (int i = tid; i < 2 * nbatch; i += kThreads) s_dctl[i] = gctl[i];
    const float* gwn = reinterpret_cast<const float*>(blob + h->off_gemm_dwn);
    for (int i = tid; i < 2 * nbatch * 16; i += kThreads) s_dwn[i] = gwn[i];
    const int32_t* ghdr = reinterpret_cast<const int32_t*>(blob + h->off_gemm_dids);
    for (int i = tid; i < (int)(sizeof(fe_drain_hdr) / 4); i += kThreads) reinterpret_cast<int32_t*>(s_dhdr)[i] = ghdr[i];
    const float* gmid = reinterpret_cast<const float*>(blob + h->off_gemm_mid);
    for (int i = tid; i < a.kpairs; i += kThreads) s_mid[i] = (i & 1) ? gmid[a.kpairs + i] : gmid[i];
    // rows a tile does not use are never read unpredicated, but keep the buffer defined
    float4* z = reinterpret_cast<float4*>(s_samp);
    for (int i = tid; i < kMaxSlots * rs / 16; i += kThreads) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    fence_proxy_async();
  }
  if (tid == 0) {
    mbar_init(bar(BAR_SAMP_FULL), 2);
    mbar_init(bar(BAR_SAMP_EMPTY), kProducerWarps);
    mbar_init(bar(BAR_A_FULL + 0), 8);    // a stage = two production units x four warps
    mbar_init(bar(BAR_A_FULL + 1), 8);
    mbar_init(bar(BAR_B_FULL + 0), 1);
    mbar_init(bar(BAR_B_FULL + 1), 1);
    mbar_init(bar(BAR_STAGE_FREE + 0), kNumMmaWarps);
    mbar_init(bar(BAR_STAGE_FREE + 1), kNumMmaWarps);
    mbar_init(bar(BAR_ACC_FULL), kNumMmaWarps);
    mbar_init(bar(BAR_ACC_EMPTY), kDrainWarps);
    mbar_init(bar(BAR_PROD_DONE + 0), kProducerWarps);
    mbar_init(bar(BAR_PROD_DONE + 1), kProducerWarps);
    mbar_init(bar(BAR_SCOUT_FULL + 0), kDrainWarps);
    mbar_init(bar(BAR_SCOUT_FULL + 1), kDrainWarps);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kMmaWarp0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(s_tmem)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;
  const int T = (int)a.T;
  const uint32_t b_stage_bytes = (uint32_t)fe_gemm_b_stage_bytes(a.nhalf);

  if (warp == kLoaderWarp) {
    // ================================ loader ==========================================================
    const unsigned char* gB = blob + h->off_gemm_b;
    const uint32_t row_bytes = (uint32_t)hop * 4u;
    uint32_t n = 0, it = 0;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++it) {
      const fe_tile_geo g = fe_tile_geometry(tile, a.tile_frames, a.total_frames, nF);
      mbar_wait_relaxed(bar(BAR_SAMP_EMPTY), (it & 1u) ^ 1u, a.error_flag, 1);   // producers are done with the previous tile's samples
      ST_TRACE(0, it, 0);
      int n_edge = 0;
      for (int row = g.row0; row <= g.row_last; ++row) {
        const int sa = row * (nF + 1) - g.sv0, sb = sa + nF;
        n_edge += (sa >= 0 && sa < g.nv) + (sb >= 0 && sb < g.nv);
      }
      fence_proxy_async();   // earlier generic writes of edge rows vs. the bulk copies below
      if (lane == 0) mbar_arrive_expect_tx(bar(BAR_SAMP_FULL), (uint32_t)(g.nv - n_edge) * row_bytes);
      __syncwarp();
      // per utterance segment: its ordinary hop blocks are contiguous; box heights = binary digits of their count
      for (int row = g.row0; row <= g.row_last; ++row) {
        const int v_lo = max(g.sv0 - row * (nF + 1), 1), v_hi = min(g.sv0 + g.nv - 1 - row * (nF + 1), nF - 1);
        const int cnt = v_hi - v_lo + 1;
        if (cnt <= 0) continue;
        if (lane < 8 && ((cnt >> lane) & 1)) {
          const int first = cnt & ~((2 << lane) - 1);          // blocks taken by the larger boxes
          const int s = row * (nF + 1) + v_lo + first - g.sv0;  // slot of this box's first block
          row_box(a, smem_u32(s_samp + s * rs), &maps.m[lane], bar(BAR_SAMP_FULL), v_lo - 1 + first, row);
        }
      }
      // edge blocks: v = 0 (reflect about sample 0) and v = nF (tail of the utterance + reflect about sample T-1)
      for (int row = g.row0; row <= g.row_last; ++row) {
        const float* x = a.wave + row_src(a, row);
        for (int e2 = 0; e2 < 2; ++e2) {
          const int v = e2 ? nF : 0;
          const int s = row * (nF + 1) + v - g.sv0;
          if (s < 0 || s >= g.nv) continue;
          float val[8];   // hop <= 256: at most 8 elements per lane, all loads in flight before the first store
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int e = lane + 32 * u;
            int idx = (v - 1) * hop + e;
            idx = idx < 0 ? -idx : idx;
            idx = idx >= T ? 2 * (T - 1) - idx : idx;
            val[u] = e < hop ? __ldg(x + idx) : 0.0f;
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int e = lane + 32 * u;
            if (e < hop) *reinterpret_cast<float*>(s_samp + swz((uint32_t)(s * rs + e * 4))) = val[u];
          }
        }
      }
      __syncwarp();
      if (lane == 0) ST_TRACE(9, it, 0);
      if (lane == 0) mbar_arrive(bar(BAR_SAMP_FULL));
      // the next tile's ordinary hop blocks -> L2 now, so that its boxes (issued once the producers release the sample
      // buffer) do not wait for HBM
      if (tile + (int)gridDim.x < a.n_tiles) {
        const fe_tile_geo gn = fe_tile_geometry(tile + gridDim.x, a.tile_frames, a.total_frames, nF);
        for (int row = gn.row0; row <= gn.row_last; ++row) {
          const int v_lo = max(gn.sv0 - row * (nF + 1), 1), v_hi = min(gn.sv0 + gn.nv - 1 - row * (nF + 1), nF - 1);
          const int cnt = v_hi - v_lo + 1;
          if (cnt <= 0) continue;
          if (lane < 8 && ((cnt >> lane) & 1)) {
            const int first = cnt & ~((2 << lane) - 1);
            row_prefetch(a, &maps.m[lane], v_lo - 1 + first, row);
          }
        }
      }
      if (lane == 0) {
        for (int q = 0; q < a.nstages; ++q, ++n) {
          const uint32_t s = n & 1u, par = (n >> 1) & 1u;
          mbar_wait_relaxed(bar(BAR_STAGE_FREE + s), par ^ 1u, a.error_flag, 2);   // the MMAs that read slot s have retired
          mbar_arrive_expect_tx(bar(BAR_B_FULL + s), b_stage_bytes);
          bulk_g2s(smem_u32(smem + L.b_stage + s * b_stage_bytes), gB + (size_t)q * b_stage_bytes, b_stage_bytes,
                   bar(BAR_B_FULL + s));
        }
      }
      __syncwarp();
    }
  } else if (warp >= kMmaWarp0) {
    // ================================ MMA issuers =====================================================
    // A lone thread issues one tcgen05.mma per ~100 cycles when its operands live in ordinary registers (a per-lane
    // "waterfall" around every UTCHMMA; tests/cuda/ts_probe.cu), slower than the tensor pipe retires them.  The
    // four sub-GEMMs own separate accumulators, so two warps issue two each, and everything the issuing thread
    // needs is derived from warp-uniform values under elect.sync, so the descriptors live in uniform registers.
    {
      const int sub0 = (4 / kNumMmaWarps) * __shfl_sync(0xffffffffu, warp - kMmaWarp0, 0);
      const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
      const uint32_t idesc = (1u << 4) | ((uint32_t)(a.nhalf >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
      const uint32_t b_lbo = (uint32_t)a.nhalf * 16u;
      const uint32_t smem_a = smem_u32(smem + L.a_stage), smem_b = smem_u32(smem + L.b_stage);
      const uint32_t tile_bytes_a = fe_gemm_tile_bytes(kTileM), tile_bytes_b = fe_gemm_tile_bytes(a.nhalf);
      uint32_t n = 0, it = 0;
      for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++it) {
        mbar_wait_relaxed(bar(BAR_ACC_EMPTY), (it & 1u) ^ 1u, a.error_flag, 3);   // previous tile's accumulators read
        tc_fence_after();
        if (sub0 == 0 && lane == 0) ST_TRACE(8, it, 0);
        for (int q = 0; q < a.nstages; ++q, ++n) {
          const uint32_t s = n & 1u, par = (n >> 1) & 1u;
          mbar_wait_relaxed(bar(BAR_B_FULL + s), par, a.error_flag, 4);
          if (sub0 == 0 && lane == 0) ST_TRACE(10, it, q);
          mbar_wait_relaxed(bar(BAR_A_FULL + s), par, a.error_flag, 5);
          tc_fence_after();
          if (sub0 == 0 && lane == 0) ST_TRACE(3, it, q);
          const uint32_t a_base = smem_a + s * kAStageBytes;
          const uint32_t b_base = smem_b + s * b_stage_bytes;
          if (elect_one()) {
            // this warp's sub-GEMMs: A_hi B_hi + A_lo B_hi + A_hi B_lo, alternating accumulators
#ifdef FE_EXP_TWO_PRODUCTS   // timing experiment: two of the three split-fp16 products (results wrong: what the tensor work costs)
            constexpr int kProducts = 2;
#else
            constexpr int kProducts = 3;
#endif
#pragma unroll
            for (int pr = 0; pr < kProducts; ++pr) {
#pragma unroll
              for (int ds = 0; ds < 4 / kNumMmaWarps; ++ds) {
                const int sub = sub0 + ds;
                const uint64_t da = make_desc(a_base + (2 * sub + (pr == 1 ? 1 : 0)) * tile_bytes_a, kTileM * 16, 128);
                const uint64_t db = make_desc(b_base + (2 * sub + (pr == 2 ? 1 : 0)) * tile_bytes_b, b_lbo, 128);
                umma_f16(tmem_u + (uint32_t)(sub * a.nhalf), da, db, idesc, (q > 0 || pr > 0) ? 1u : 0u);
              }
            }
            umma_commit(bar(BAR_STAGE_FREE + s));
            if (q == a.nstages - 1) umma_commit(bar(BAR_ACC_FULL));
          }
          __syncwarp();
        }
      }
    }
  } else if (warp >= kProducerWarp0) {
    // ================================ producers (warps 8..19) =========================================
    const int pw = warp - kProducerWarp0;
    const int grp = pw >> 2;               // production units (stage, K half = grp)
    const int quarter = pw & 3;
    const int m = quarter * 32 + lane;
    uint32_t n0 = 0, it = 0;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++it, n0 += (uint32_t)a.nstages) {
      const fe_tile_geo g = fe_tile_geometry(tile, a.tile_frames, a.total_frames, nF);
      const int mm = min(m, g.count - 1);                 // rows past the end of the stream repeat the last frame
      const int row = (g.g0 + mm) / nF;
      const int slot = mm + (row - g.row0);               // backward hop block; the forward one is slot + 1
      const uint32_t tp = it & 1u;
      // the drain warps have scouted this tile's hop blocks (max |x| each) one tile ahead, from global memory
      mbar_wait(bar(BAR_SCOUT_FULL + tp), (it >> 1) & 1u, a.error_flag, 10);
      float scale, unscale;
      {
        const float* gm = s_gmax + tp * kGmaxStride;
        fe_gemm_frame_scale(2.0f * fmaxf(gm[slot], gm[slot + 1]), scale, unscale);
      }
      mbar_wait(bar(BAR_SAMP_FULL), tp, a.error_flag, 6);
      if (tid == kProducerWarp0 * 32) ST_TRACE(1, it, 0);
      if (grp == 0) s_us2[tp * kTileM + m] = unscale * unscale;
      const uint32_t brow = (uint32_t)(slot * rs), frow = brow + (uint32_t)rs;   // byte offsets into the sample buffer
      float mid_re = 0.0f, mid_im = 0.0f;
#pragma unroll 1
      for (int q = 0; q < a.nstages; ++q) {
        const uint32_t n = n0 + (uint32_t)q, sl = n & 1u, par = (n >> 1) & 1u;
        produce_unit(s_samp, brow, frow, hop, q, grp, m, scale, s_mid, mid_re, mid_im, smem + L.a_stage + sl * kAStageBytes,
                     bar(BAR_STAGE_FREE + sl), par ^ 1u, bar(BAR_A_FULL + sl), a.error_flag, lane);
        if (lane == 0 && quarter == 0) ST_TRACE(2, it, q);
      }
      // each group files its own partial of bin n_fft/4 (fixed unit -> group mapping: the sum does not depend on the tile)
      s_midp[(tp * kProducerGroups + grp) * kTileM + m] = make_float2(mid_re, mid_im);
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(bar(BAR_SAMP_EMPTY));
        mbar_arrive(bar(BAR_PROD_DONE + tp));
      }
    }
  } else {
    // ================================ drain (warps 0..15) =============================================
    const int quarter = warp & 3;          // TMEM lane quarter
    const int run = (warp >> 2) & 1;       // 0: bins k (ascending) + bin n_fft/4, 1: bins n_fft/2 - k
    const int half = warp >> 3;            // columns [half * n_fft/8, (half + 1) * n_fft/8)
    const int m = quarter * 32 + lane;
    const fe_drain_w* w_run = s_dw + run * npairs;
    const uint32_t* ctl_run = s_dctl + run * nbatch;
    const float* wn_run = s_dwn + run * nbatch * 16;
    const uint32_t tbase = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const int k_begin = half * (a.nhalf >> 1), k_end = k_begin + (a.nhalf >> 1);
    // block maxima of this CTA's first two tiles (afterwards: tile i + 2 behind the drain of tile i)
    for (int pre = 0; pre < 2; ++pre) {
      const int tile = blockIdx.x + pre * gridDim.x;
      if (tile < a.n_tiles) {
        const fe_tile_geo g = fe_tile_geometry(tile, a.tile_frames, a.total_frames, nF);
        scout_tile_global(a, nF, hop, g, s_gmax + pre * kGmaxStride, warp, kDrainWarps, lane);
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(BAR_SCOUT_FULL + pre));
    }
    uint32_t it = 0;
    for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++it) {
      const fe_tile_geo g = fe_tile_geometry(tile, a.tile_frames, a.total_frames, nF);
      const int mm = min(m, g.count - 1);
      const int row = (g.g0 + mm) / nF;
      const int t = (g.g0 + mm) - row * nF;
      const uint32_t tp = it & 1u;
      // the producers' per-frame values of this tile (scale, bin n_fft/4 partials)
      mbar_wait(bar(BAR_PROD_DONE + tp), (it >> 1) & 1u, a.error_flag, 9);
      emit_store emit;
      emit.base = a.energies;
      emit.off = (uint32_t)((row * nfil) * nF + t);
      emit.n_frames = (uint32_t)nF;
      emit.n_filter = nfil;
      emit.valid = m < g.count;
      emit.us2 = s_us2[tp * kTileM + m];
      emit.vmax = 0.0f;
      float p_mid = 0.0f;
      if (run == 0 && half == 1) {
        const float2 v0 = s_midp[(tp * kProducerGroups + 0) * kTileM + m], v1 = s_midp[(tp * kProducerGroups + 1) * kTileM + m];
        const float bs = (float)(1 << FE_GEMM_B_SCALE_LOG2);   // scaled sample units -> accumulator units
        const float re = (v0.x + v1.x) * bs, im = (v0.y + v1.y) * bs;
        p_mid = fmaf(re, re, im * im);
      }
      fe_drain_state st;
      fe_drain_init(st, *s_dhdr, run, half);
      mbar_wait(bar(BAR_ACC_FULL), tp, a.error_flag, 8);
      tc_fence_after();
      if (lane == 0 && quarter == 0) ST_TRACE(4, it, warp >> 2);
      if (run == 0) drain_walk<0>(tbase, a.nhalf, k_begin, k_end, w_run, ctl_run, wn_run, st, emit, bar(BAR_ACC_EMPTY), lane);
      else drain_walk<1>(tbase, a.nhalf, k_begin, k_end, w_run, ctl_run, wn_run, st, emit, bar(BAR_ACC_EMPTY), lane);
      if (lane == 0 && quarter == 0) ST_TRACE(5, it, warp >> 2);
      // the segments that straddle the column halves, then the runs' leftovers = the filters that straddle bin n_fft/4
      float* l0p = s_exl0 + ((tp * 2 + run) * 2) * kTileM + m;   // [class] stride kTileM
      if (half == 0) {
        l0p[0] = fe_drain_leftover(st, 0, 0.0f, 0.0f);
        l0p[kTileM] = fe_drain_leftover(st, 1, 0.0f, 0.0f);
        quarter_bar(quarter);
      } else {
        quarter_bar(quarter);
        const float l0[2] = {l0p[0], l0p[kTileM]};
        float left[2];
        fe_drain_join_halves(st, *s_dhdr, run, l0, p_mid, left, emit);
        float* ex = s_exch + tp * 2 * kTileM + m;
        if (run == 1) {
          if (s_dhdr->merge[0]) ex[0] = left[0]; else emit(s_dhdr->last[1][0], left[0]);
          if (s_dhdr->merge[1]) ex[kTileM] = left[1]; else emit(s_dhdr->last[1][1], left[1]);
          runs_bar(quarter);
        } else {
          runs_bar(quarter);
          emit(s_dhdr->last[0][0], s_dhdr->merge[0] ? left[0] + ex[0] : left[0]);
          emit(s_dhdr->last[0][1], s_dhdr->merge[1] ? left[1] + ex[kTileM] : left[1]);
        }
      }
      if (a.group_max) {
        const int grp_id = (int)((a.row_base + row) / a.top_db_group);
        const int grp0 = __shfl_sync(0xffffffffu, grp_id, 0);
        if (__all_sync(0xffffffffu, grp_id == grp0)) {
          // energies are >= 0: the unsigned order of the bit patterns is the float order, one REDUX does the warp
          const unsigned wmax = __reduce_max_sync(0xffffffffu, __float_as_uint(emit.vmax));
          if (lane == 0) atomicMax(a.group_max + grp0, wmax);
        } else if (emit.valid) {
          atomicMax(a.group_max + grp_id, __float_as_uint(emit.vmax));
        }
      }
      if (lane == 0 && quarter == 0) ST_TRACE(6, it, warp >> 2);
      // the block maxima two tiles ahead (the producers finished reading this parity's maxima long before this tile's
      // MMAs ended)
      {
        const int tile2 = tile + 2 * (int)gridDim.x;
        if (tile2 < a.n_tiles) {
          const fe_tile_geo g2 = fe_tile_geometry(tile2, a.tile_frames, a.total_frames, nF);
          scout_tile_global(a, nF, hop, g2, s_gmax + tp * kGmaxStride, warp, kDrainWarps, lane);
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(BAR_SCOUT_FULL + tp));
        if (lane == 0 && quarter == 0) ST_TRACE(7, it, warp >> 2);
      }
    }
  }

  // ---- teardown -------------------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (warp == kMmaWarp0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

typedef CUresult (*encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

encode_tiled_fn get_encode() {
  static std::atomic<encode_tiled_fn> cached{nullptr};
  encode_tiled_fn fn = cached.load(std::memory_order_relaxed);
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess) {
      fn = (encode_tiled_fn)p;
      cached.store(fn, std::memory_order_relaxed);
    }
  }
  return fn;
}

}  // namespace

#ifdef FE_GEMM_TRACE
int* fe_trace_host_flag = nullptr;
#endif
int32_t fe_gemm_compiled(void) { return 1; }

bool fe_gemm_supported(const b200fe_params* p) {
  if (p->n_filter < 1 || p->n_filter > FE_GEMM_MAX_FILTERS) return false;
  if (p->win_length != 2 * p->hop_length || p->win_length > p->n_fft) return false;
  const int kpairs = p->win_length / 2, nhalf = p->n_fft / 4;
  if (kpairs % 32 != 0 || kpairs < 32 || kpairs > 256) return false;
  if (nhalf % 16 != 0 || nhalf < 32 || nhalf > 128) return false;   // 4 accumulators fit TMEM; two column halves of whole batches
  return make_layout(p->hop_length, nhalf, kpairs).total <= 227 * 1024;
}

bool fe_gemm_preferred(const b200fe_params* p) {
  (void)p;
  // measured on B200 (profiles/): the tensor-core variant is several times faster than the FFT variant on the
  // LFCC configuration, so AUTO takes it wherever it is supported
  return true;
}
bool fe_gemm_variant_built(void) { return true; }
bool fe_gemm_auto_prefers(const b200fe_params* p) { return fe_gemm_supported(p) && fe_gemm_preferred(p); }

int64_t fe_gemm_workspace_bytes(const b200fe_params* p, int64_t chunk_rows, int64_t T) {
  (void)p; (void)chunk_rows; (void)T;
  return 65536;  // error flag (+ trace buffer in FE_GEMM_TRACE builds)
}

bool fe_stream_supported(const b200fe_params* p, int64_t T, int64_t rows) {
  if (!fe_gemm_supported(p)) return false;
  const int64_t nF = 1 + T / p->hop_length;
  if (nF < 2 || rows * nF >= (int64_t)1 << 30 || rows * nF * p->n_filter >= (int64_t)1 << 31) return false;   // 32-bit element offsets
  if (T <= p->n_fft / 2 || (T & 3) != 0) return false;
  return true;
}

cudaError_t fe_stream_launch(const b200fe_params* p, const fe_fft_args& fa, int64_t row_base, int64_t rows,
                             void* gemm_ws, cudaStream_t stream, int* launches) {
  *launches = 0;
  stream_args a;
  const bool in_place = fa.in_place != 0 && fa.wave_chunk && fa.offsets && fa.lengths;
  a.wave = in_place ? fa.wave : (fa.wave_chunk ? fa.wave_chunk : fa.wave + row_base * fa.T);
  a.offsets = in_place ? fa.offsets : nullptr;
  a.lengths = in_place ? fa.lengths : nullptr;
  a.flat_rel = in_place ? fa.flat_rel : -1;
  a.dense_rel = in_place ? fa.dense_rel : 0;
  a.tables = fa.tables;
  a.energies = fa.out;
  a.group_max = fa.group_max;
  a.error_flag = (int*)gemm_ws;
  a.T = fa.T;
  a.row_base = row_base;
  a.rows = (int32_t)rows;
  a.n_frames = fa.n_frames;
  a.n_filter = p->n_filter;
  a.hop = p->hop_length;
  a.nhalf = p->n_fft / 4;
  a.kpairs = p->win_length / 2;
  a.nstages = a.kpairs / 32;
  a.total_frames = (int32_t)(rows * fa.n_frames);
  a.tile_frames = fe_tile_frames(fa.n_frames);
  a.n_tiles = (a.total_frames + a.tile_frames - 1) / a.tile_frames;
  a.top_db_group = fa.top_db_group;

  // 4-D tensor maps over the launch's rows: {32 floats, hop/32, ordinary hop blocks of a row, rows}, boxes of 2^k blocks.
  // Encoding the eight maps costs several microseconds of host time -- a quarter of a small-batch call -- and a
  // caller that reuses its buffers (the evaluation loop, a captured graph's eager warm-up, bench.py) asks for the same
  // maps again and again: a small per-thread cache keyed by what the encoding depends on (no locks, re-entrant).
  struct map_key {
    const void* base;
    int64_t rows, T;
    int32_t hop, n_frames;
    bool ragged;
    bool operator==(const map_key& o) const { return base == o.base && rows == o.rows && T == o.T && hop == o.hop && n_frames == o.n_frames && ragged == o.ragged; }
  };
  struct map_entry { map_key key; tmaps8 maps; bool valid; };
  constexpr int kMapCache = 8;
  thread_local map_entry cache[kMapCache];
  thread_local int cache_next = 0;
  const map_key key{(const void*)a.wave, rows, fa.T, a.hop, fa.n_frames, in_place};
  const tmaps8* maps_p = nullptr;
  for (int i = 0; i < kMapCache; ++i)
    if (cache[i].valid && cache[i].key == key) { maps_p = &cache[i].maps; break; }
  if (!maps_p) {
    encode_tiled_fn enc = get_encode();
    if (!enc) return cudaErrorNotSupported;
    map_entry& e = cache[cache_next];
    cache_next = (cache_next + 1) % kMapCache;
    e.valid = false;
    // ragged input: rows start anywhere (in 16-byte steps) above the base: the last two dimensions count those steps
    // (2^31 per 32 GB) and the 32 GB strides (32 of them: 1 TB of reach, beyond any device's memory)
    const cuuint64_t gdim[5] = {32, (cuuint64_t)(a.hop / 32), (cuuint64_t)(fa.n_frames - 1), in_place ? (cuuint64_t)1 << 31 : (cuuint64_t)rows, 32};
    const cuuint64_t gstride[4] = {128, (cuuint64_t)a.hop * 4, in_place ? (cuuint64_t)16 : (cuuint64_t)fa.T * 4, (cuuint64_t)1 << 35};
    const cuuint32_t estride[5] = {1, 1, 1, 1, 1};
    for (int k = 0; k < 8; ++k) {
      const cuuint32_t box[5] = {32, (cuuint32_t)(a.hop / 32), 1u << k, 1, 1};
      CUresult r = enc(&e.maps.m[k], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, in_place ? 5 : 4, (void*)a.wave, gdim, gstride, box, estride,
                       CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                       CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      if (r != CUDA_SUCCESS) return cudaErrorInvalidValue;
    }
    e.key = key;
    e.valid = true;
    maps_p = &e.maps;
  }
  const int smem = make_layout(a.hop, a.nhalf, a.kpairs).total;
  if (smem > 227 * 1024) return cudaErrorInvalidConfiguration;
  const int dev = fe_current_device();
  if (dev < 0) return cudaErrorInvalidDevice;
  {
    cudaError_t e = fe_ensure_smem((const void*)fe_stream_kernel, (size_t)smem);
    if (e != cudaSuccess) return e;
  }
  const int sms = fe_device_sms(dev);
  const int grid = a.n_tiles < sms ? a.n_tiles : sms;
#ifdef FE_GEMM_TRACE
  {   // debug build: a host-mapped copy of the timeout flag, printed by the process at exit
    static int* host_flag = nullptr;
    extern int* fe_trace_host_flag;
    if (!host_flag) {
      cudaHostAlloc((void**)&host_flag, 256, cudaHostAllocMapped);
      for (int i = 0; i < 64; ++i) host_flag[i] = 0;
      int* dptr = nullptr;
      cudaHostGetDevicePointer((void**)&dptr, host_flag, 0);
      cudaMemcpyToSymbol(g_fe_host_flag, &dptr, sizeof(dptr));
      fe_trace_host_flag = host_flag;
      static struct printer { int* p; ~printer() { fprintf(stderr, "fe_stream timeout codes per warp (code*100000+cta):"); for (int i = 0; i < kThreads / 32; ++i) fprintf(stderr, " w%d:%d", i, p[i]); fprintf(stderr, "\n"); } } pr{host_flag};
    }
  }
  cudaError_t e = cudaMemsetAsync(a.error_flag, 0, 65536, stream);
#else
  cudaError_t e = cudaMemsetAsync(a.error_flag, 0, 4, stream);
#endif
  if (e != cudaSuccess) return e;
  fe_stream_kernel<<<grid, kThreads, smem, stream>>>(*maps_p, a);
  *launches = 1;
  return cudaGetLastError();
}
