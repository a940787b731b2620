// Masked implicit-GEMM convolution / linear for sm_100a: TMA (tiled + im2col) -> 128B-swizzled
// shared memory -> tcgen05.mma (bf16 x bf16 -> fp32 in TMEM) -> tcgen05.ld epilogue.
//
// Replaces F.conv2d / F.linear / F.conv1d(k=1) on the masked weight and their autograd
// backward (utils/mask_layers.py:26-34, :70, :110-118 of the reference).  The mask never
// appears here as a separate pass: fprop/dgrad consume bf16 weights that were masked while
// being staged (tp_stage_weights), wgrad applies the mask in its finalize step.
//
// Two persistent, warp-specialised kernels (1 CTA / SM):
//   warp 0     : TMA producer (one elected lane)
//   warp 1     : TMEM allocator + tcgen05.mma issuer (one elected lane)
//   warps 2..  : epilogue (TMEM -> registers -> global).  fprop / dgrad: 320 threads, 8 epilogue warps, two per TMEM
//                lane quarter; wgrad: 192 threads, 4 epilogue warps, one per quarter
//
//   k_igemm_fwd  : D[pixels, Cout] = A[pixels, K] * W[Cout, K]^T          (fprop, dgrad)
//                  A tile 128 pixels x 64 channels by TMA im2col (any r,s,stride,pad) or by
//                  a plain 2-D TMA box (1x1/s1 convs, linear); both K-major, SWIZZLE_128B.
//   k_igemm_wgrad: D[Cout, (tap,cin)] = dY^T[Cout, pixels] * Xcol[pixels, (tap,cin)]
//                  contraction over pixels: both operands MN-major, SWIZZLE_128B; split-K
//                  partials in fp32, summed in fixed order + masked + permuted to OIHW by
//                  k_wgrad_finalize (deterministic, no atomics).
#include "tp_common.cuh"
#include "tp_ptx.cuh"
#include <cuda.h>
#include <mutex>

namespace tp {
using namespace ptx;

constexpr int kBlockM = 128;         // UMMA M
constexpr int kBlockK = 64;          // 64 bf16 = 128 B = one swizzle row
constexpr int kThreads = 192;          // wgrad kernel: TMA warp, MMA warp, 4 epilogue warps
constexpr int kFwdThreads = 320;       // fwd kernel: TMA warp, MMA warp, 8 epilogue warps (two per TMEM lane quarter)
constexpr int kMaxTaps = 64;

// smem pipeline depth of the fwd kernel: stage = A tile (16 KB) + weight tile (block_n x 64 bf16)
__host__ __device__ constexpr int fwd_stages(int block_n) {
  return block_n == 256 ? 4 : (block_n == 128 ? 6 : 8);
}

struct TapEntry { uint16_t off_w, off_h; int32_t kofs; };

constexpr int kMaxCls = 4;

// One "class" of output pixels.  fprop and stride-1 dgrad have a single class (every output pixel, every tap).  The
// dgrad of a strided convolution splits dX into stride_h x stride_w parity classes: class (a, b) = the input pixels
// (stride*h' + a, stride*w' + b), each a stride-1 gather over dY with its own subset of taps (possibly none: those
// pixels only receive the fused addend, or zero).  All classes run in ONE launch: a work item is (class, M tile, N tile).
struct ClsEntry {
  int M;                    // iteration pixels of this class (n_img * P_it * Q_it)
  int P_it, Q_it;           // iteration grid per image
  int ntaps, tap0;          // taps[tap0 .. tap0 + ntaps)
  int base_w, base_h;       // im2col coordinate of iteration pixel (p,q): base + q*step
  int oah, oaw;             // output pixel = (p*osh + oah, q*osw + oaw)
  int tile0, m_tiles;       // first work item of the class; 128-pixel M tiles it has
};

struct FwdParams {
  int M, N;                 // iteration pixels (all classes), output channels
  int ncls;
  ClsEntry cls[kMaxCls];
  int cchunks;              // K loop = ntaps x cchunks blocks of 64 channels
  int a_mode;               // 0: tiled 2-D A[M, K];  1: im2col 4-D
  int step_w, step_h;
  long long out_img_pix;    // output pixels per image
  int out_row_pix;          // output pixels per row
  int osh, osw;
  int linear;               // output pixel index == iteration pixel index (single class, unit output stride)
  int ldc;                  // elements between consecutive output pixels
  int staged_store;         // 1 (16-byte aligned rows): the epilogue stages 32x64 sub-tiles in smem, then stores full lines
  __nv_bfloat16* out;
  const float* bias;
  const __nv_bfloat16* addend;   // optional: out = acc (+ bias) + addend[pixel][channel] (same layout as out)
  float* stats;                  // optional (linear output only): per-channel sum / sum of squares of the bf16 outputs
                                 // of every 32-row group, [ceil(M/128)*4][2][N] fp32 — BatchNorm statistics without
                                 // another pass over the activation (SURVEY.md §8(f) row 1)
  // BNB instantiation (dgrad whose output is the gradient of a BatchNorm+ReLU output, no residual): the epilogue turns dz into
  // g = dz * [y*scale + shift > 0] (the forward's own ReLU decision) and accumulates the BatchNorm backward sums of g
  const __nv_bfloat16* bn_y;     // the BatchNorm INPUT y (same layout as out)
  const float* bn_weight; const float* bn_bias; const float* bn_mean; const float* bn_invstd;   // per channel (weight / bias may be NULL)
  const uint32_t* kmask;         // optional K-block occupancy of the weight operand: [ceil(N/64)][kmask_words] bitmasks over
  int kmask_words;               // 64-column K blocks (tp_stage_weights); empty blocks are neither loaded nor multiplied
  TapEntry taps[kMaxTaps];
};

// The staging call leaves the number of empty blocks behind the last mask row: zero (any iid unstructured mask) means
// the K loop needs no per-block test at all.
__device__ __forceinline__ const uint32_t* live_kmask(const uint32_t* km, int words, int N) {
  if (km && __ldg(km + (size_t)((N + 63) >> 6) * words) == 0u) return nullptr;
  return km;
}

// Which K blocks of an output-channel tile hold any non-zero weight: the OR of the occupancy words of the tile's 64-row
// groups.  Producer and MMA thread walk the K loop with one of these each and must take identical decisions: a block is
// processed when its bit is set, or when it is the last one and nothing was processed yet (the accumulator must be
// written at least once).
struct KSkip {
  const uint32_t* base; int words, g0, g1; int cur_w; uint32_t bits;
  __device__ __forceinline__ void begin(const uint32_t* km, int wds, int n0, int block_n, int N) {
    base = km; words = wds; cur_w = -1; bits = 0u;
    g0 = n0 >> 6; g1 = min((min(n0 + block_n, N) + 63) >> 6, ((N + 63) >> 6));
  }
  __device__ __forceinline__ bool on(int kb) {
    const int wi = kb >> 5;
    if (wi != cur_w) {
      cur_w = wi; bits = 0u;
      if (wi < words) for (int g = g0; g < g1; ++g) bits |= __ldg(base + (size_t)g * words + wi);
      else bits = 0xffffffffu;                    // a block outside the mask (never produced by the staging kernels): dense
    }
    return (bits >> (kb & 31)) & 1u;
  }
};

struct WgParams {
  int Mc;                   // Cout
  int Kpix;                 // contraction length = n_img * P_it * Q_it (dY pixels)
  int P_it, Q_it;
  int chunks, cchunks;      // N axis = chunks of 64 K-columns; chunk -> (tap = chunk / cchunks, cc = chunk % cchunks)
  int nb;                   // chunks per N tile (1..4)
  int b_mode;               // 0: tiled 2-D Xcol[pixels, Kcols];  1: im2col over X
  int base_w, base_h, step_w, step_h;
  int m_tiles, n_tiles, splits, kb_per_split, kblocks;
  float* partial;           // [m_tiles*n_tiles*splits][128][nb*64]
  const uint32_t* kmask;    // optional: the fprop occupancy mask of this layer's weights ([ceil(Cout/64)][kmask_words] bits over
  int kmask_words;          // 64-column blocks of (tap, cin)): an output tile whose blocks are all masked out is not computed
  TapEntry taps[kMaxTaps];
};

// wgrad work item (128 output channels x nvalid 64-column chunks): true when every 64x64 block of it is empty in the
// occupancy mask, i.e. every mask entry under it is zero (tp_stage_weights marks a block occupied as soon as one mask
// entry is non-zero) — dW = mask * (...) is zero there whatever the activations are.
__device__ __forceinline__ bool wg_item_empty(const uint32_t* __restrict__ km, int words, int row_groups, int m_t,
                                              int chunk0, int nvalid) {
  for (int r = 2 * m_t; r < 2 * m_t + 2 && r < row_groups; ++r)
    for (int c = chunk0; c < chunk0 + nvalid; ++c)
      if ((__ldg(km + (size_t)r * words + (c >> 5)) >> (c & 31)) & 1u) return false;
  return true;
}

__device__ __forceinline__ void decompose_pixel(int m, int P, int Q, int& n, int& p, int& q) {
  q = m % Q; int t = m / Q; p = t % P; n = t / P;
}

// ============================================================================================
struct AMaps { CUtensorMap m[kMaxCls]; };      // activation-side tensor map of every class

// work item -> (class, M tile, N tile); identical in the three roles
__device__ __forceinline__ void decode_tile(const FwdParams& p, int tile, int n_tiles, int& c, int& m_t, int& n_t) {
  c = 0;
#pragma unroll
  for (int j = 1; j < kMaxCls; ++j) if (j < p.ncls && tile >= p.cls[j].tile0) c = j;
  const int local = tile - p.cls[c].tile0;
  m_t = local / n_tiles; n_t = local - m_t * n_tiles;     // m-major: CTAs running together share A tiles, weights stay in L2
}

// One CTA per 128 x BLOCK_N tile, one walk over the K blocks.  A CTA-pair walk (two M tiles per UMMA, half the weight
// tile per CTA) and a weight-stationary walk (a CTA keeps one N tile's weight blocks in smem) were built and measured
// neutral-to-slower: the weight bytes crossing L2 -> SM do not pace these layers (profiles/r01_notes.md, r02_notes.md).
//
// MULTI = false: one class of output pixels (fprop, stride-1 dgrad) — the class decode, the per-row destination
// arithmetic and the "class without taps" handling are compiled out (they cost the short-K layers up to 1.7x when they
// sat in the common kernel: 1600 more instructions around loops that run once per 2-4 us tile).
//
// BNB = true (single class, linear output): the BatchNorm backward reduction of the layer that FEEDS this convolution is
// done here, in the dgrad epilogue, instead of by k_bn_bwd_reduce (one read of dz and one of y per such layer less, one
// launch less): after the bf16 gradient sub-tile has been staged, each lane re-reads it row-coalesced together with the
// matching y values, applies the ReLU gate, stores g and adds sum(g), sum(g * xhat) of its 8 channels x 8 rows; rows are
// then combined by the same fixed-order xor tree as the forward statistics.  Output: g, and [32-row group][2][N] partials.
template <int BLOCK_N, bool MULTI, bool BNB>
__global__ void __launch_bounds__(kFwdThreads, 1)
k_igemm_fwd(const __grid_constant__ AMaps tmA, const __grid_constant__ CUtensorMap tmB,
            const __grid_constant__ FwdParams p) {
  static_assert(!BNB || !MULTI, "BatchNorm-backward epilogue: single class");
  constexpr int kABytes = kBlockM * kBlockK * 2;           // 16 KB
  constexpr int kBBytes = BLOCK_N * kBlockK * 2;
  constexpr int kStageBytes = kABytes + kBBytes;
  constexpr int kStages = fwd_stages(BLOCK_N);
  constexpr int kAccStages = BLOCK_N == 256 ? 2 : 4;      // TMEM accumulator ring (512 columns at most)
  constexpr uint32_t kTmemCols = (kAccStages * BLOCK_N <= 32) ? 32 : (kAccStages * BLOCK_N <= 64) ? 64 :
                                 (kAccStages * BLOCK_N <= 128) ? 128 : (kAccStages * BLOCK_N <= 256) ? 256 : 512;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  pdl_trigger();
  constexpr int kStgBytes = 32 * 128;                      // one epilogue warp's 32 rows x 64 bf16 columns
  uint8_t* stg_base = smem + kStages * kStageBytes;        // 8 warps x 4 KB (1024-B aligned)
  uint64_t* full_bar = (uint64_t*)(stg_base + 8 * kStgBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tfull_bar = empty_bar + kStages;
  uint64_t* tempty_bar = tfull_bar + kAccStages;
  uint32_t* tmem_slot = (uint32_t*)(tempty_bar + kAccStages);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_tiles = (p.N + BLOCK_N - 1) / BLOCK_N;
  // work items: (class) x (M tile) x (N tile), classes back to back; CTA b takes items b, b + gridDim.x, ...
  const int cta = (int)blockIdx.x, n_cta = (int)gridDim.x;
  const int total_tiles = p.cls[p.ncls - 1].tile0 + p.cls[p.ncls - 1].m_tiles * n_tiles;
  const int my_items = total_tiles > cta ? (total_tiles - cta + n_cta - 1) / n_cta : 0;
  auto get_tile = [&](int w, int& ci, int& m_t, int& n_t) {
    ci = 0;
    const int tile = cta + w * n_cta;
    if (MULTI) decode_tile(p, tile, n_tiles, ci, m_t, n_t);
    else { m_t = tile / n_tiles; n_t = tile - m_t * n_tiles; }   // m-major: CTAs running together share A tiles, weights stay in L2
  };

  if (warp == 0 && lane == 0) {
    for (int j = 0; j < p.ncls; ++j) prefetch_tmap(&tmA.m[j]);
    prefetch_tmap(&tmB);
    for (int i = 0; i < kStages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    // tempty: one arrival per epilogue warp
    for (int i = 0; i < kAccStages; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 8); }
    fence_mbar_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, kTmemCols); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();          // barriers, TMEM and descriptor prefetch above overlap the previous grid's tail; global memory from here on

  if (warp == 0) {
    // ------------------------------ TMA producer ------------------------------
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      const uint32_t* const km = live_kmask(p.kmask, p.kmask_words, p.N);
      for (int w = 0; w < my_items; ++w) {
        int ci, m_t, n_t; get_tile(w, ci, m_t, n_t);
        const ClsEntry& ce = p.cls[MULTI ? ci : 0];
        const CUtensorMap* const mapA = &tmA.m[MULTI ? ci : 0];
        const int m0 = m_t * kBlockM;
        int cn = 0, cp = 0, cq = 0;
        if (p.a_mode == 1) decompose_pixel(m0, ce.P_it, ce.Q_it, cn, cp, cq);
        const int cw = ce.base_w + cq * p.step_w, ch = ce.base_h + cp * p.step_h;
        auto load_block = [&](const TapEntry& te, int cc) {
          mbar_wait(&empty_bar[stage], phase ^ 1, 1);
          uint8_t* sA = smem + stage * kStageBytes;
          uint8_t* sB = sA + kABytes;
          mbar_arrive_expect_tx(&full_bar[stage], kStageBytes);
          if (p.a_mode == 1)
            tma_load_im2col_4d(sA, mapA, &full_bar[stage], cc * kBlockK, cw, ch, cn, te.off_w, te.off_h);
          else
            tma_load_2d(sA, mapA, &full_bar[stage], te.kofs + cc * kBlockK, m0);
          tma_load_2d(sB, &tmB, &full_bar[stage], te.kofs + cc * kBlockK, n_t * BLOCK_N);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        };
        const int tap_base = MULTI ? ce.tap0 : 0;     // single class: a static table offset (no dependent parameter load)
        if (!km) {
          // dense walk — nested tap / channel-chunk loops: no integer division on the single producer thread
          // (the first ncu source view showed the producer, not TMA or the tensor pipe, as the limiter)
          for (int tap = 0; tap < ce.ntaps; ++tap) {
            const TapEntry te = p.taps[tap_base + tap];
            for (int cc = 0; cc < p.cchunks; ++cc) load_block(te, cc);
          }
        } else {
          // some weight blocks are empty: all-zero blocks are neither loaded nor multiplied
          KSkip ks; bool any = false;
          ks.begin(km, p.kmask_words, n_t * BLOCK_N, BLOCK_N, p.N);
          for (int tap = 0; tap < ce.ntaps; ++tap) {
            const TapEntry te = p.taps[tap_base + tap];
            for (int cc = 0; cc < p.cchunks; ++cc) {
              const bool last = tap == ce.ntaps - 1 && cc == p.cchunks - 1;
              if (!ks.on((te.kofs >> 6) + cc) && !(last && !any)) continue;
              any = true;
              load_block(te, cc);
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------ MMA issuer ------------------------------
    if (lane == 0) {
      constexpr uint32_t idesc = make_idesc_bf16(kBlockM, BLOCK_N, 0, 0);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      const uint32_t* const km = live_kmask(p.kmask, p.kmask_words, p.N);
      for (int w = 0; w < my_items; ++w) {
        const int tile = cta + w * n_cta;
        if (MULTI) {      // a class no tap reaches has no accumulator: its tiles belong to the epilogue warps alone
          int ci0, mt0, nt0; decode_tile(p, tile, n_tiles, ci0, mt0, nt0);
          if (p.cls[ci0].ntaps == 0) continue;
        }
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1, 2);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * BLOCK_N);
        auto mma_block = [&](uint32_t accumulate) {
          mbar_wait(&full_bar[stage], phase, 3);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + stage * kStageBytes);
          const uint32_t b_addr = a_addr + kABytes;
          const uint64_t adesc = make_smem_desc(a_addr, 16, 1024, kLayoutSW128);
          const uint64_t bdesc = make_smem_desc(b_addr, 16, 1024, kLayoutSW128);
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k) {
            // advance 16 elements (32 B) along K inside the 128-B swizzle row: +2 in 16-B units
            umma_bf16(d_tmem, adesc + (uint64_t)(2 * k), bdesc + (uint64_t)(2 * k), idesc, accumulate | (uint32_t)k);
          }
          umma_commit(&empty_bar[stage]);        // frees this smem stage when the MMAs have read it
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        };
        if (!MULTI && !km) {
          // dense single-class walk: no tile arithmetic at all on this thread (it paces the tensor pipe)
          const int kiters = p.cls[0].ntaps * p.cchunks;
          for (int it = 0; it < kiters; ++it) mma_block((uint32_t)it);
        } else {
          int ci = 0, m_t = 0, n_t = 0;
          if (MULTI) decode_tile(p, tile, n_tiles, ci, m_t, n_t); else n_t = tile % n_tiles;
          const ClsEntry& ce = p.cls[MULTI ? ci : 0];       // a class without taps issues nothing: its epilogue writes the addend (or zero) alone
          if (!km) {
            const int kiters = ce.ntaps * p.cchunks;
            for (int it = 0; it < kiters; ++it) mma_block((uint32_t)it);
          } else {
            KSkip ks; uint32_t any = 0;
            ks.begin(km, p.kmask_words, n_t * BLOCK_N, BLOCK_N, p.N);
            for (int tap = 0; tap < ce.ntaps; ++tap) {
              const int kb0 = p.taps[(MULTI ? ce.tap0 : 0) + tap].kofs >> 6;
              for (int cc = 0; cc < p.cchunks; ++cc) {
                const bool last = tap == ce.ntaps - 1 && cc == p.cchunks - 1;
                if (!ks.on(kb0 + cc) && !(last && !any)) continue;               // same decision as the producer
                mma_block(any);
                any = 1;
              }
            }
          }
        }
        umma_commit(&tfull_bar[acc]);            // accumulator complete -> epilogue
        if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    // ------------------------------ epilogue ------------------------------
    // 8 epilogue warps: the HBM-bound layers were limited by how fast 4 warps could drain TMEM (ncu: 3.5 TB/s of
    // DRAM traffic at 30 % tensor activity).  Two warps share each TMEM lane quarter and split the columns.
    const int quarter = warp & 3;             // TMEM lane quarter this warp may access
    const int half = (warp - 2) >> 2;         // which half of the 64-column chunks this warp drains
    int acc = 0; uint32_t acc_phase = 0;
    for (int w = 0; w < my_items; ++w) {
      int ci, m_t, n_t; get_tile(w, ci, m_t, n_t);
      const ClsEntry& ce = p.cls[MULTI ? ci : 0];
      const bool has_acc = MULTI ? ce.ntaps > 0 : true;   // a class no tap reaches: the accumulator was never written, its value is zero
      const int row = m_t * kBlockM + quarter * 32 + lane;
      const bool row_ok = row < ce.M;
      long long opix = 0;
      if (row_ok && !p.staged_store) {    // generic output mapping, one division chain per tile
        opix = row;
        if (MULTI || !p.linear) {
          int n, pp, qq; decompose_pixel(row, ce.P_it, ce.Q_it, n, pp, qq);
          opix = (long long)n * p.out_img_pix + (long long)(pp * p.osh + ce.oah) * p.out_row_pix + (qq * p.osw + ce.oaw);
        }
      }
      __nv_bfloat16* orow = p.out + opix * p.ldc;
      // staged-path geometry of this lane: rows r_in + 4i of the warp's 32, 16-byte column c16 of each 128-byte row
      const int r_in = lane >> 3, c16 = lane & 7;
      const long long wrow0 = (long long)m_t * kBlockM + quarter * 32;        // first row of this warp's 32
      const int rows_left = (int)(ce.M - wrow0 < 32 ? (ce.M - wrow0 < 0 ? 0 : ce.M - wrow0) : 32);
      const long long ldc = p.ldc;
      const int N = p.N;
      // element offset of output row i (rows r_in + 4i): the iteration pixel itself for a single class; for parity classes
      // the destination pixel — ONE division chain for the first row, the other seven follow by stepping 4 pixels
      long long ooff[MULTI ? 8 : 1];
      const long long rbase = (wrow0 + r_in) * ldc + c16 * 8;
      if (MULTI && p.staged_store) {
        int n, pp, qq; decompose_pixel((int)(wrow0 + r_in), ce.P_it, ce.Q_it, n, pp, qq);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const long long px = (long long)n * p.out_img_pix + (long long)(pp * p.osh + ce.oah) * p.out_row_pix + (qq * p.osw + ce.oaw);
          ooff[i] = px * ldc + c16 * 8;
          qq += 4;
          while (qq >= ce.Q_it) { qq -= ce.Q_it; if (++pp == ce.P_it) { pp = 0; ++n; } }
        }
      }
      auto row_off = [&](int i) -> long long { return MULTI ? ooff[MULTI ? i : 0] : rbase + (long long)(i * 4) * ldc; };
      if (MULTI && !has_acc) {
        // parity class no tap reaches (e.g. 3 of the 4 classes of a 1x1 stride-2 convolution): dX there is the fused addend
        // or zero — plain coalesced copies / stores; no accumulator exists, so no hand-shake with the MMA thread either
        if (p.staged_store) {
#pragma unroll 1
          for (int c = half * 64; c < BLOCK_N; c += 128) {
            const int n0 = n_t * BLOCK_N + c;
            if (n0 >= N) break;
            if (n0 + c16 * 8 + 8 > N) continue;
            uint4 z[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              z[i] = make_uint4(0u, 0u, 0u, 0u);
              if (p.addend && i * 4 + r_in < rows_left) z[i] = *reinterpret_cast<const uint4*>(p.addend + row_off(i) + n0);
            }
#pragma unroll
            for (int i = 0; i < 8; ++i)
              if (i * 4 + r_in < rows_left) *reinterpret_cast<uint4*>(p.out + row_off(i) + n0) = z[i];
          }
        } else if (row_ok && half == 0) {
          for (int j = n_t * BLOCK_N; j < min(p.N, (n_t + 1) * BLOCK_N); ++j)
            orow[j] = p.addend ? p.addend[opix * p.ldc + j] : __float2bfloat16_rn(0.f);
        }
        continue;
      }
      mbar_wait(&tfull_bar[acc], acc_phase, 4);
      tc_fence_after();
      const uint32_t t_base = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * BLOCK_N);
      if (p.staged_store) {
        // TMEM -> registers -> 128B-swizzled smem sub-tile (32 rows x 64 cols) -> coalesced global
        // stores, so every output line leaves the SM as full 128-byte rows instead of 32 scattered 16-byte pieces.
        // Everything that does not depend on the column chunk is hoisted (row pointers, validity, swizzled
        // staging offsets) and the staging buffer is addressed through the shared window (st/ld.shared, not
        // generic): the ncu source view of the first version had this loop at 2.3 us per 128x256 tile — longer
        // than the tile's MMAs (1.1 us) — with its stalls on generic LD/ST and re-loaded kernel parameters.
        const uint32_t buf = smem_u32(stg_base + (warp - 2) * kStgBytes);
        __nv_bfloat16* const gout = p.out;
        const __nv_bfloat16* const gadd = p.addend;
        {
        const float* bias = p.bias;
        float* stats = p.stats ? p.stats + (long long)(m_t * 4 + quarter) * 2 * N + c16 * 8 : nullptr;
        const uint32_t wr_base = buf + lane * 128;                              // my row (TMEM lane) in the staging tile
        const uint32_t wr_sw = (uint32_t)(lane & 7);
        const uint32_t rd_even = buf + r_in * 128 + ((uint32_t)(c16 ^ r_in) << 4);          // rows r_in + 8j
        const uint32_t rd_odd = buf + (r_in + 4) * 128 + ((uint32_t)(c16 ^ (r_in + 4)) << 4);  // rows r_in + 4 + 8j
        uint4 a_pref[8];
#pragma unroll 1
        for (int c = half * 64; c < BLOCK_N; c += 128) {
          const int n0 = n_t * BLOCK_N + c;
          if (n0 >= N) break;
          const bool col_ok = n0 + c16 * 8 + 8 <= N;
          // both 32-column halves of the chunk are requested before the one wait
          uint32_t v[64];
          tmem_ld_32x32(t_base + (uint32_t)c, v);
          tmem_ld_32x32(t_base + (uint32_t)(c + 32), v + 32);
          if (gadd) {
            // addend sub-tile of THIS chunk was prefetched into registers one chunk earlier (coalesced: 8 lanes
            // cover one 128-byte row, 4 rows per instruction); stage it, then prefetch the next chunk's
            if (c == half * 64) {
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                a_pref[i] = make_uint4(0u, 0u, 0u, 0u);
                if (i * 4 + r_in < rows_left && col_ok) a_pref[i] = *reinterpret_cast<const uint4*>(gadd + row_off(i) + n0);
              }
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) sts128(((i & 1) ? rd_odd : rd_even) + (uint32_t)((i >> 1) * 1024), a_pref[i]);
            if (c + 128 < BLOCK_N && n0 + 128 < N) {
              const bool col_ok2 = n0 + 128 + c16 * 8 + 8 <= N;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                a_pref[i] = make_uint4(0u, 0u, 0u, 0u);
                if (i * 4 + r_in < rows_left && col_ok2) a_pref[i] = *reinterpret_cast<const uint4*>(gadd + row_off(i) + n0 + 128);
              }
            }
            __syncwarp();
          }
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 64; j += 8) {
            float f[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) f[q] = __uint_as_float(v[j + q]);
            if (bias) {
#pragma unroll
              for (int q = 0; q < 8; ++q) if (n0 + j + q < N) f[q] += bias[n0 + j + q];
            }
            const uint32_t waddr = wr_base + (((uint32_t)(j >> 3) ^ wr_sw) << 4);   // 16-byte chunk j/8 of my row, swizzled
            if (gadd) {
              // fused skip-gradient accumulation: each thread reads its own row of the staged addend back before
              // overwriting it with the result
              const uint4 a = lds128(waddr);
              const __nv_bfloat162* ah = reinterpret_cast<const __nv_bfloat162*>(&a);
#pragma unroll
              for (int q = 0; q < 4; ++q) { const float2 t2 = __bfloat1622float2(ah[q]); f[2 * q] += t2.x; f[2 * q + 1] += t2.y; }
            }
            __nv_bfloat162 h0 = __floats2bfloat162_rn(f[0], f[1]);
            __nv_bfloat162 h1 = __floats2bfloat162_rn(f[2], f[3]);
            __nv_bfloat162 h2 = __floats2bfloat162_rn(f[4], f[5]);
            __nv_bfloat162 h3 = __floats2bfloat162_rn(f[6], f[7]);
            uint4 pk;
            pk.x = *(uint32_t*)&h0; pk.y = *(uint32_t*)&h1; pk.z = *(uint32_t*)&h2; pk.w = *(uint32_t*)&h3;
            sts128(waddr, pk);
          }
          __syncwarp();
          // smem -> global, coalesced: 8 lanes write one full 128-byte output row, 4 rows per instruction.
          // Plain stores are fire-and-forget, so the staging buffer is free again after this read-back
          // (a TMA store here made every chunk wait ~2 us for the previous store to drain: 9 us per tile).
          uint4 o[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) o[i] = lds128(((i & 1) ? rd_odd : rd_even) + (uint32_t)((i >> 1) * 1024));
          if (BNB) {
            // gate + BatchNorm backward sums on the row-coalesced view: this lane owns channels n0 + c16*8 .. +8 of rows r_in + 4i
            uint4 yv[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              yv[i] = make_uint4(0u, 0u, 0u, 0u);
              if (i * 4 + r_in < rows_left && col_ok) yv[i] = *reinterpret_cast<const uint4*>(p.bn_y + row_off(i) + n0);
            }
            float sc[8], sf[8], is_[8], nm[8], s1[8], s2[8];
            if (col_ok) {
              const int cb = n0 + c16 * 8;
#pragma unroll
              for (int q = 0; q < 8; q += 4) {
                const float4 one4 = make_float4(1.f, 1.f, 1.f, 1.f), zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
                const float4 a4 = p.bn_weight ? *reinterpret_cast<const float4*>(p.bn_weight + cb + q) : one4;
                const float4 b4 = p.bn_bias ? *reinterpret_cast<const float4*>(p.bn_bias + cb + q) : zero4;
                const float4 m4 = *reinterpret_cast<const float4*>(p.bn_mean + cb + q), i4 = *reinterpret_cast<const float4*>(p.bn_invstd + cb + q);
                is_[q] = i4.x; is_[q + 1] = i4.y; is_[q + 2] = i4.z; is_[q + 3] = i4.w;
                nm[q] = m4.x; nm[q + 1] = m4.y; nm[q + 2] = m4.z; nm[q + 3] = m4.w;
                // scale / shift exactly as k_bn_finalize_stats computed them for the forward apply pass
                sc[q] = a4.x * i4.x; sc[q + 1] = a4.y * i4.y; sc[q + 2] = a4.z * i4.z; sc[q + 3] = a4.w * i4.w;
                sf[q] = fmaf(-m4.x, sc[q], b4.x); sf[q + 1] = fmaf(-m4.y, sc[q + 1], b4.y);
                sf[q + 2] = fmaf(-m4.z, sc[q + 2], b4.z); sf[q + 3] = fmaf(-m4.w, sc[q + 3], b4.w);
              }
            } else {
#pragma unroll
              for (int q = 0; q < 8; ++q) { sc[q] = 0.f; sf[q] = 0.f; is_[q] = 0.f; nm[q] = 0.f; }
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) { s1[q] = 0.f; s2[q] = 0.f; }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              if (i * 4 + r_in < rows_left) {
                __nv_bfloat162* gh = reinterpret_cast<__nv_bfloat162*>(&o[i]);
                const __nv_bfloat162* yh = reinterpret_cast<const __nv_bfloat162*>(&yv[i]);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  float2 d2 = __bfloat1622float2(gh[q]);
                  const float2 y2 = __bfloat1622float2(yh[q]);
                  // the forward wrote z = max(fma(y, scale, shift), 0): same expression, same operands -> same decision
                  if (!(fmaf(y2.x, sc[2 * q], sf[2 * q]) > 0.f)) d2.x = 0.f;
                  if (!(fmaf(y2.y, sc[2 * q + 1], sf[2 * q + 1]) > 0.f)) d2.y = 0.f;
                  gh[q] = __floats2bfloat162_rn(d2.x, d2.y);                    // exact: d2 is a bf16 value or zero
                  s1[2 * q] += d2.x;     s2[2 * q] = fmaf(d2.x, (y2.x - nm[2 * q]) * is_[2 * q], s2[2 * q]);
                  s1[2 * q + 1] += d2.y; s2[2 * q + 1] = fmaf(d2.y, (y2.y - nm[2 * q + 1]) * is_[2 * q + 1], s2[2 * q + 1]);
                }
              }
            }
#pragma unroll
            for (int i = 0; i < 8; ++i)
              if (i * 4 + r_in < rows_left && col_ok) *reinterpret_cast<uint4*>(gout + row_off(i) + n0) = o[i];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              s1[q] += __shfl_xor_sync(0xffffffffu, s1[q], 8);  s2[q] += __shfl_xor_sync(0xffffffffu, s2[q], 8);
              s1[q] += __shfl_xor_sync(0xffffffffu, s1[q], 16); s2[q] += __shfl_xor_sync(0xffffffffu, s2[q], 16);
            }
            if (r_in == 0 && col_ok) {
              float4* d1 = reinterpret_cast<float4*>(stats + n0);
              float4* d2 = reinterpret_cast<float4*>(stats + N + n0);
              d1[0] = make_float4(s1[0], s1[1], s1[2], s1[3]); d1[1] = make_float4(s1[4], s1[5], s1[6], s1[7]);
              d2[0] = make_float4(s2[0], s2[1], s2[2], s2[3]); d2[1] = make_float4(s2[4], s2[5], s2[6], s2[7]);
            }
          } else {
#pragma unroll
          for (int i = 0; i < 8; ++i)
            if (i * 4 + r_in < rows_left && col_ok) *reinterpret_cast<uint4*>(gout + row_off(i) + n0) = o[i];
          if (stats) {
            // BatchNorm batch statistics of exactly the values just stored (bf16-rounded): this thread owns 8 channels
            // of rows r_in, r_in+4, ...; a fixed-order xor tree over the 4 row groups finishes the 32 rows
            float s1[8], s2[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) { s1[q] = 0.f; s2[q] = 0.f; }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              if (i * 4 + r_in < rows_left) {
                const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&o[i]);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                  const float2 t2 = __bfloat1622float2(h2[q]);
                  s1[2 * q] += t2.x; s2[2 * q] = fmaf(t2.x, t2.x, s2[2 * q]);
                  s1[2 * q + 1] += t2.y; s2[2 * q + 1] = fmaf(t2.y, t2.y, s2[2 * q + 1]);
                }
              }
            }
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              s1[q] += __shfl_xor_sync(0xffffffffu, s1[q], 8);  s2[q] += __shfl_xor_sync(0xffffffffu, s2[q], 8);
              s1[q] += __shfl_xor_sync(0xffffffffu, s1[q], 16); s2[q] += __shfl_xor_sync(0xffffffffu, s2[q], 16);
            }
            if (r_in == 0 && col_ok) {
              float4* d1 = reinterpret_cast<float4*>(stats + n0);
              float4* d2 = reinterpret_cast<float4*>(stats + N + n0);
              d1[0] = make_float4(s1[0], s1[1], s1[2], s1[3]); d1[1] = make_float4(s1[4], s1[5], s1[6], s1[7]);
              d2[0] = make_float4(s2[0], s2[1], s2[2], s2[3]); d2[1] = make_float4(s2[4], s2[5], s2[6], s2[7]);
            }
          }
          }   // !BNB
          __syncwarp();
        }
        }   // has_acc
      } else {
#pragma unroll 1
      for (int c = half * 32; c < BLOCK_N; c += 64) {
        uint32_t v[32];
        tmem_ld_32x32(t_base + (uint32_t)c, v);
        tmem_ld_wait();
        const int n0 = n_t * BLOCK_N + c;
        if (row_ok && n0 < p.N) {
          float f[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
          if (p.bias) {
#pragma unroll
            for (int j = 0; j < 32; ++j) if (n0 + j < p.N) f[j] += p.bias[n0 + j];
          }
          if (p.addend) {
            const __nv_bfloat16* ar = p.addend + opix * p.ldc + n0;
            for (int j = 0; j < 32; ++j) if (n0 + j < p.N) f[j] += __bfloat162float(ar[j]);
          }
          __nv_bfloat16* dst = orow + n0;
          if (n0 + 32 <= p.N && (((uintptr_t)dst) & 15) == 0) {
#pragma unroll
            for (int j = 0; j < 32; j += 8) {
              __nv_bfloat162 h0 = __floats2bfloat162_rn(f[j], f[j + 1]);
              __nv_bfloat162 h1 = __floats2bfloat162_rn(f[j + 2], f[j + 3]);
              __nv_bfloat162 h2 = __floats2bfloat162_rn(f[j + 4], f[j + 5]);
              __nv_bfloat162 h3 = __floats2bfloat162_rn(f[j + 6], f[j + 7]);
              uint4 pk;
              pk.x = *(uint32_t*)&h0; pk.y = *(uint32_t*)&h1; pk.z = *(uint32_t*)&h2; pk.w = *(uint32_t*)&h3;
              *(uint4*)(dst + j) = pk;
            }
          } else {
            for (int j = 0; j < 32; ++j) if (n0 + j < p.N) dst[j] = __float2bfloat16_rn(f[j]);
          }
        }
      }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      if (++acc == kAccStages) { acc = 0; acc_phase ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, kTmemCols); }
}

// ============================================================================================
__global__ void __launch_bounds__(kThreads, 1)
k_igemm_wgrad(const __grid_constant__ CUtensorMap tmA /* dY [Kpix, Cout] */,
              const __grid_constant__ CUtensorMap tmB /* X im2col or Xcol tiled */,
              const __grid_constant__ WgParams p) {
  constexpr int kABytes = kBlockM * kBlockK * 2;          // 2 boxes of [64 pixels x 64 couts] = 16 KB
  constexpr int kChunkBytes = 64 * kBlockK * 2;           // 8 KB per 64-column chunk
  constexpr int kMaxNb = 4;
  constexpr int kStageBytes = kABytes + kMaxNb * kChunkBytes;   // 48 KB
  constexpr int kStages = 4;
  constexpr uint32_t kTmemCols = 512;                     // 2 accumulator stages x 256 columns
  pdl_trigger();
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint64_t* full_bar = (uint64_t*)(smem + kStages * kStageBytes);
  uint64_t* empty_bar = full_bar + kStages;
  uint64_t* tfull_bar = empty_bar + kStages;
  uint64_t* tempty_bar = tfull_bar + 2;
  uint32_t* tmem_slot = (uint32_t*)(tempty_bar + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int items = p.m_tiles * p.n_tiles * p.splits;
  const int ncols = p.nb * 64;
  const int row_groups = (p.Mc + 63) >> 6;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA); prefetch_tmap(&tmB);
    for (int i = 0; i < kStages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 4); }
    fence_mbar_init();
  }
  if (warp == 1) { tmem_alloc(tmem_slot, kTmemCols); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  const uint32_t* const km = live_kmask(p.kmask, p.kmask_words, p.Mc);     // null: no empty block anywhere (or no mask given)

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0; uint32_t phase = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x) {
        // split-major order: the CTAs running at the same time work on the SAME pixel range for different
        // (m, n) tiles, so each X / dY chunk comes from HBM once and from L2 for the siblings (ncu: 35.7 GB of
        // DRAM reads per step with tile-major order vs ~23 GB algorithmic)
        const int ntile = p.m_tiles * p.n_tiles;
        const int split = item / ntile, tile = item - split * ntile;
        const int n_t = tile / p.m_tiles, m_t = tile % p.m_tiles;
        const int kb0 = split * p.kb_per_split;
        const int kb1 = min(p.kblocks, kb0 + p.kb_per_split);
        const int chunk0 = n_t * p.nb;
        const int nvalid = min(p.nb, p.chunks - chunk0);
        if (km && wg_item_empty(km, p.kmask_words, row_groups, m_t, chunk0, nvalid)) continue;   // all three roles skip the same items
        // Everything that needs an integer division is hoisted out of the K loop (one producer thread
        // feeds the whole SM): per-chunk (tap, channel) coordinates once per item, and the pixel
        // coordinate of a K block advanced incrementally by 64 = sn*P*Q + sp*Q + sq.
        int c_c[4]; uint16_t c_ow[4], c_oh[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int chunk = min(chunk0 + j, p.chunks - 1), tap = chunk / p.cchunks;
          c_c[j] = (chunk - tap * p.cchunks) * 64; c_ow[j] = p.taps[tap].off_w; c_oh[j] = p.taps[tap].off_h;
        }
        int cn, cp, cq; decompose_pixel(kb0 * kBlockK, p.P_it, p.Q_it, cn, cp, cq);
        const int sq = kBlockK % p.Q_it, t1 = kBlockK / p.Q_it, sp = t1 % p.P_it, sn = t1 / p.P_it;
        for (int kb = kb0; kb < kb1; ++kb) {
          const int pix0 = kb * kBlockK;
          mbar_wait(&empty_bar[stage], phase ^ 1, 11);
          mbar_arrive_expect_tx(&full_bar[stage], kABytes + nvalid * kChunkBytes);
          uint8_t* sA = smem + stage * kStageBytes;
          uint8_t* sB = sA + kABytes;
          tma_load_2d(sA, &tmA, &full_bar[stage], m_t * kBlockM, pix0);
          tma_load_2d(sA + kChunkBytes, &tmA, &full_bar[stage], m_t * kBlockM + 64, pix0);
          if (p.b_mode == 1) {
            const int cw = p.base_w + cq * p.step_w, ch = p.base_h + cp * p.step_h;
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (j < nvalid)
                tma_load_im2col_4d(sB + j * kChunkBytes, &tmB, &full_bar[stage], c_c[j], cw, ch, cn, c_ow[j], c_oh[j]);
            cq += sq; if (cq >= p.Q_it) { cq -= p.Q_it; cp += 1; }
            cp += sp; if (cp >= p.P_it) { cp -= p.P_it; cn += 1; }
            cn += sn;
          } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
              if (j < nvalid) tma_load_2d(sB + j * kChunkBytes, &tmB, &full_bar[stage], (chunk0 + j) * 64, pix0);
          }
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      const uint32_t idesc = make_idesc_bf16(kBlockM, ncols, 1, 1);
      int stage = 0; uint32_t phase = 0;
      int acc = 0; uint32_t acc_phase = 0;
      for (int item = blockIdx.x; item < items; item += gridDim.x) {
        const int split = item / (p.m_tiles * p.n_tiles);
        if (km) {
          const int tile = item - split * (p.m_tiles * p.n_tiles), n_t = tile / p.m_tiles, m_t = tile - n_t * p.m_tiles;
          if (wg_item_empty(km, p.kmask_words, row_groups, m_t, n_t * p.nb, min(p.nb, p.chunks - n_t * p.nb))) continue;
        }
        const int kb0 = split * p.kb_per_split;
        const int kb1 = min(p.kblocks, kb0 + p.kb_per_split);
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1, 12);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * 256);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase, 13);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(smem + stage * kStageBytes);
          const uint32_t b_addr = a_addr + kABytes;
          // MN-major SW128: 64 MN elements per 128-B row, 8 K rows per 1024-B atom (SBO),
          // next 64-wide MN block at LBO = 64 rows * 128 B
          const uint64_t adesc = make_smem_desc(a_addr, kChunkBytes, 1024, kLayoutSW128);
          const uint64_t bdesc = make_smem_desc(b_addr, kChunkBytes, 1024, kLayoutSW128);
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k) {
            // 16 K rows = 2 swizzle atoms = 2048 B
            umma_bf16(d_tmem, adesc + (uint64_t)(128 * k), bdesc + (uint64_t)(128 * k), idesc, (kb > kb0 || k > 0));
          }
          umma_commit(&empty_bar[stage]);
          if (++stage == kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&tfull_bar[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1; }
      }
    }
  } else {
    const int quarter = warp & 3;
    int acc = 0; uint32_t acc_phase = 0;
    for (int item = blockIdx.x; item < items; item += gridDim.x) {
      const int ntile = p.m_tiles * p.n_tiles;
      const int split = item / ntile, tile = item - split * ntile;
      if (km) {
        const int n_t = tile / p.m_tiles, m_t = tile - n_t * p.m_tiles;
        if (wg_item_empty(km, p.kmask_words, row_groups, m_t, n_t * p.nb, min(p.nb, p.chunks - n_t * p.nb))) continue;
      }
      float* prow = p.partial + (((long long)tile * p.splits + split) * kBlockM + quarter * 32 + lane) * ncols;
      mbar_wait(&tfull_bar[acc], acc_phase, 14);
      tc_fence_after();
      const uint32_t t_base = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * 256);
#pragma unroll 1
      for (int c = 0; c < ncols; c += 32) {
        uint32_t v[32];
        tmem_ld_32x32(t_base + (uint32_t)c, v);
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          *(uint4*)(prow + c + j) = make_uint4(v[j], v[j + 1], v[j + 2], v[j + 3]);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty_bar[acc]);
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, kTmemCols); }
}

// dW[co][ci][tap] (fp32 OIHW) = mask * sum_split partial   — fixed summation order (deterministic, no atomics).
// Grid (Cout, K chunks): a CTA owns KT = 256 / sl consecutive K columns (kk = tap*cin_p + ci) of one output channel;
// its 256 threads are KT k-lanes x `sl` split-lanes.  Split lane j folds splits j, j+sl, ... with eight independent
// loads in flight, the lanes are then combined in lane order.  (The first version looped over the K chunks inside one
// CTA per channel: 18 dependent rounds of L2/DRAM latency for a 3x3x64 layer — 50-80 us for 150 KB of output.)
__global__ void __launch_bounds__(256) k_wgrad_finalize(const float* __restrict__ partial, const float* __restrict__ mask,
                                                        float* __restrict__ dw, int cout, int cin_real, int cin_p, int rs,
                                                        int nb, int m_tiles, int n_tiles, int splits, int sl,
                                                        const uint32_t* __restrict__ kmask, int kmask_words) {
  pdl_enter();
  __shared__ float s_lane[256];
  const uint32_t* const km = live_kmask(kmask, kmask_words, cout);
  const int co = blockIdx.x;
  const int m_t = co / kBlockM, r = co % kBlockM;
  const int ktot = rs * cin_p;
  const int ncols = nb * 64;
  const int KT = 256 / sl;
  const int kl = threadIdx.x % KT, sj = threadIdx.x / KT;
  const int kk = blockIdx.y * KT + kl;
  const long long sstride = (long long)kBlockM * ncols;          // floats between consecutive splits of a tile
  float a[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  // a work item the GEMM skipped has no partials (the workspace holds whatever was there): its gradient is exactly zero
  const int chunks = (ktot + 63) >> 6;
  const bool skipped = km && kk < ktot &&
                       wg_item_empty(km, kmask_words, (cout + 63) >> 6, m_t, ((kk >> 6) / nb) * nb, min(nb, chunks - ((kk >> 6) / nb) * nb));
  if (kk < ktot && !skipped) {
    const int chunk = kk >> 6, n_t = chunk / nb, col = (chunk - n_t * nb) * 64 + (kk & 63);
    const float* base = partial + ((((long long)n_t * m_tiles + m_t) * splits) * kBlockM + r) * ncols + col;
    int sp = sj;
    for (; sp + 7 * sl < splits; sp += 8 * sl) {
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = __ldcs(base + (long long)(sp + j * sl) * sstride);
#pragma unroll
      for (int j = 0; j < 8; ++j) a[j] += v[j];
    }
    for (; sp < splits; sp += sl) a[0] += __ldcs(base + (long long)sp * sstride);
  }
  s_lane[sj * KT + kl] = ((a[0] + a[1]) + (a[2] + a[3])) + ((a[4] + a[5]) + (a[6] + a[7]));
  __syncthreads();
  if (sj == 0 && kk < ktot) {
    float acc = 0.f;
    for (int j = 0; j < sl; ++j) acc += s_lane[j * KT + kl];
    const int tap = kk / cin_p, ci = kk - tap * cin_p;
    if (ci < cin_real) {
      const long long o = ((long long)co * cin_real + ci) * rs + tap;
      dw[o] = skipped ? 0.f : mask[o] * acc;
    }
  }
}

// db[c] = sum over pixels of dy[pix][c]  (bias gradient), dy bf16 [npix, ldc], c % 8 == 0.
// Two stages, both in fixed order (deterministic): every CTA of a (pixel split x channel tile) grid sums its pixels — a thread
// owns one 16-byte vector of 8 channels and walks the pixel axis, 4 rows in flight — into part[split][c]; a small kernel
// folds the splits.  (The first version ran ONE CTA per 32 channels over all pixels with 2-byte loads: 200 us per layer —
// 41 % of the DeiT-S step, profiles/r02_launches_deit_B64.md.)
__global__ void __launch_bounds__(256) k_colsum_part(const __nv_bfloat16* __restrict__ dy, long long npix, int c, int ldc,
                                                     float* __restrict__ part) {
  pdl_enter();
  __shared__ float s_acc[256][9];
  const int tx = threadIdx.x, ty = threadIdx.y, TX = blockDim.x, TY = blockDim.y;
  const int cvec = blockIdx.y * TX + tx;
  const bool act = cvec * 8 < c;
  float a[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = 0.f;
  auto add8 = [&](const uint4& v) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) { const float2 f = __bfloat1622float2(h[i]); a[2 * i] += f.x; a[2 * i + 1] += f.y; }
  };
  if (act) {
    const long long stride = (long long)gridDim.x * TY;
    long long p = (long long)blockIdx.x * TY + ty;
    const __nv_bfloat16* src = dy + (size_t)cvec * 8;
    for (; p + 3 * stride < npix; p += 4 * stride) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = *reinterpret_cast<const uint4*>(src + (size_t)(p + u * stride) * ldc);
#pragma unroll
      for (int u = 0; u < 4; ++u) add8(v[u]);
    }
    for (; p < npix; p += stride) add8(*reinterpret_cast<const uint4*>(src + (size_t)p * ldc));
  }
  const int tid = ty * TX + tx;
#pragma unroll
  for (int i = 0; i < 8; ++i) s_acc[tid][i] = a[i];
  __syncthreads();
  if (ty == 0 && act) {
    float r[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) r[i] = 0.f;
    for (int j = 0; j < TY; ++j)
#pragma unroll
      for (int i = 0; i < 8; ++i) r[i] += s_acc[j * TX + tx][i];
#pragma unroll
    for (int i = 0; i < 8; ++i) part[(size_t)blockIdx.x * c + cvec * 8 + i] = r[i];
  }
}

__global__ void __launch_bounds__(256) k_colsum_fold(const float* __restrict__ part, int nparts, int c, float* __restrict__ db) {
  pdl_enter();
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= c) return;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
  int j = 0;
  for (; j + 3 < nparts; j += 4) {                    // four independent chains, combined in a fixed order
    s0 += part[(size_t)j * c + ch]; s1 += part[(size_t)(j + 1) * c + ch];
    s2 += part[(size_t)(j + 2) * c + ch]; s3 += part[(size_t)(j + 3) * c + ch];
  }
  for (; j < nparts; ++j) s0 += part[(size_t)j * c + ch];
  db[ch] = (s0 + s1) + (s2 + s3);
}

// ============================================================================================
// host side
// ============================================================================================
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
typedef CUresult (*PFN_encodeIm2col)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                     const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*, CUtensorMapInterleave,
                                     CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled g_encodeTiled = nullptr;
static PFN_encodeIm2col g_encodeIm2col = nullptr;
static int g_driver_version = 0;

static int load_driver_fns() {
  static std::once_flag once;
  static int rc = TP_OK;
  std::call_once(once, []() {
    void* f1 = nullptr; void* f2 = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f1, cudaEnableDefault, &q) != cudaSuccess || !f1 ||
        cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &f2, cudaEnableDefault, &q) != cudaSuccess || !f2) {
      set_last_cuda_error(cudaErrorUnknown, "cudaGetDriverEntryPoint(cuTensorMapEncode*)");
      rc = TP_ERR_CUDA;
      return;
    }
    g_encodeTiled = (PFN_encodeTiled)f1;
    g_encodeIm2col = (PFN_encodeIm2col)f2;
    cudaDriverGetVersion(&g_driver_version);
  });
  return rc;
}

static int fail_cu(CUresult r, const char* what) {
  static thread_local char buf[128];
  snprintf(buf, sizeof(buf), "%s -> CUresult %d", what, (int)r);
  set_last_cuda_error(cudaErrorInvalidValue, buf);
  return TP_ERR_CUDA;
}

// 2-D bf16 tensor [rows][cols] (cols contiguous, row stride ld elements), box = [box_rows][64 cols], SW128.
static int make_tiled_map(CUtensorMap* m, const void* ptr, uint64_t cols, uint64_t rows, uint64_t ld_elems, uint32_t box_rows) {
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld_elems * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t es[2] = {1, 1};
  CUresult r = g_encodeTiled(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, es,
                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail_cu(r, "cuTensorMapEncodeTiled");
  return TP_OK;
}

// im2col map over NHWC bf16 [n][h][w][c]: `pixels` consecutive iteration positions x 64 channels.
// Iteration grid (P_it x Q_it per image) starts at (base_h, base_w) and advances by (step_h, step_w).
static int make_im2col_map(CUtensorMap* m, const void* ptr, int n, int h, int w, int c,
                           int base_w, int base_h, int step_w, int step_h, int P_it, int Q_it, uint32_t pixels) {
  cuuint64_t dims[4] = {(cuuint64_t)c, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
  cuuint64_t strides[3] = {(cuuint64_t)c * 2, (cuuint64_t)w * c * 2, (cuuint64_t)h * w * c * 2};
  // bounding box: base positions run from `lower` while < extent + upper  =>  count = Q_it
  int lower[2] = {base_w, base_h};
  int upper[2] = {(Q_it - 1) * step_w + 1 + base_w - w, (P_it - 1) * step_h + 1 + base_h - h};
  cuuint32_t es[4] = {1, (cuuint32_t)step_w, (cuuint32_t)step_h, 1};
  CUresult r = g_encodeIm2col(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, lower, upper,
                              64, pixels, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail_cu(r, "cuTensorMapEncodeIm2col");
  // Driver quirk (CUDA <= 13.1 drivers, see CUTLASS copy_traits_sm90_im2col.hpp): for tensors
  // smaller than 128 KiB bit 21 of the second descriptor word must be cleared.
  if (g_driver_version <= 13010 && (size_t)n * h * w * c * 2 < 131072)
    reinterpret_cast<uint64_t*>(m)[1] &= ~(1ull << 21);
  return TP_OK;
}

// Split-K factor of the wgrad GEMM.  Every (tile, split) item costs its share of the K loop plus a fixed 128 x 256
// fp32 partial tile (written once, read once by the finalize pass), so the cheapest choice is the SMALLEST split
// count that reaches the minimal makespan over the persistent CTAs — not "as many as fit in two waves": at a per-GPU
// batch of 64 the partial tiles were most of the wgrad traffic (54 layers x ~300 items x 128 KB, twice).
static int pick_wgrad_splits(int tiles, int kblocks, int nb) {
  const int sms = sm_count();
  int smax = (2 * sms) / tiles;
  if (smax > kblocks) smax = kblocks;
  if (smax < 1) smax = 1;
  const double c_kb = 0.30;                         // us per 64-pixel K block (48 KB of operands, one 128x256x64 MMA group)
  const double c_part = 0.33 * nb;                  // us to drain one partial tile from TMEM to global
  const double c_fin = 0.013 * nb;                  // us of finalize traffic per partial tile (read once at ~5 TB/s)
  int best = 1; double best_cost = 1e30;
  for (int s = 1; s <= smax; ++s) {
    const int kb = (kblocks + s - 1) / s;
    const int s_eff = (kblocks + kb - 1) / kb;      // no empty splits
    const long long items = (long long)tiles * s_eff;
    const long long waves = (items + sms - 1) / sms;
    const double cost = (double)waves * (kb * c_kb + c_part) + (double)items * c_fin;
    if (cost < best_cost - 1e-9) { best_cost = cost; best = s_eff; }
  }
  return best;
}

static bool is_plain_gemm(const tp_conv_desc* d) {
  return d->r == 1 && d->s == 1 && d->stride_h == 1 && d->stride_w == 1 && d->pad_h == 0 && d->pad_w == 0;
}

static int pick_block_n(long long m_tiles, int n) {
  // favour wide tiles (fewer re-reads of the activation tile), but keep the last wave full
  const int sms = sm_count();
  if (const char* e = getenv("TP_IGEMM_BN")) {        // experiments only: force the tile width
    const int f = atoi(e);
    if ((f == 64 || f == 128 || f == 256) && (f == 64 || n > f / 2)) return f;
  }
  int best = 64; double best_score = -1;
  const int cands[3] = {256, 128, 64};
  const double weight[3] = {1.0, 0.92, 0.75};
  for (int i = 0; i < 3; ++i) {
    int bn = cands[i];
    if (bn > 64 && n <= bn / 2) continue;
    long long tiles = m_tiles * ((n + bn - 1) / bn);
    long long waves = (tiles + sms - 1) / sms;
    double eff = (double)tiles / (double)(waves * sms) * weight[i];
    if (eff > best_score) { best_score = eff; best = bn; }
  }
  return best;
}

template <int BN, bool MULTI, bool BNB = false>
static int launch_fwd(const AMaps& a, const CUtensorMap& b, FwdParams& p, cudaStream_t st) {
  constexpr int kTail = 8 * 32 * 128 + 1024 + 512;    // epilogue staging, alignment slack, barriers
  constexpr int smem = fwd_stages(BN) * (kBlockM * kBlockK * 2 + BN * kBlockK * 2) + kTail;
  const int n_tiles = (p.N + BN - 1) / BN;
  static bool attr_set = false;
  if (!attr_set) {
    TP_CUDA_CHECK(cudaFuncSetAttribute(k_igemm_fwd<BN, MULTI, BNB>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_set = true;
  }
  // work items: per class, (M tiles) x (N tiles), classes back to back
  long long ctiles = 0;
  for (int c = 0; c < p.ncls; ++c) {
    p.cls[c].m_tiles = (int)((p.cls[c].M + kBlockM - 1) / kBlockM);
    if (ctiles > 0x7fffffffll) return TP_ERR_UNSUPPORTED;
    p.cls[c].tile0 = (int)ctiles;
    ctiles += (long long)p.cls[c].m_tiles * n_tiles;
  }
  if (ctiles > 0x7fffffffll || ctiles <= 0) return TP_ERR_UNSUPPORTED;
  const int grid = (int)(ctiles < sm_count() ? ctiles : sm_count());
  TP_CUDA_CHECK(launch(k_igemm_fwd<BN, MULTI, BNB>, grid, kFwdThreads, smem, st, a, b, p));
  TP_LAUNCH_CHECK();
  return TP_OK;
}

static int run_fwd(const AMaps& a, const CUtensorMap& b, FwdParams& p, int bn, cudaStream_t st) {
  // 16-byte aligned output rows -> the epilogue stages 32x64 sub-tiles through smem and writes full 128-byte lines
  // (for any pixel mapping: a strided dgrad's parity classes compute the destination pixel of each row)
  p.linear = p.ncls == 1 && p.osh == 1 && p.osw == 1 && p.cls[0].oah == 0 && p.cls[0].oaw == 0 &&
             p.out_row_pix == p.cls[0].Q_it && p.out_img_pix == (long long)p.cls[0].P_it * p.cls[0].Q_it;
  p.staged_store = (p.ldc % 8 == 0 && p.N % 8 == 0 && (((uintptr_t)p.out) & 15) == 0 &&
                    (!p.addend || (((uintptr_t)p.addend) & 15) == 0)) ? 1 : 0;
  if (p.stats && !(p.staged_store && p.linear)) return TP_ERR_UNSUPPORTED;
  // the general-mapping instantiation only where it is needed: parity classes, or a single class whose output is not
  // the iteration order itself
  if (!p.linear) {
    if (bn == 256) return launch_fwd<256, true>(a, b, p, st);
    if (bn == 128) return launch_fwd<128, true>(a, b, p, st);
    return launch_fwd<64, true>(a, b, p, st);
  }
  if (p.bn_y) {      // BatchNorm-backward epilogue (needs the linear staged path; the caller checked the shapes)
    if (!p.staged_store || !p.stats) return TP_ERR_UNSUPPORTED;
    if (bn == 256) return launch_fwd<256, false, true>(a, b, p, st);
    if (bn == 128) return launch_fwd<128, false, true>(a, b, p, st);
    return launch_fwd<64, false, true>(a, b, p, st);
  }
  if (bn == 256) return launch_fwd<256, false>(a, b, p, st);
  if (bn == 128) return launch_fwd<128, false>(a, b, p, st);
  return launch_fwd<64, false>(a, b, p, st);
}

}  // namespace tp

using namespace tp;

extern "C" {

size_t tp_conv_workspace_bytes(const tp_conv_desc* d, int op) {
  if (!d) return 0;
  if (op != 2) return 256;
  // wgrad: split-K partial tiles
  const int cin_p = d->cin;
  const int ktot = ((d->r * d->s * cin_p) + 63) / 64 * 64;
  const int chunks = ktot / 64;
  const int nb = chunks >= 4 ? 4 : chunks;
  const int m_tiles = (d->cout + kBlockM - 1) / kBlockM;
  const int n_tiles = (chunks + nb - 1) / nb;
  const long long kpix = (long long)d->n * d->p * d->q;
  const int kblocks = (int)((kpix + 63) / 64);
  const int sms = sm_count();
  int splits = (2 * sms) / (m_tiles * n_tiles);          // upper bound of pick_wgrad_splits()
  if (splits > kblocks) splits = kblocks;
  if (splits < 1) splits = 1;
  return (size_t)m_tiles * n_tiles * splits * kBlockM * nb * 64 * sizeof(float) + 1024;
}

size_t tp_conv_stats_rows(const tp_conv_desc* d) {
  if (!d) return 0;
  const long long M = (long long)d->n * d->p * d->q;
  return (size_t)((M + kBlockM - 1) / kBlockM) * 4;
}

int tp_conv_fprop(const tp_conv_desc* d, const void* x, const void* wf, const void* bias_f32,
                  void* y, void* ws, size_t ws_bytes, void* stream) {
  return tp_conv_fprop_stats(d, x, wf, nullptr, bias_f32, y, nullptr, ws, ws_bytes, stream);
}

int tp_conv_fprop_stats(const tp_conv_desc* d, const void* x, const void* wf, const void* kmask_f, const void* bias_f32,
                        void* y, void* stats, void* ws, size_t ws_bytes, void* stream) {
  (void)ws; (void)ws_bytes;
  if (!d || !x || !wf || !y) return TP_ERR_INVALID;
  if (stats && (d->cout % 8 != 0 || (((uintptr_t)y) & 15) != 0 || (((uintptr_t)stats) & 15) != 0)) return TP_ERR_UNSUPPORTED;
  if (d->cin % 8 != 0 || d->r * d->s > kMaxTaps) return TP_ERR_UNSUPPORTED;
  if (d->r * d->s > 1 && d->cin % 64 != 0) return TP_ERR_UNSUPPORTED;
  int rc = load_driver_fns(); if (rc) return rc;
  rc = bind_device_of(d ? (const void*)x : nullptr); if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  FwdParams p = {};
  p.M = d->n * d->p * d->q; p.N = d->cout;
  p.ncls = 1;
  ClsEntry& ce = p.cls[0];
  ce.M = p.M; ce.P_it = d->p; ce.Q_it = d->q; ce.ntaps = d->r * d->s; ce.tap0 = 0; ce.oah = 0; ce.oaw = 0;
  p.cchunks = (d->cin + 63) / 64;
  p.out_img_pix = (long long)d->p * d->q; p.out_row_pix = d->q;
  p.osh = 1; p.osw = 1;
  p.ldc = d->cout; p.out = (__nv_bfloat16*)y; p.bias = (const float*)bias_f32;
  p.stats = (float*)stats;
  p.kmask = (const uint32_t*)kmask_f; p.kmask_words = (int)tp_kblock_mask_words((int64_t)d->r * d->s * d->cin);
  for (int r = 0; r < d->r; ++r) for (int s = 0; s < d->s; ++s) {
    TapEntry& t = p.taps[r * d->s + s];
    t.off_w = (uint16_t)s; t.off_h = (uint16_t)r; t.kofs = (r * d->s + s) * d->cin;
  }
  AMaps ta; CUtensorMap tb;
  if (is_plain_gemm(d)) {
    p.a_mode = 0;
    rc = make_tiled_map(&ta.m[0], x, (uint64_t)d->cin, (uint64_t)p.M, (uint64_t)d->cin, kBlockM); if (rc) return rc;
  } else {
    p.a_mode = 1;
    ce.base_w = -d->pad_w; ce.base_h = -d->pad_h; p.step_w = d->stride_w; p.step_h = d->stride_h;
    rc = make_im2col_map(&ta.m[0], x, d->n, d->h, d->w, d->cin, ce.base_w, ce.base_h, p.step_w, p.step_h, d->p, d->q, kBlockM);
    if (rc) return rc;
  }
  for (int c = 1; c < kMaxCls; ++c) ta.m[c] = ta.m[0];
  const int bn = pick_block_n((p.M + kBlockM - 1) / kBlockM, p.N);
  rc = make_tiled_map(&tb, wf, (uint64_t)d->r * d->s * d->cin, (uint64_t)d->cout, (uint64_t)d->r * d->s * d->cin, (uint32_t)bn);
  if (rc) return rc;
  return run_fwd(ta, tb, p, bn, st);
}

struct BnGate { const void* y; const float* weight; const float* bias; const float* mean; const float* invstd; float* partial; };

static int conv_dgrad_impl(const tp_conv_desc* d, const void* dy, const void* wd, const void* kmask_d, const void* addend,
                           void* dx, const BnGate* gate, void* stream);

int tp_conv_dgrad(const tp_conv_desc* d, const void* dy, const void* wd, const void* kmask_d, const void* addend,
                  void* dx, void* ws, size_t ws_bytes, void* stream) {
  (void)ws; (void)ws_bytes;
  return conv_dgrad_impl(d, dy, wd, kmask_d, addend, dx, nullptr, stream);
}

int tp_conv_dgrad_bnrelu(const tp_conv_desc* d, const void* dy, const void* wd, const void* kmask_d,
                         const void* bn_y, const void* bn_weight, const void* bn_bias, const void* bn_mean, const void* bn_invstd,
                         void* g, void* partial, void* stream) {
  if (!d || !bn_y || !bn_mean || !bn_invstd || !partial) return TP_ERR_INVALID;
  if (d->stride_h != 1 || d->stride_w != 1 || d->cin % 8 != 0) return TP_ERR_UNSUPPORTED;
  if ((((uintptr_t)bn_y) | ((uintptr_t)bn_weight) | ((uintptr_t)bn_bias) | ((uintptr_t)bn_mean) | ((uintptr_t)bn_invstd) | ((uintptr_t)partial)) & 15)
    return TP_ERR_UNSUPPORTED;
  BnGate bn = {bn_y, (const float*)bn_weight, (const float*)bn_bias, (const float*)bn_mean, (const float*)bn_invstd, (float*)partial};
  return conv_dgrad_impl(d, dy, wd, kmask_d, nullptr, g, &bn, stream);
}

size_t tp_conv_dgrad_partial_rows(const tp_conv_desc* d) {
  if (!d) return 0;
  const long long M = (long long)d->n * d->h * d->w;
  return (size_t)((M + kBlockM - 1) / kBlockM) * 4;
}

static int conv_dgrad_impl(const tp_conv_desc* d, const void* dy, const void* wd, const void* kmask_d, const void* addend,
                           void* dx, const BnGate* gate, void* stream) {
  if (!d || !dy || !wd || !dx) return TP_ERR_INVALID;
  // here the contraction runs over (r', s', cout): channel count of dY must be TMA friendly
  const int cop = d->cout;                       // caller passes dY with cout % 8 == 0 (padded if needed)
  if (cop % 8 != 0 || d->r * d->s > kMaxTaps) return TP_ERR_UNSUPPORTED;
  if (d->r * d->s > 1 && cop % 64 != 0) return TP_ERR_UNSUPPORTED;
  int rc = load_driver_fns(); if (rc) return rc;
  rc = bind_device_of(d ? (const void*)dy : nullptr); if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int R = d->r, S = d->s;
  const long long ktot = (long long)R * S * cop;
  const int sh = d->stride_h, sw = d->stride_w;
  FwdParams p = {};
  p.N = d->cin;
  p.cchunks = (cop + 63) / 64;
  p.out_img_pix = (long long)d->h * d->w; p.out_row_pix = d->w;
  p.ldc = d->cin; p.out = (__nv_bfloat16*)dx; p.bias = nullptr; p.addend = (const __nv_bfloat16*)addend;
  p.kmask = (const uint32_t*)kmask_d; p.kmask_words = (int)tp_kblock_mask_words(ktot);
  p.step_w = 1; p.step_h = 1;
  if (gate) {
    p.bn_y = (const __nv_bfloat16*)gate->y; p.bn_weight = gate->weight; p.bn_bias = gate->bias; p.bn_mean = gate->mean; p.bn_invstd = gate->invstd;
    p.stats = gate->partial;
  }
  AMaps ta; CUtensorMap tb;
  if (sh == 1 && sw == 1) {
    // dX = conv(dY, rot180(W)^T) with padding (R-1-pad): wd is stored already rotated
    p.M = d->n * d->h * d->w;
    p.ncls = 1; p.osh = 1; p.osw = 1;
    ClsEntry& ce = p.cls[0];
    ce.M = p.M; ce.P_it = d->h; ce.Q_it = d->w; ce.ntaps = R * S; ce.tap0 = 0; ce.oah = 0; ce.oaw = 0;
    for (int r = 0; r < R; ++r) for (int s = 0; s < S; ++s) {
      TapEntry& t = p.taps[r * S + s];
      t.off_w = (uint16_t)s; t.off_h = (uint16_t)r; t.kofs = (r * S + s) * cop;
    }
    if (is_plain_gemm(d)) {
      p.a_mode = 0;
      rc = make_tiled_map(&ta.m[0], dy, (uint64_t)cop, (uint64_t)p.M, (uint64_t)cop, kBlockM); if (rc) return rc;
    } else {
      p.a_mode = 1;
      ce.base_w = -(S - 1 - d->pad_w); ce.base_h = -(R - 1 - d->pad_h);
      rc = make_im2col_map(&ta.m[0], dy, d->n, d->p, d->q, cop, ce.base_w, ce.base_h, 1, 1, d->h, d->w, kBlockM);
      if (rc) return rc;
    }
    for (int c = 1; c < kMaxCls; ++c) ta.m[c] = ta.m[0];
  } else {
    // strided conv: dX splits into stride_h x stride_w parity classes; each class is a stride-1 gather over dY with its
    // own subset of taps, written to every stride-th pixel.  ONE launch covers all classes (round 1: a memset / memcpy
    // of dX plus one launch per class with scattered 16-byte stores — 2.5-4x the roofline of these layers); a class
    // no tap reaches is written by the epilogue alone (the fused addend, or zero).
    if (sh * sw > kMaxCls || R * S > kMaxTaps) return TP_ERR_UNSUPPORTED;
    p.a_mode = 1; p.osh = sh; p.osw = sw;
    int nc = 0, nt = 0; long long Mtot = 0;
    for (int a = 0; a < sh; ++a) for (int b = 0; b < sw; ++b) {
      const int Hc = (d->h - a + sh - 1) / sh, Wc = (d->w - b + sw - 1) / sw;   // pixels of this class
      if (Hc <= 0 || Wc <= 0) continue;
      ClsEntry& ce = p.cls[nc];
      ce.M = d->n * Hc * Wc; ce.P_it = Hc; ce.Q_it = Wc; ce.oah = a; ce.oaw = b; ce.tap0 = nt; ce.ntaps = 0;
      // taps: input row h = sh*h' + a receives dY row p = h' + (a + pad - r)/sh when divisible
      int dh_min = 1 << 30, dw_min = 1 << 30;
      for (int r = 0; r < R; ++r) if ((a + d->pad_h - r) % sh == 0) dh_min = min(dh_min, (a + d->pad_h - r) / sh);
      for (int s = 0; s < S; ++s) if ((b + d->pad_w - s) % sw == 0) dw_min = min(dw_min, (b + d->pad_w - s) / sw);
      if (dh_min != (1 << 30) && dw_min != (1 << 30)) {
        for (int r = 0; r < R; ++r) {
          if ((a + d->pad_h - r) % sh != 0) continue;
          for (int s = 0; s < S; ++s) {
            if ((b + d->pad_w - s) % sw != 0) continue;
            TapEntry& t = p.taps[nt++];
            t.off_h = (uint16_t)((a + d->pad_h - r) / sh - dh_min);
            t.off_w = (uint16_t)((b + d->pad_w - s) / sw - dw_min);
            t.kofs = ((R - 1 - r) * S + (S - 1 - s)) * cop;          // wd stores tap (r,s) at rotated position (R-1-r, S-1-s)
            ++ce.ntaps;
          }
        }
      } else { dh_min = 0; dw_min = 0; }
      ce.base_w = dw_min; ce.base_h = dh_min;
      rc = make_im2col_map(&ta.m[nc], dy, d->n, d->p, d->q, cop, ce.base_w, ce.base_h, 1, 1, Hc, Wc, kBlockM); if (rc) return rc;
      Mtot += ce.M; ++nc;
    }
    if (nc == 0) return TP_OK;
    for (int c = nc; c < kMaxCls; ++c) ta.m[c] = ta.m[0];
    p.ncls = nc; p.M = (int)Mtot;
  }
  long long m_tiles = 0;
  for (int c = 0; c < p.ncls; ++c) m_tiles += (p.cls[c].M + kBlockM - 1) / kBlockM;
  const int bn = pick_block_n(m_tiles, p.N);
  rc = make_tiled_map(&tb, wd, (uint64_t)ktot, (uint64_t)d->cin, (uint64_t)ktot, (uint32_t)bn); if (rc) return rc;
  return run_fwd(ta, tb, p, bn, st);
}

int tp_conv_wgrad(const tp_conv_desc* d, const void* x, const void* dy, const void* mask, const void* kmask_f,
                  int cin_real, void* dw, void* db, void* ws, size_t ws_bytes, void* stream) {
  if (!d || !x || !dy || !mask || !dw || !ws) return TP_ERR_INVALID;
  if (d->cin % 8 != 0 || d->cout % 8 != 0 || d->r * d->s > kMaxTaps || cin_real > d->cin) return TP_ERR_UNSUPPORTED;
  if (d->r * d->s > 1 && d->cin % 64 != 0) return TP_ERR_UNSUPPORTED;
  int rc = load_driver_fns(); if (rc) return rc;
  rc = bind_device_of(d ? (const void*)x : nullptr); if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int rs = d->r * d->s;
  WgParams p = {};
  p.Mc = d->cout;
  p.Kpix = d->n * d->p * d->q;
  p.P_it = d->p; p.Q_it = d->q;
  const int ktot = (rs * d->cin + 63) / 64 * 64;
  p.chunks = ktot / 64;
  p.cchunks = (d->cin + 63) / 64;
  p.nb = p.chunks >= 4 ? 4 : p.chunks;
  p.m_tiles = (d->cout + kBlockM - 1) / kBlockM;
  p.n_tiles = (p.chunks + p.nb - 1) / p.nb;
  p.kblocks = (p.Kpix + 63) / 64;
  const int sms = sm_count();
  int splits = pick_wgrad_splits(p.m_tiles * p.n_tiles, p.kblocks, p.nb);
  p.kb_per_split = (p.kblocks + splits - 1) / splits;
  splits = (p.kblocks + p.kb_per_split - 1) / p.kb_per_split;     // no empty splits
  p.splits = splits;
  const size_t need = (size_t)p.m_tiles * p.n_tiles * splits * kBlockM * p.nb * 64 * sizeof(float);
  if (ws_bytes < need) return TP_ERR_WORKSPACE;
  p.partial = (float*)ws;
  p.kmask = (const uint32_t*)kmask_f; p.kmask_words = (int)tp_kblock_mask_words((int64_t)rs * d->cin);
  for (int r = 0; r < d->r; ++r) for (int s = 0; s < d->s; ++s) {
    TapEntry& t = p.taps[r * d->s + s];
    t.off_w = (uint16_t)s; t.off_h = (uint16_t)r; t.kofs = (r * d->s + s) * d->cin;
  }
  CUtensorMap ta, tb;
  rc = make_tiled_map(&ta, dy, (uint64_t)d->cout, (uint64_t)p.Kpix, (uint64_t)d->cout, 64); if (rc) return rc;
  if (is_plain_gemm(d)) {
    p.b_mode = 0;
    rc = make_tiled_map(&tb, x, (uint64_t)d->cin, (uint64_t)p.Kpix, (uint64_t)d->cin, 64); if (rc) return rc;
  } else {
    p.b_mode = 1;
    p.base_w = -d->pad_w; p.base_h = -d->pad_h; p.step_w = d->stride_w; p.step_h = d->stride_h;
    rc = make_im2col_map(&tb, x, d->n, d->h, d->w, d->cin, p.base_w, p.base_h, p.step_w, p.step_h, d->p, d->q, 64);
    if (rc) return rc;
  }
  constexpr int smem = 4 * (kBlockM * kBlockK * 2 + 4 * 64 * kBlockK * 2) + 1024 + 256;
  static bool attr_set = false;
  if (!attr_set) {
    TP_CUDA_CHECK(cudaFuncSetAttribute(k_igemm_wgrad, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_set = true;
  }
  const int items = p.m_tiles * p.n_tiles * splits;
  launch(k_igemm_wgrad, items < sms ? items : sms, kThreads, smem, st, ta, tb, p);
  TP_LAUNCH_CHECK();
  // split lanes only pay when there are many splits (skinny layers); wide-K layers keep all 256 threads on K
  const int sl = splits >= 64 ? 8 : (splits >= 32 ? 4 : (splits >= 16 ? 2 : 1));
  const int fin_kt = 256 / sl;
  launch(k_wgrad_finalize, dim3(d->cout, (rs * d->cin + fin_kt - 1) / fin_kt), 256, 0, st, 
      p.partial, (const float*)mask, (float*)dw, d->cout, cin_real, d->cin, rs, p.nb, p.m_tiles, p.n_tiles, splits, sl,
      p.kmask, p.kmask_words);
  TP_LAUNCH_CHECK();
  if (db) {
    // the split-K partials are dead once the finalize above has run (same stream): the workspace holds the column partials now
    const int c = d->cout, cv = c / 8;
    int tx = 1;
    while (tx < cv && tx < 256) tx <<= 1;
    const int ty = 256 / tx, ctiles = (cv + tx - 1) / tx;
    long long gx = ((long long)p.Kpix + (long long)ty * 4 - 1) / ((long long)ty * 4);          // >= 4 pixel rows per thread
    const long long want = (long long)sms * 4 / ctiles, fit = (long long)(ws_bytes / ((size_t)c * sizeof(float)));
    if (gx > want) gx = want;
    if (gx > fit) gx = fit;
    if (gx < 1) gx = 1;
    if ((((uintptr_t)dy) & 15) != 0) return TP_ERR_INVALID;
    launch(k_colsum_part, dim3((unsigned)gx, (unsigned)ctiles), dim3(tx, ty), 0, st, (const __nv_bfloat16*)dy, (long long)p.Kpix, c, c, (float*)ws);
    launch(k_colsum_fold, (c + 255) / 256, 256, 0, st, (const float*)ws, (int)gx, c, (float*)db);
    TP_LAUNCH_CHECK();
  }
  return TP_OK;
}

}  // extern "C"
