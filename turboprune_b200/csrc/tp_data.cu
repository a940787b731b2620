// Data path either side of the model (SURVEY.md §8(f) row 3), sm_100a, HBM-bound:
//
//   k_cifar_augment : the airbench-style GPU augmentation of the reference's CifarLoader.__iter__
//                     (utils/dataset.py:192-226): random translate = batch_crop of the reflect-padded images (:43-69),
//                     per-image left-right flip (:38-40) and cutout (:72-98), fused into ONE gather pass — the
//                     reference runs a masked-assignment loop over 2(2r+1) shifts, a where() and a masked_fill(), each a
//                     full pass.  The random draws (shifts, flip mask, cutout corners) stay torch's: their RNG stream is
//                     part of the parity contract, exactly like set_er_mask.
//   k_cifar_epoch   : a whole CifarLoader epoch from the uint8 NHWC data set in one launch: normalisation, the epoch-0
//                     pre-flip, translate (reflect padding as index arithmetic), flip, cutout and the epoch's shuffle.
//                     One CTA per output image; the source image's bytes cross L2 -> SM once (16-byte cp.async into a
//                     double-buffered shared-memory stage), normalisation is a per-CTA table of the C x 256 byte values,
//                     the fp32 NCHW output leaves as whole 128-byte lines of float4 stores.
//   k_synth_normal / k_synth_labels : the synthetic on-device generator standing in for FFCV / the CIFAR tensors
//                     (no data sets here): counter-based Philox4x32-10 -> Box-Muller, four values per counter, written
//                     with 16-byte stores straight into the batch buffer (N(0,1) images — FFCV hands over
//                     mean/std-normalised fp32, dataset.py:391 — and uniform int64 labels).
#include "tp_common.cuh"

namespace tp {

// out[n][c][y][x] = cut(n, y, x) ? 0 : src[n][c][y + r + sy[n]][xf + r + sx[n]],  xf = flip[n] ? W-1-x : x
// src is [N][C][H+2r][W+2r] (r = 0 and no shifts: plain flip / cutout); every array of draws is optional.
__global__ void __launch_bounds__(256) k_cifar_augment(const float* __restrict__ src, float* __restrict__ out,
                                                       const long long* __restrict__ shifts, const unsigned char* __restrict__ flip,
                                                       const long long* __restrict__ cut_y, const long long* __restrict__ cut_x,
                                                       int cut_size, int N, int C, int H, int W, int r) {
  const int Hp = H + 2 * r, Wp = W + 2 * r;
  const long long total = (long long)N * C * H * W;
  for (long long i = blockIdx.x * 256ll + threadIdx.x; i < total; i += (long long)gridDim.x * 256) {
    const int x = (int)(i % W); long long t = i / W;
    const int y = (int)(t % H); t /= H;
    const int c = (int)(t % C); const int n = (int)(t / C);
    float v = 0.f;
    bool cut = false;
    if (cut_y) {
      const long long dy = y - cut_y[n], dx = x - cut_x[n];
      cut = dy >= 0 && dy < cut_size && dx >= 0 && dx < cut_size;
    }
    if (!cut) {
      const int sy = shifts ? (int)shifts[2 * n] : 0, sx = shifts ? (int)shifts[2 * n + 1] : 0;
      const int xf = (flip && flip[n]) ? W - 1 - x : x;
      v = src[(((long long)n * C + c) * Hp + (y + r + sy)) * Wp + (xf + r + sx)];
    }
    out[i] = v;
  }
}

// ---- one CIFAR epoch straight from the uint8 data set (CifarLoader.__iter__, utils/dataset.py:192-226) -----------------
// The reference normalises the whole set once (images / 255 -> sub_(mean) -> div_(std)), pre-flips it, reflect-pads it,
// then every epoch crops, flips, cuts out and gathers each batch: a dozen full passes.  Here output image j is built from
// source image i = perm[j] in one pass, the reflect padding being index arithmetic on the unpadded source.  A byte's
// normalised value depends only on (byte, channel): each CTA tabulates the C x 256 values once in shared memory, so a pixel
// is two shared-memory loads.  The next image's bytes are copied into the second of two staging buffers (cp.async) while
// the current one is written out.
constexpr int kEpochThreads = 256;
constexpr int kEpochMaxC = 4;
constexpr int kEpochMaxImageBytes = 20 * 1024;            // 256*C*4 + 2 staging buffers stay under the default 48 KiB

struct EpochNorm { float mean[kEpochMaxC], std[kEpochMaxC]; };

// p in [-(n-1), 2n-2]: the index F.pad(..., "reflect") reads for padded position p + r
__device__ __forceinline__ int reflect_index(int p, int n) { return p < 0 ? -p : (p >= n ? 2 * (n - 1) - p : p); }

// the reference's arithmetic on CUDA, one rounding per step like torch's separate kernels: images / 255 is ATen's
// CUDA true-divide by a CPU scalar, i.e. a multiply by the fp32 reciprocal; Normalize's sub_ / div_ take tensor operands
__device__ __forceinline__ float cifar_normalize(unsigned int u, float mean, float std) {
  return __fdiv_rn(__fsub_rn(__fmul_rn((float)u, 1.0f / 255.0f), mean), std);
}

// copy one source image into shared memory: 16-byte cp.async when aligned (completes at the next wait_group), else bytes
__device__ __forceinline__ void stage_image(unsigned char* dst, const unsigned char* s, int bytes, bool vec) {
  if (vec) {
    for (int q = threadIdx.x; q < bytes / 16; q += kEpochThreads)
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;"
                   :: "r"((unsigned)__cvta_generic_to_shared(dst + 16 * q)), "l"(s + 16 * q) : "memory");
  } else {
    for (int q = threadIdx.x; q < bytes; q += kEpochThreads) dst[q] = s[q];
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}

__global__ void __launch_bounds__(kEpochThreads) k_cifar_epoch(
    const unsigned char* __restrict__ src, const long long* __restrict__ labels, float* __restrict__ out,
    long long* __restrict__ labels_out, const long long* __restrict__ perm, const long long* __restrict__ shifts,
    const unsigned char* __restrict__ preflip, const unsigned char* __restrict__ flip, int flip_all,
    const long long* __restrict__ cut_y, const long long* __restrict__ cut_x, int cut_size, EpochNorm norm,
    int N, int C, int H, int W) {
  extern __shared__ __align__(16) unsigned char smem[];
  const int bytes = H * W * C, stage = (bytes + 15) & ~15;
  float* lut = reinterpret_cast<float*>(smem);                  // [C][256] normalised value of each byte
  unsigned char* const buf = smem + C * 256 * 4;                // two staging buffers of one source image, [H][W][C]
  const int hw = H * W;
  const bool vec_in = (bytes & 15) == 0 && (((uintptr_t)src) & 15) == 0;
  const bool vec_out = (W & 3) == 0 && (((uintptr_t)out) & 15) == 0;
#pragma unroll
  for (int c = 0; c < kEpochMaxC; ++c)                           // unrolled: the parameter struct is indexed by constants
    if (c < C)
      for (int u = threadIdx.x; u < 256; u += kEpochThreads) lut[c * 256 + u] = cifar_normalize(u, norm.mean[c], norm.std[c]);
  int j = blockIdx.x;
  if (j < N) stage_image(buf, src + (long long)(perm ? perm[j] : j) * bytes, bytes, vec_in);
  for (int it = 0; j < N; j += gridDim.x, ++it) {
    const int i = perm ? (int)perm[j] : j;
    const int jn = j + gridDim.x;
    if (jn < N) {
      stage_image(buf + ((it + 1) & 1) * stage, src + (long long)(perm ? perm[jn] : jn) * bytes, bytes, vec_in);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    if (labels && threadIdx.x == 0) labels_out[j] = labels[i];
    const int sy = shifts ? (int)shifts[2 * i] : 0, sx = shifts ? (int)shifts[2 * i + 1] : 0;
    const bool pre = preflip && preflip[i];
    const bool fin = flip_all || (flip && flip[i]);
    const int cy = cut_y ? (int)cut_y[i] : 0, cx = cut_x ? (int)cut_x[i] : 0;
    const int csz = cut_y ? cut_size : 0;
    __syncthreads();                                              // image `it` and the table are in shared memory
    const unsigned char* img = buf + (it & 1) * stage;
    float* o = out + (long long)j * C * hw;
    // output pixel (c, y, x) <- source byte (reflect(y + sy), reflect(x1 + sx), c), x1 = fin ? W-1-x : x, the column
    // mirrored again when the image was pre-flipped; zero inside the cutout square
    auto pixel = [&](int c, int y, int x, int yy) -> float {
      if (y - cy >= 0 && y - cy < csz && x - cx >= 0 && x - cx < csz) return 0.f;
      int xx = reflect_index((fin ? W - 1 - x : x) + sx, W);
      if (pre) xx = W - 1 - xx;
      return lut[(c << 8) + img[(yy * W + xx) * C + c]];
    };
    if (vec_out) {
      const int w4 = W >> 2;
      for (int q = threadIdx.x; q < C * H * w4; q += kEpochThreads) {
        const int x = (q % w4) << 2, t = q / w4, y = t % H, c = t / H;
        const int yy = reflect_index(y + sy, H);
        float4 v;
        v.x = pixel(c, y, x, yy); v.y = pixel(c, y, x + 1, yy); v.z = pixel(c, y, x + 2, yy); v.w = pixel(c, y, x + 3, yy);
        st_stream(reinterpret_cast<float4*>(o + ((long long)c * H + y) * W + x), v);
      }
    } else {
      for (int q = threadIdx.x; q < C * hw; q += kEpochThreads) {
        const int x = q % W, t = q / W, y = t % H, c = t / H;
        o[q] = pixel(c, y, x, reflect_index(y + sy, H));
      }
    }
    __syncthreads();                                              // this buffer is restaged in the next iteration
  }
}

// ---- Philox4x32-10 (Salmon et al., SC'11): counter (ctr, 0, 0, 0) with key (seed_lo, seed_hi) --------------------------
__device__ __forceinline__ void philox4x32_10(unsigned long long ctr, unsigned long long seed, unsigned int (&o)[4]) {
  unsigned int c0 = (unsigned int)ctr, c1 = (unsigned int)(ctr >> 32), c2 = 0u, c3 = 0u;
  unsigned int k0 = (unsigned int)seed, k1 = (unsigned int)(seed >> 32);
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const unsigned int hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const unsigned int hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    const unsigned int n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  o[0] = c0; o[1] = c1; o[2] = c2; o[3] = c3;
}

// mode 0: raw 32-bit words (tests pin the stream against the oracle bit for bit); mode 1: N(0,1) by Box-Muller
__global__ void __launch_bounds__(256) k_synth_normal(float* __restrict__ out, long long n, unsigned long long seed,
                                                      unsigned long long offset, int mode) {
  const long long n4 = (n + 3) >> 2;
  for (long long q = blockIdx.x * 256ll + threadIdx.x; q < n4; q += (long long)gridDim.x * 256) {
    unsigned int u[4];
    philox4x32_10(offset + (unsigned long long)q, seed, u);
    float f[4];
    if (mode == 0) {
#pragma unroll
      for (int j = 0; j < 4; ++j) f[j] = __uint_as_float(u[j]);
    } else {
      // (0, 1] uniforms from the top 24 bits; two Box-Muller pairs
      const float inv = 1.0f / 16777216.0f;
#pragma unroll
      for (int j = 0; j < 4; j += 2) {
        const float u1 = ((float)(u[j] >> 8) + 1.0f) * inv, u2 = (float)(u[j + 1] >> 8) * inv;
        const float rad = sqrtf(-2.0f * logf(u1));
        float sn, cs; sincospif(2.0f * u2, &sn, &cs);
        f[j] = rad * cs; f[j + 1] = rad * sn;
      }
    }
    if (4 * q + 3 < n && (((uintptr_t)out) & 15) == 0) {
      st_stream((float4*)out + q, make_float4(f[0], f[1], f[2], f[3]));
    } else {
      for (int j = 0; j < 4; ++j) if (4 * q + j < n) out[4 * q + j] = f[j];
    }
  }
}

__global__ void __launch_bounds__(256) k_synth_labels(long long* __restrict__ out, long long n, int num_classes,
                                                      unsigned long long seed, unsigned long long offset) {
  const long long n4 = (n + 3) >> 2;
  for (long long q = blockIdx.x * 256ll + threadIdx.x; q < n4; q += (long long)gridDim.x * 256) {
    unsigned int u[4];
    philox4x32_10(offset + (unsigned long long)q, seed, u);
    for (int j = 0; j < 4; ++j)
      if (4 * q + j < n) out[4 * q + j] = (long long)(((unsigned long long)u[j] * (unsigned long long)num_classes) >> 32);
  }
}

}  // namespace tp

using namespace tp;

extern "C" {

int tp_cifar_augment(const void* src, void* out, const int64_t* shifts, const uint8_t* flip,
                     const int64_t* cut_y, const int64_t* cut_x, int cut_size,
                     int n, int c, int h, int w, int r, void* stream) {
  if (!src || !out || n <= 0 || c <= 0 || h <= 0 || w <= 0 || r < 0) return TP_ERR_INVALID;
  if ((cut_y == nullptr) != (cut_x == nullptr) || (cut_y && cut_size <= 0)) return TP_ERR_INVALID;
  if (shifts && r == 0) return TP_ERR_INVALID;
  const long long total = (long long)n * c * h * w;
  const long long g = (total + 255) / 256, gm = (long long)sm_count() * 16;
  k_cifar_augment<<<(unsigned)(g < gm ? g : gm), 256, 0, (cudaStream_t)stream>>>(
      (const float*)src, (float*)out, (const long long*)shifts, (const unsigned char*)flip,
      (const long long*)cut_y, (const long long*)cut_x, cut_size, n, c, h, w, r);
  TP_LAUNCH_CHECK();
  return TP_OK;
}

int tp_cifar_epoch(const uint8_t* src, const int64_t* labels, void* out, int64_t* labels_out, const int64_t* perm,
                   const int64_t* shifts, int r, const uint8_t* preflip, const uint8_t* flip, int flip_all,
                   const int64_t* cut_y, const int64_t* cut_x, int cut_size, const float* mean, const float* std,
                   int n, int c, int h, int w, void* stream) {
  if (!src || !out || !mean || !std || n <= 0 || c <= 0 || c > kEpochMaxC || h <= 0 || w <= 0) return TP_ERR_INVALID;
  if ((long long)h * w * c > kEpochMaxImageBytes) return TP_ERR_INVALID;
  if ((labels == nullptr) != (labels_out == nullptr)) return TP_ERR_INVALID;
  if (r < 0 || r >= h || r >= w || (shifts && r == 0)) return TP_ERR_INVALID;         // reflect padding needs r < h, w
  if (flip && flip_all) return TP_ERR_INVALID;
  if ((cut_y == nullptr) != (cut_x == nullptr)) return TP_ERR_INVALID;
  if (cut_y && (cut_size <= 0 || cut_size > h || cut_size > w)) return TP_ERR_INVALID;
  EpochNorm norm{};
  for (int k = 0; k < c; ++k) { norm.mean[k] = mean[k]; norm.std[k] = std[k]; }
  const int smem = c * 256 * 4 + 2 * ((h * w * c + 15) & ~15);
  const int g = n < sm_count() * 8 ? n : sm_count() * 8;
  k_cifar_epoch<<<g, kEpochThreads, smem, (cudaStream_t)stream>>>(
      src, (const long long*)labels, (float*)out, (long long*)labels_out, (const long long*)perm, (const long long*)shifts,
      preflip, flip, flip_all ? 1 : 0, (const long long*)cut_y, (const long long*)cut_x, cut_size, norm, n, c, h, w);
  TP_LAUNCH_CHECK();
  return TP_OK;
}

int tp_synth_normal(void* out, int64_t numel, uint64_t seed, uint64_t counter_offset, int raw_words, void* stream) {
  if (!out || numel < 0) return TP_ERR_INVALID;
  if (numel == 0) return TP_OK;
  const long long g = ((numel + 3) / 4 + 255) / 256, gm = (long long)sm_count() * 16;
  k_synth_normal<<<(unsigned)(g < gm ? g : gm), 256, 0, (cudaStream_t)stream>>>((float*)out, numel, seed, counter_offset, raw_words ? 0 : 1);
  TP_LAUNCH_CHECK();
  return TP_OK;
}

int tp_synth_labels(void* out, int64_t numel, int num_classes, uint64_t seed, uint64_t counter_offset, void* stream) {
  if (!out || numel < 0 || num_classes <= 0) return TP_ERR_INVALID;
  if (numel == 0) return TP_OK;
  const long long g = ((numel + 3) / 4 + 255) / 256, gm = (long long)sm_count() * 8;
  k_synth_labels<<<(unsigned)(g < gm ? g : gm), 256, 0, (cudaStream_t)stream>>>((long long*)out, numel, num_classes, seed, counter_offset);
  TP_LAUNCH_CHECK();
  return TP_OK;
}

}  // extern "C"
