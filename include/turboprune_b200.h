/*
 * turboprune_b200 — C ABI of the B200-native (sm_100a) TurboPrune hot path.
 *
 * Plain C types only: device pointers as void*, sizes as int64_t / size_t, the CUDA
 * stream as an opaque void* (a cudaStream_t / CUstream; NULL = default stream).  No
 * torch or C++ types cross this boundary.  All device buffers are owned by the caller
 * (the Python host keeps them as torch tensors); nothing here allocates or frees device
 * memory except where a function says so.  Return value: 0 = ok, negative = error code
 * (see tp_strerror).  No exceptions cross the ABI.  Functions are re-entrant across
 * streams; the only global state is an init-once device-property / driver-entry cache.
 *
 * Each entry point cites the reference call site (relative to the TurboPrune repo) it
 * replaces.  The reference has no FFI of its own (pure Python); INTEGRATION.md shows the
 * ctypes binding a maintainer adds on the reference side.
 */
#ifndef TURBOPRUNE_B200_H
#define TURBOPRUNE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- error codes -------------------------------------------------------------------- */
#define TP_OK                 0
#define TP_ERR_INVALID       -1   /* bad argument (null pointer, negative size, unsupported shape) */
#define TP_ERR_WORKSPACE     -2   /* workspace too small: call the matching *_workspace_bytes */
#define TP_ERR_CUDA          -3   /* a CUDA runtime/driver call failed (see tp_last_cuda_error) */
#define TP_ERR_K_RANGE       -4   /* k out of [1, N] — torch.kthvalue raises for this (k == 0!) */
#define TP_ERR_UNSUPPORTED   -5   /* valid request this build does not implement */
#define TP_ERR_DEVICE        -6   /* not an sm_100 device */

const char* tp_strerror(int code);
const char* tp_last_cuda_error(void);      /* text of the last CUDA error seen by this thread */
int         tp_abi_version(void);          /* bumps when a signature changes */
int         tp_device_sm_count(void);      /* cached multiprocessor count of the current device */
/* Programmatic dependent launch for the train-step kernels (default off; TP_PDL=1 in the environment turns it on).
 * Returns the previous setting.  A debugging / A-B switch: results are bit-identical either way. */
int         tp_set_pdl(int on);

/* ---- score kinds (utils/pruning_utils.py) ------------------------------------------- */
#define TP_SCORE_MAG      0   /* |m*w|      prune_mag :75, prune_random_* :109-116 (w := randn draw) */
#define TP_SCORE_SNIP     1   /* |(g*w)*m|  prune_snip :190 */
#define TP_SCORE_SYNFLOW  2   /* |(m*g)*w|  prune_synflow :267 */

/* ---- pruning: score -> exact global k-th smallest -> mask ----------------------------
 * Replaces, in one call, utils/pruning_utils.py:73-87 (prune_mag), :186-203 (prune_snip),
 * :263-283 (prune_synflow): per-layer score, torch.cat, torch.kthvalue(k), torch.where.
 *
 *   w, g, m, mask_out : HOST arrays of n_seg DEVICE pointers (fp32; g may be NULL for
 *                       TP_SCORE_MAG; mask_out[i] may alias nothing else; it may be NULL
 *                       as a whole to only compute the threshold)
 *   numel             : HOST array of n_seg element counts
 *   k                 : 1-indexed rank, k = int((1-density)*N) computed by the caller in
 *                       float64 exactly as the reference does; k < 1 or k > N -> TP_ERR_K_RANGE
 *   thr_out           : DEVICE float — the k-th smallest score (bit-exact torch.kthvalue)
 *   new mask          : mask_out[i][j] = score <= thr ? 0.f : 1.f   (ties pruned)
 *   info_out          : optional HOST int64[4] = {path (0 bracketed single sweep, 1 exact
 *                       3-pass radix fallback), candidates, n_lt, nan_threshold}
 * The call synchronises the stream once (it has to learn whether the fast path held); see tp_topk_enqueue /
 * tp_topk_finish for the non-blocking form.
 */
size_t tp_topk_workspace_bytes(int n_seg, int64_t total_numel);
int tp_topk_threshold_mask(const void* const* w, const void* const* g, const void* const* m,
                           void* const* mask_out, const int64_t* numel, int n_seg,
                           int64_t k, int score_kind, float* thr_out,
                           void* ws, size_t ws_bytes, int64_t* info_out, void* stream);
/* The same call split in two, for callers that must not block the stream (benchmarks, a pruning step queued behind
 * other work): tp_topk_enqueue issues the whole fast path — one memset and ONE cooperative kernel (sample, bracket,
 * sweep, resolve, patch, see csrc/tp_prune.cu) — and returns without synchronising; tp_topk_finish synchronises,
 * reads the status back and, only if the bracket missed (adversarial ties) or the threshold is NaN, runs the exact
 * radix fallback / the all-ones apply pass.  Masks and thr_out must not be consumed before tp_topk_finish returned.
 * table_cached != 0: `ws` still holds the segment table uploaded by an earlier call with identical pointers (no
 * host->device copy; w / g may then be NULL).  Both take the same numel / n_seg / k / score_kind / ws. */
int tp_topk_enqueue(const void* const* w, const void* const* g, const void* const* m,
                    void* const* mask_out, const int64_t* numel, int n_seg,
                    int64_t k, int score_kind, float* thr_out,
                    void* ws, size_t ws_bytes, int table_cached, void* stream);
int tp_topk_finish(const void* const* m, void* const* mask_out, const int64_t* numel, int n_seg,
                   int64_t k, int score_kind, float* thr_out,
                   void* ws, size_t ws_bytes, int64_t* info_out, void* stream);

/* mask_out = score <= *thr ? 0 : 1 with a caller-supplied DEVICE threshold
 * (utils/pruning_utils.py:84-87,140-143).  thr semantics follow fp32 compare: a NaN
 * threshold keeps everything. */
int tp_apply_threshold(const void* const* w, const void* const* g, const void* const* m,
                       void* const* mask_out, const int64_t* numel, int n_seg,
                       int score_kind, const float* thr, void* ws, size_t ws_bytes, void* stream);

/* zeros_out[i] = #(m[i] == 0) for every segment plus zeros_out[n_seg] = total, one launch,
 * no host sync (utils/custom_models.py:51-62 does 54 .item() syncs).  zeros_out: DEVICE int64[n_seg+1]. */
int tp_count_zeros(const void* const* m, const int64_t* numel, int n_seg,
                   int64_t* zeros_out, void* ws, size_t ws_bytes, void* stream);

/* ---- weight staging: fp32 (mask*w) -> bf16 tensor-core operand layouts ------------------
 * Replaces the per-forward `mask * weight` (utils/mask_layers.py:25,69,109) and the autocast
 * fp32->bf16 cast of the product: one pass writes
 *   wf [Cout][R][S][Cin_p]  (fprop  B operand, K-major, K = (r,s,ci))  and optionally
 *   wd [Cin_p2][R][S][Cout_p] with taps rotated by 180 deg (dgrad B operand, K = (r,s,co)).
 * w, mask: fp32 OIHW [Cout][Cin][R][S].  Cin_p / Cout_p: channel counts padded (zero filled).
 */
int tp_stage_weights(const void* w, const void* mask, int cout, int cin, int r, int s,
                     void* wf, int cin_p, int wf_ld, void* wd, int cout_p, int cin_p2,
                     void* kmask_f, void* kmask_d, void* stream);
/* K-block occupancy masks ("skip all-zero tiles", BASELINE.json north_star; the reference multiplies the dense
 * mask*weight every forward, utils/mask_layers.py:25-34).  For every group of 64 ROWS of a staged operand (wf: output
 * channels; wd: input channels) a bitmask over its 64-column K blocks: bit b of word (b / 32) is set when the 64 x 64 block
 * holds a non-zero masked weight.  kmask_f: uint32 [ceil(cout/64)][tp_kblock_mask_words(wf_ld)] + 1, kmask_d: uint32
 * [ceil(cin/64)][tp_kblock_mask_words(r*s*cout_p)] + 1; the trailing element is the number of EMPTY blocks (zero lets the
 * GEMM kernels drop the per-block test entirely); both optional (NULL = not produced); the staging call zeroes and fills
 * them.  tp_conv_fprop_stats / tp_conv_dgrad skip a K block (no TMA load, no MMA) when it is empty for every row group
 * of their output-channel tile; results are bit-identical to the dense walk for finite activations (a skipped block only
 * ever adds +-0). */
size_t tp_kblock_mask_words(int64_t columns);
/* wf_ld: elements between consecutive rows of wf (0 = dense, R*S*cin_p); columns past R*S*cin_p are the caller's
 * zero padding (the 7x7x3 stem GEMM runs with K = 152 for 147 real columns). */

/* The same staging for MANY layers in one launch (the bf16 "weight shadow" refreshed once per optimizer step —
 * SURVEY.md §8(f) row 2; replaces the per-layer mul + cast launches K1/K2 of mask_layers.py:25-34).
 * wf / wd are persistent buffers owned by the caller, zero-initialised once (channel padding is never rewritten);
 * wd may be NULL (layer without an input gradient).  table_cached != 0: `ws` still holds the table uploaded by an
 * earlier call with identical items — no host->device copy, so the call can be captured into a CUDA graph. */
typedef struct tp_stage_item {
  const void* w; const void* mask;   /* fp32 OIHW [cout][cin][r][s] */
  void* wf; void* wd;                /* bf16 [cout][r*s*cin_p], bf16 [cin][r*s*cout_p] or NULL */
  int32_t cout, cin, r, s, cin_p, cout_p, wf_ld;   /* wf_ld: 0 = dense */
  void* kmask_f; void* kmask_d;      /* K-block occupancy masks of wf / wd (NULL = not produced); inside kmask_all */
} tp_stage_item;
size_t tp_stage_batched_workspace_bytes(int n_items);
/* kmask_all / kmask_bytes: the one buffer all items' occupancy masks live in (zeroed here by a single memset; may be NULL) */
int tp_stage_weights_batched(const tp_stage_item* items, int n_items, int table_cached, void* kmask_all, size_t kmask_bytes,
                             void* ws, size_t ws_bytes, void* stream);

/* NCHW/NHWC fp32 or bf16 activation -> NHWC bf16 with channels padded to c_pad (zero fill).
 * src_dtype: 0 = fp32, 1 = bf16.  Strides in elements. */
int tp_to_nhwc_bf16(const void* src, int src_dtype, int64_t sn, int64_t sc, int64_t sh, int64_t sw,
                    int n, int c, int h, int w, void* dst, int c_pad, void* stream);

/* Explicit im2col for inputs with 8 (padded) channels — the 3-channel stem conv, whose rows are
 * too narrow for a 128-byte TMA row.  x: NHWC bf16 [n][h][w][8]; xcol: [n*p*q][kp] bf16 with
 * column (r*S+s)*8 + c, zero for columns >= r*s*8; kp % 8 == 0, kp >= r*s*8.  The stem conv then runs as a
 * plain GEMM (1x1 tp_conv_desc with cin = kp) through tp_conv_fprop / tp_conv_wgrad. */
int tp_im2col_c8(const void* x, int n, int h, int w, int r, int s, int stride_h, int stride_w,
                 int pad_h, int pad_w, int p, int q, void* xcol, int kp, void* stream);

/* The expansion straight from the framework's input tensor (src_dtype 0 = fp32, 1 = bf16; element strides; c <= 8):
 * the precision/layout conversion is fused in, no NHWC intermediate exists.  cg (c <= cg <= 8) = channels per tap:
 * column (r*S+s)*cg + ch, zero for ch >= c and for columns >= r*s*cg; kp % 8 == 0, kp >= r*s*cg.  The RGB stem uses
 * cg = 3: K = 152 instead of 392 columns. */
int tp_im2col_stem(const void* src, int src_dtype, int64_t sn, int64_t sc, int64_t sh, int64_t sw,
                   int n, int c, int h, int w, int r, int s, int cg, int stride_h, int stride_w, int pad_h, int pad_w,
                   int p, int q, void* xcol, int kp, void* stream);

/* ---- data path either side of the model (SURVEY.md §8(f) row 3) --------------------------
 * tp_cifar_augment: random translate (batch_crop of the reflect-padded images, utils/dataset.py:43-69), per-image
 * left-right flip (:38-40) and cutout (:72-98) of CifarLoader.__iter__ (:192-226) as ONE gather pass:
 *   out[n][c][y][x] = inside_cut(n,y,x) ? 0 : src[n][c][y + r + shifts[n][0]][xf + r + shifts[n][1]],  xf = flip[n] ? w-1-x : x
 * src fp32 [n][c][h+2r][w+2r] contiguous, out fp32 [n][c][h][w]; shifts int64 [n][2] in [-r, r] (NULL: no translate, then
 * r must describe the padding actually present, usually 0), flip uint8 [n] (NULL: none), cut_y / cut_x int64 [n] top-left
 * corners of a cut_size square (both NULL: none).  The draws are the caller's (torch RNG, reference order). */
int tp_cifar_augment(const void* src, void* out, const int64_t* shifts, const uint8_t* flip,
                     const int64_t* cut_y, const int64_t* cut_x, int cut_size,
                     int n, int c, int h, int w, int r, void* stream);
/* tp_cifar_epoch: one epoch of CifarLoader.__iter__ (utils/dataset.py:192-226) straight from the data set as stored,
 * src uint8 [n][h][w][c] (c <= 4, h*w*c <= 20 KiB), into out fp32 [n][c][h][w] contiguous and labels_out int64 [n]:
 *   i = perm ? perm[j] : j;  x1 = (flip_all || flip[i]) ? w-1-x : x;  yy = refl(y + shifts[i][0]);  xx = refl(x1 + shifts[i][1])
 *   xx = preflip[i] ? w-1-xx : xx;   out[j][ch][y][x] = inside_cut(i,y,x) ? 0 : (src[i][yy][xx][ch] * (1/255) - mean[ch]) / std[ch]
 *   labels_out[j] = labels[i]
 * refl(-1) = 1, refl(h) = h-2 (F.pad reflect); each arithmetic step rounds once, as torch's separate CUDA kernels do.
 * Every array but src / out is optional: perm int64 [n] (NULL: identity), shifts int64 [n][2] in [-r, r] with 0 < r < h, w
 * (NULL: no translate), preflip / flip uint8 [n] (NULL: none; flip_all != 0 flips every image and excludes flip),
 * cut_y / cut_x int64 [n] corners of a cut_size square (both NULL: none), labels / labels_out (both or neither).
 * mean / std are HOST arrays of c floats.  All NULL: the normalised set in stored order (the test loader). */
int tp_cifar_epoch(const uint8_t* src, const int64_t* labels, void* out, int64_t* labels_out, const int64_t* perm,
                   const int64_t* shifts, int r, const uint8_t* preflip, const uint8_t* flip, int flip_all,
                   const int64_t* cut_y, const int64_t* cut_x, int cut_size, const float* mean, const float* std,
                   int n, int c, int h, int w, void* stream);
/* Synthetic batches (stand-in for the FFCV / CIFAR loaders, which need data sets): Philox4x32-10, counter
 * (counter_offset + i/4, 0, 0, 0), key = seed; element i takes word i%4.  tp_synth_normal writes N(0,1) fp32 (Box-Muller
 * on 24-bit uniforms; raw_words != 0: the 32-bit words themselves, for bit-exact pinning of the stream);
 * tp_synth_labels writes int64 labels floor(word * num_classes / 2^32). */
int tp_synth_normal(void* out, int64_t numel, uint64_t seed, uint64_t counter_offset, int raw_words, void* stream);
int tp_synth_labels(void* out, int64_t numel, int num_classes, uint64_t seed, uint64_t counter_offset, void* stream);

/* ---- masked implicit-GEMM convolution / linear on tcgen05 tensor cores -----------------
 * Replaces F.conv2d / F.linear / F.conv1d(k=1) on the masked weight
 * (utils/mask_layers.py:26-34, :70, :110-118) and their autograd backward.
 * Activations are NHWC bf16 (channels_last), accumulation fp32 in TMEM.
 *
 * tp_conv_desc describes one convolution; linear layers are 1x1 convs with H = W = 1.
 */
typedef struct tp_conv_desc {
  int32_t n, h, w, cin;          /* input  [n, h, w, cin]  (cin = padded channel count, %8 == 0) */
  int32_t cout, r, s;            /* filter [cout, r, s, cin] */
  int32_t stride_h, stride_w, pad_h, pad_w;
  int32_t p, q;                  /* output [n, p, q, cout] */
} tp_conv_desc;

size_t tp_conv_workspace_bytes(const tp_conv_desc* d, int op);   /* op: 0 fprop, 1 dgrad, 2 wgrad */

/* y[n,p,q,cout] (bf16) = conv(x[n,h,w,cin] (bf16), wf (bf16, tp_stage_weights layout)) + bias */
int tp_conv_fprop(const tp_conv_desc* d, const void* x, const void* wf, const void* bias_f32,
                  void* y, void* ws, size_t ws_bytes, void* stream);
/* Same, and the epilogue also writes BatchNorm batch statistics of the bf16 outputs it stores: for every group of 32
 * output pixels one row [2][cout] fp32 = (sum, sum of squares) per channel; stats holds tp_conv_stats_rows(d) rows
 * (rows past the last pixel are written as zeros).  Consumed by tp_bn_forward_ext — the BatchNorm2d that follows
 * the convolution (torchvision graph built at utils/custom_models.py:184) then needs no statistics pass. */
size_t tp_conv_stats_rows(const tp_conv_desc* d);
int tp_conv_fprop_stats(const tp_conv_desc* d, const void* x, const void* wf, const void* kmask_f, const void* bias_f32,
                        void* y, void* stats, void* ws, size_t ws_bytes, void* stream);
/* dx[n,h,w,cin] (bf16) = conv_dgrad(dy[n,p,q,cout] (bf16), wd (bf16, rotated layout)) [+ addend[n,h,w,cin]]
 * addend (optional, bf16, same layout as dx): the gradient arriving over a skip connection, accumulated in the
 * epilogue instead of by a separate elementwise add (autograd's grad accumulation at a ResNet block input). */
int tp_conv_dgrad(const tp_conv_desc* d, const void* dy, const void* wd, const void* kmask_d, const void* addend,
                  void* dx, void* ws, size_t ws_bytes, void* stream);
/* The same dgrad when dx is the gradient of a BatchNorm+ReLU output z = relu(bn(y)) without residual (the bn1 / bn2 of a
 * torchvision block feeding conv2 / conv3, custom_models.py:184): the epilogue writes g = dx * [z > 0] (gate recomputed
 * from y with the forward's own expression) and, per group of 32 pixels and channel, sum(g) and sum(g * xhat) —
 * partial holds tp_conv_dgrad_partial_rows(d) rows of [2][cin] fp32.  tp_bn_backward_ext then needs no reduction pass over
 * the activation.  Stride-1 convolutions only; bn_weight / bn_bias may be NULL (affine = False). */
size_t tp_conv_dgrad_partial_rows(const tp_conv_desc* d);
int tp_conv_dgrad_bnrelu(const tp_conv_desc* d, const void* dy, const void* wd, const void* kmask_d,
                         const void* bn_y, const void* bn_weight, const void* bn_bias, const void* bn_mean, const void* bn_invstd,
                         void* g, void* partial, void* stream);
/* dw[cout][cin_real][r][s] (fp32, OIHW) = mask * conv_wgrad(x, dy); db[cout] = sum dy (optional).
 * kmask_f (optional): the fprop occupancy mask tp_stage_weights produced for THIS mask (a block is marked occupied as soon
 * as one mask entry under it is non-zero): 128-channel x 256-column output tiles whose blocks are all empty are neither
 * computed nor read back, their gradient is written as zero — the result is the dense walk's, bit for bit. */
int tp_conv_wgrad(const tp_conv_desc* d, const void* x, const void* dy, const void* mask, const void* kmask_f,
                  int cin_real, void* dw, void* db, void* ws, size_t ws_bytes, void* stream);

/* tp_bn_forward with the batch statistics supplied by the producing convolution (tp_conv_fprop_stats):
 * ext_stats [ext_rows][2][C] fp32 un-shifted sums; training must be non-zero.  ext_stats == NULL: identical to
 * tp_bn_forward. */
int tp_bn_forward_ext(const void* y, const void* residual, void* z, int64_t M, int C,
                      const void* weight, const void* bias, void* running_mean, void* running_var,
                      void* num_batches_tracked, float momentum, float eps, int training, int relu,
                      void* save_mean, void* save_invstd, const void* ext_stats, int64_t ext_rows,
                      void* ws, size_t ws_bytes, void* stream);

/* ---- fused BatchNorm (+ residual add) (+ ReLU) on NHWC bf16 activations ------------------
 * SURVEY.md §8(f) row 1: the unmasked torchvision BatchNorm2d / ReLU / `out += identity` ops between
 * the masked convolutions (module graph built at utils/custom_models.py:184, run inside
 * harness_definitions/base_harness.py:124,127).  y, residual, z, dz, dy, dres: bf16 [M][C], C % 8 == 0.
 *   forward : z = [relu]( (y - mean) * invstd * weight + bias [+ residual] )
 *             training != 0: batch statistics (biased var), running stats updated with `momentum`
 *             (unbiased var), *num_batches_tracked += 1, save_mean / save_invstd written (fp32 [C]);
 *             training == 0: running statistics.
 *   backward: g = relu ? dz * gate : dz  (relu == 1: gate = z > 0 from the saved output; relu == 2: gate recomputed
 *             from y, weight, bias — z is not read);  dres = g (optional);  dweight = sum g*xhat; dbias = sum g;
 *             dy = weight*invstd * (g - mean(g) - xhat * mean(g*xhat))
 * Reductions use per-CTA partials folded in fixed order (deterministic).
 */
size_t tp_bn_workspace_bytes(int64_t m, int c);
int tp_bn_forward(const void* y, const void* residual, void* z, int64_t m, int c,
                  const void* weight, const void* bias, void* running_mean, void* running_var,
                  void* num_batches_tracked, float momentum, float eps, int training, int relu,
                  void* save_mean, void* save_invstd, void* ws, size_t ws_bytes, void* stream);
int tp_bn_backward(const void* dz, const void* z, const void* y, int64_t m, int c, const void* weight, const void* bias,
                   const void* save_mean, const void* save_invstd, int relu, void* dy, void* dres,
                   void* dweight, void* dbias, void* ws, size_t ws_bytes, void* stream);

/* Max pooling on NHWC bf16 (square window k, stride, symmetric padding with -inf, NaN propagates like
 * torch): forward writes y [n,p,q,c] and the uint8 arg-max window index idx [n,p,q,c]; backward gathers
 * dx [n,h,w,c] from dy through idx (deterministic, no atomics).  c % 8 == 0. */
/* tp_bn_backward for a gradient that already is g = dz * [z > 0] with its partial sums (tp_conv_dgrad_bnrelu):
 * fold, coefficients, apply pass dy = k0 g + k1 y + k2; dweight / dbias as in tp_bn_backward. */
int tp_bn_backward_ext(const void* g, const void* y, int64_t M, int C, const void* weight, const void* bias,
                       const void* save_mean, const void* save_invstd, const void* partial_rows, int64_t n_rows,
                       void* dy, void* dweight, void* dbias, void* ws, size_t ws_bytes, void* stream);
int tp_maxpool_forward(const void* x, void* y, void* idx, int n, int h, int w, int c, int k, int stride, int pad,
                       int p, int q, void* stream);
int tp_maxpool_backward(const void* dy, const void* idx, void* dx, int n, int h, int w, int c, int k, int stride, int pad,
                        int p, int q, void* stream);

/* ---- optimizer ------------------------------------------------------------------------
 * torch.optim.SGD(momentum, weight_decay) as configured at
 * harness_definitions/standard_pruning_harness.py:70-75, one launch for all segments:
 *   g += wd*w; buf = first ? g : mu*buf + g; w -= lr*buf     (masked weights keep decaying)
 * lr is read from a DEVICE float (so LR schedules do not re-record CUDA graphs).
 * table_cached != 0: `ws` still holds the segment table of an earlier call with identical pointers — no
 * host->device copy is issued, which makes the call capturable into a CUDA graph.
 */
int tp_sgd_momentum(void* const* w, const void* const* g, void* const* buf, const int64_t* numel,
                    int n_seg, const float* lr_dev, float momentum, float weight_decay,
                    int first_step, int table_cached, void* ws, size_t ws_bytes, void* stream);
size_t tp_segtable_workspace_bytes(int n_seg);

/* ---- gradient exchange over NVLink/NVSwitch peer memory ---------------------------------
 * Replaces the c10d Reducer's per-bucket  grad/W -> ncclAllReduce(SUM) -> copy back
 * (harness_definitions/base_harness.py:81) with one kernel: every rank reads its peers'
 * bucket copies directly over NVLink, sums them in fixed rank order (bit-identical on all
 * ranks), scales by `scale` (1/W), multiplies by an optional mask and writes `out`.
 *
 *   peer_bufs   : HOST array of `world` DEVICE pointers — the symmetric bucket buffer of
 *                 every rank as mapped into THIS process (peer_bufs[rank] is the local one)
 *   signal_pads : HOST array of `world` DEVICE pointers to uint32 signal pads (>= 4 KiB
 *                 each, zero-initialised once); used for the cross-GPU barriers
 *   mask        : optional fp32 mask in bucket layout (NULL = none)
 *   algo        : 0 = one-shot pull (every rank reads all W copies), 1 = two-shot
 *                 (reduce-scatter of shards + all-gather, via the same symmetric buffers)
 *   timeout_ms  : bounded spin on the barrier; on expiry the kernel sets *status_dev != 0
 *                 (optional DEVICE int) instead of hanging
 */
int tp_p2p_allreduce_mask(void* const* peer_bufs, void* const* signal_pads, int rank, int world,
                          int64_t numel, const void* mask, float scale, void* out,
                          int algo, int timeout_ms, int* status_dev, void* stream);

/* NVLS variant of the two-shot schedule: the reduction and the broadcast happen inside the NVSwitch.
 *   multicast_buf : DEVICE pointer — the multicast mapping of the same symmetric bucket (element 0 of the bucket's
 *                   data, e.g. torch symmetric memory's `multicast_ptr` + the signal-pad bytes); rank r issues
 *                   multimem.ld_reduce.add.v4.f32 on shard r, scales / masks, multimem.st's the result to all replicas.
 * Every replica receives the value rank r computed (replicas stay bit-identical); the switch, not this kernel,
 * fixes the order of the W-term sum, so against tp_p2p_allreduce_mask the result may differ in the last bit for W > 2.
 */
int tp_p2p_allreduce_nvls(void* const* peer_bufs, void* const* signal_pads, void* multicast_buf, int rank, int world,
                          int64_t numel, const void* mask, float scale, void* out,
                          int timeout_ms, int* status_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TURBOPRUNE_B200_H */
