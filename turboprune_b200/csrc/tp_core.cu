// Error plumbing, device cache and the segment-table upload shared by all kernels.
#include "tp_common.cuh"
#include <stdlib.h>
#include <string.h>
#include <vector>

namespace tp {

static thread_local char g_last_err[512] = "";

void set_last_cuda_error(cudaError_t e, const char* where) {
  snprintf(g_last_err, sizeof(g_last_err), "%s: %s (%s)", where, cudaGetErrorName(e), cudaGetErrorString(e));
}

static int g_pdl = -1;
bool pdl_enabled() {
  // measured (profiles/r02_notes.md, experiment 9): per-GPU batch 64: 7.68 -> 7.58 ms per step; batch 512: 42.14 -> 42.74 ms.
  // Opt-in (TP_PDL=1 or tp_set_pdl(1)) until the trigger placement is tuned per kernel.
  if (g_pdl < 0) { const char* e = getenv("TP_PDL"); g_pdl = (e && e[0] == '1') ? 1 : 0; }
  return g_pdl == 1;
}

int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

typedef int (*PFN_cuCtxGetCurrent)(void**);
static PFN_cuCtxGetCurrent g_ctx_get_current = nullptr;

int bind_device_of(const void* p) {
  if (!p) return TP_OK;
  // Fast path (and the only path taken while a CUDA graph is being captured): a context is already
  // current on this thread — nothing to do, no runtime call.
  static bool looked_up = false;
  if (!looked_up) {
    void* fn = nullptr; cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuCtxGetCurrent", &fn, cudaEnableDefault, &q) == cudaSuccess) g_ctx_get_current = (PFN_cuCtxGetCurrent)fn;
    looked_up = true;
  }
  if (g_ctx_get_current) {
    void* ctx = nullptr;
    if (g_ctx_get_current(&ctx) == 0 && ctx != nullptr) return TP_OK;
  }
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return TP_OK; }
  if (a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged) {
    TP_CUDA_CHECK(cudaSetDevice(a.device));   // CUDA 12+: initialises and binds the primary context
  }
  return TP_OK;
}

int upload_segs(Arena& ar, const void* const* w, const void* const* g, const void* const* m,
                void* const* mo, void* const* buf, const int64_t* numel, int n_seg,
                Seg** dev_out, long long* tiles_out, long long* total_out, cudaStream_t st) {
  if (n_seg <= 0 || !numel) return TP_ERR_INVALID;
  std::vector<Seg> h(n_seg);
  long long start = 0, tile = 0;
  for (int i = 0; i < n_seg; ++i) {
    if (numel[i] < 0) return TP_ERR_INVALID;
    h[i].w = w ? (const float*)w[i] : nullptr;
    h[i].g = g ? (const float*)g[i] : nullptr;
    h[i].m = m ? (const float*)m[i] : nullptr;
    h[i].mo = mo ? (float*)mo[i] : nullptr;
    h[i].buf = buf ? (float*)buf[i] : nullptr;
    h[i].n = numel[i];
    h[i].start = start;
    h[i].tile0 = tile;
    start += numel[i];
    tile += (numel[i] + kTileElems - 1) / kTileElems;
  }
  Seg* d = (Seg*)ar.take(sizeof(Seg) * n_seg);
  if (!d) return TP_ERR_WORKSPACE;
  // pageable source: the runtime stages the bytes before returning, so `h` may die.
  TP_CUDA_CHECK(cudaMemcpyAsync(d, h.data(), sizeof(Seg) * n_seg, cudaMemcpyHostToDevice, st));
  *dev_out = d;
  if (tiles_out) *tiles_out = tile;
  if (total_out) *total_out = start;
  return TP_OK;
}

}  // namespace tp

extern "C" {

const char* tp_strerror(int code) {
  switch (code) {
    case TP_OK: return "ok";
    case TP_ERR_INVALID: return "invalid argument";
    case TP_ERR_WORKSPACE: return "workspace too small";
    case TP_ERR_CUDA: return "CUDA error (see tp_last_cuda_error)";
    case TP_ERR_K_RANGE: return "kthvalue(): selected number k out of range";
    case TP_ERR_UNSUPPORTED: return "unsupported configuration";
    case TP_ERR_DEVICE: return "device is not sm_100 (B200)";
    default: return "unknown error";
  }
}

const char* tp_last_cuda_error(void) { return tp::g_last_err; }
int tp_abi_version(void) { return 9; }
int tp_device_sm_count(void) { return tp::sm_count(); }
int tp_set_pdl(int on) { const int prev = tp::pdl_enabled() ? 1 : 0; tp::g_pdl = on ? 1 : 0; return prev; }

size_t tp_segtable_workspace_bytes(int n_seg) {
  return tp::align_up(sizeof(tp::Seg) * (size_t)(n_seg > 0 ? n_seg : 1), 256) + 256;
}

}  // extern "C"
