// Host side of libqnnpack.so: the qnnpack.h C ABI implemented over the sm_100a kernels.
//
// Mirrors, entry point by entry point (reference paths relative to its root):
//   qnnp_initialize / qnnp_deinitialize          src/init.c:244-270
//   qnnp_create_convolution2d_nhwc_q8            src/convolution.c:39-378   (validation order, kernel choice :180-189)
//   qnnp_setup_convolution2d_nhwc_q8             src/convolution.c:380-492
//   qnnp_create/setup_fully_connected_nc_q8      src/fully-connected.c:25-161
//   qnnp_run_operator                            src/operator-run.c:639-844 (dwconv / gemm / conv cases)
//   qnnp_delete_operator                         src/operator-delete.c:15-28
// What changes: weights are packed for UMMA instead of for 4x4c2 SSE2 tiles (src/qnnpack/pack.h), no
// indirection buffer is ever built (src/indirection.c), run = one kernel launch on a CUDA stream.
// There is no CPU fallback: without a compute-capability-10.x device initialisation fails.
#include <cuda.h>
#include <cuda_runtime.h>
#include <math.h>
#include <pthread.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <initializer_list>
#include <new>
#include <vector>

#include "../../include/qnnpack.h"
#include "../../include/qnnpack_cuda.h"
#include "q8_dwconv_sm100.cuh"
#include "q8_eltwise_sm100.cuh"
#include "q8_igemm_sm100.cuh"
#include "requant_dev.cuh"

namespace q8 {
cudaError_t measure_int8_peak(int num_sms, int iters, int reps, cudaStream_t stream, double* tops, double* ms_out);
cudaError_t launch_q8_igemm(const IgemmParams& p, int mode, int vec, const void* tmap_a, const IgemmStoreMaps* store_maps,
                            int grid, int max_smem_optin, cudaStream_t stream);
cudaError_t launch_q8_gemm2sm(const IgemmParams& p, const void* tmap_a, const void* tmap_b, const IgemmStoreMaps& smaps, int clusters,
                              int max_smem_optin, cudaStream_t stream);
}

#define QNNP_EXPORT extern "C" __attribute__((visibility("default")))

namespace {

// ------------------------------------------------------------------------------------------------
// library state
// ------------------------------------------------------------------------------------------------
struct Library {
  bool initialized = false;
  enum qnnp_status init_status = qnnp_status_uninitialized;
  int device = -1;
  int num_sms = 0;
  int max_smem_optin = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  std::atomic<unsigned long long> launches{0};
  std::atomic<unsigned long long> dw_umma_launches{0};
  int32_t* dbg_acc = nullptr;
};
Library g_lib;
pthread_once_t g_once = PTHREAD_ONCE_INIT;

void log_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  fprintf(stderr, "Error in QNNPACK(b200): ");
  vfprintf(stderr, fmt, ap);
  fputc('\n', stderr);
  va_end(ap);
}

enum qnnp_status map_cuda(cudaError_t e, const char* what) {
  if (e == cudaSuccess) return qnnp_status_success;
  log_error("%s: %s", what, cudaGetErrorString(e));
  return e == cudaErrorMemoryAllocation ? qnnp_status_out_of_memory : qnnp_status_unsupported_hardware;
}

void init_once() {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    log_error("no CUDA device available (%s); this library has no CPU path", cudaGetErrorString(e));
    g_lib.init_status = qnnp_status_unsupported_hardware;
    return;
  }
  int dev = 0;
  const char* env = getenv("QNNP_CUDA_DEVICE");
  if (env != nullptr) {
    dev = atoi(env);
  } else if (cudaGetDevice(&dev) != cudaSuccess) {
    dev = 0;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, dev) != cudaSuccess || prop.major != 10) {
    log_error("device %d is not a compute-capability 10.x (B200-class) GPU", dev);
    g_lib.init_status = qnnp_status_unsupported_hardware;
    return;
  }
  if (cudaSetDevice(dev) != cudaSuccess ||
      cudaStreamCreateWithFlags(&g_lib.own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    g_lib.init_status = qnnp_status_unsupported_hardware;
    return;
  }
  g_lib.device = dev;
  g_lib.num_sms = prop.multiProcessorCount;
  g_lib.max_smem_optin = (int) prop.sharedMemPerBlockOptin;
  g_lib.stream = g_lib.own_stream;
  g_lib.initialized = true;
  g_lib.init_status = qnnp_status_success;
}

// The CUDA "current device" is per thread; callers may come from any thread.
void bind_device() {
  int cur = -1;
  if (cudaGetDevice(&cur) != cudaSuccess || cur != g_lib.device) cudaSetDevice(g_lib.device);
}

// cuTensorMapEncodeTiled through the runtime's driver-entry-point lookup (no link-time dependency on libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = []() -> EncodeTiledFn {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      return nullptr;
    return (EncodeTiledFn) p;
  }();
  return fn;
}

// Activation matrix [M][in_stride] (first K bytes of a row used) as {16 B of K, M rows, K/16 chunks}; box = {16, 128, skc}.
// sw32 != 0 (K % 32 == 0): 32-byte K slabs instead of 16-byte chunks — {32 B, M rows, K/32 slabs}, box {32, 128, skc/2},
// written with the 32-byte swizzle.  Same bytes at the same shared-memory offsets per (slab, row) block, but every 32-byte
// sector of the activations is requested from the L2 once instead of twice (see DESIGN.md §4.2 / §4.1).
bool make_tmap_a(CUtensorMap* tm, const uint8_t* in, size_t M, size_t in_stride, int K, int skc, int sw32) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (fn == nullptr) return false;
  if (sw32) {
    const cuuint64_t gdim[3] = {32, (cuuint64_t) M, (cuuint64_t) (K / 32)};
    const cuuint64_t gstride[2] = {(cuuint64_t) in_stride, 32};
    const cuuint32_t box[3] = {32, (cuuint32_t) q8::kTileM, (cuuint32_t) (skc / 2)};
    const cuuint32_t estride[3] = {1, 1, 1};
    return fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t*>(in), gdim, gstride, box, estride,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
  }
  const cuuint64_t gdim[3] = {16, (cuuint64_t) M, (cuuint64_t) (K / 16)};
  const cuuint64_t gstride[2] = {(cuuint64_t) in_stride, 16};
  const cuuint32_t box[3] = {16, (cuuint32_t) q8::kTileM, (cuuint32_t) skc};
  const cuuint32_t estride[3] = {1, 1, 1};
  return fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t*>(in), gdim, gstride, box, estride,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Output matrix [M][out_stride] (first N bytes of a row used) as a 2-D tensor {N, M} for the panel epilogue's stores:
// box = {width, rows}, shared-memory side swizzled to match the panel (width 128 / 64 / 32 bytes; 16: none).
bool make_tmap_out(void* tm, uint8_t* out, size_t M, size_t N, size_t out_stride, int width, int rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (fn == nullptr) return false;
  const cuuint64_t gdim[2] = {(cuuint64_t) N, (cuuint64_t) M};
  const cuuint64_t gstride[1] = {(cuuint64_t) out_stride};
  const cuuint32_t box[2] = {(cuuint32_t) width, (cuuint32_t) rows};
  const cuuint32_t estride[2] = {1, 1};
  const CUtensorMapSwizzle sw = width == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                             : width == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                                           : width == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  return fn((CUtensorMap*) tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, out, gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
            CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Row-major u8 matrix [rows][stride] (first K bytes of a row used) as a 2-D tensor {K, rows}; box = 128 bytes of K x 128
// rows, 128-byte swizzle: the K-major SWIZZLE_128B operand image of the CTA-pair GEMM.  Out-of-range bytes read zero.
bool make_tmap_kmajor_sw128(CUtensorMap* tm, const uint8_t* base, size_t rows, size_t K, size_t stride) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (fn == nullptr) return false;
  const cuuint64_t gdim[2] = {(cuuint64_t) K, (cuuint64_t) rows};
  const cuuint64_t gstride[1] = {(cuuint64_t) stride};
  const cuuint32_t box[2] = {128, 128};
  const cuuint32_t estride[2] = {1, 1};
  return fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t*>(base), gdim, gstride, box, estride,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

inline size_t round_up(size_t x, size_t q) { return (x + q - 1) / q * q; }
inline size_t ceil_div(size_t x, size_t q) { return (x + q - 1) / q; }
constexpr int kCtlReserve = 2048;  // static SmemCtl + 1024-byte alignment slack

// NHWC activations for the depthwise tensor-core kernel: stride 1 -> {C, W, H, N}; stride 2 -> {C, 2, W/2, H, N}
// (even/odd input columns become a dimension of their own, so each parity plane is one dense box).
// pair != 0: boxes of 32 channels (one full 32-byte sector per pixel and request) written with the 32-byte swizzle
bool make_tmap_dw(CUtensorMap* tm, const uint8_t* in, size_t N, size_t H, size_t W, size_t C, size_t in_stride, int s,
                  int box_px, int box_rows, int nb, int pair) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (fn == nullptr) return false;
  const cuuint32_t estride[5] = {1, 1, 1, 1, 1};
  const cuuint32_t cb = pair ? 32 : 16;
  const CUtensorMapSwizzle sw = pair ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  if (s == 1) {
    const cuuint64_t gdim[4] = {C, W, H, N};
    const cuuint64_t gstride[3] = {in_stride, W * in_stride, H * W * in_stride};
    const cuuint32_t box[4] = {cb, (cuuint32_t) box_px, (cuuint32_t) box_rows, (cuuint32_t) nb};
    return fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<uint8_t*>(in), gdim, gstride, box, estride,
              CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
  }
  const cuuint64_t gdim[5] = {C, 2, W / 2, H, N};
  const cuuint64_t gstride[4] = {in_stride, 2 * in_stride, W * in_stride, H * W * in_stride};
  const cuuint32_t box[5] = {cb, 1, (cuuint32_t) box_px, (cuuint32_t) box_rows, (cuuint32_t) nb};
  return fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 5, const_cast<uint8_t*>(in), gdim, gstride, box, estride,
            CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

inline int idiv_floor(int a, int b) { return (a >= 0) ? a / b : -((-a + b - 1) / b); }

// Border class bits of output position o along one axis (bit k: tap k lies inside [0, n)), as the depthwise epilogue computes them.
inline uint32_t dw_border_bits(int o, int s, int pad, int n) {
  const int i0 = o * s - pad;
  const int lo = i0 < 0 ? -i0 : 0, hi = i0 + 3 - n > 0 ? i0 + 3 - n : 0;
  return hi >= 3 ? 0u : (((7u << lo) & 7u) & (7u >> hi));
}

// Border-class biases of the depthwise tensor-core kernel (DwTcParams::bias_smem).  The epilogue reads 4 x 16 bytes of bias
// per unit; from the global table (64 classes x C int32: 147 KB at C = 576, far more than the L1 left beside the kernel's
// shared memory) those loads stall the requantisation — replacing them by a constant made 14x14x384 26 % and 7x7x960 23 %
// faster (profiles/r3a_dw_layers.txt).  A geometry produces only the row classes of its output rows times the column classes
// of its output columns (9 with padding <= 1 on images >= 3 pixels), so those rows of the table are copied into shared memory
// wherever they fit beside the plan's ring and resident weights.  QNNP_CUDA_DW_BIAS_GLOBAL=1 keeps the global table.
void plan_dw_bias_classes(q8::DwTcParams* p, int smem_limit) {
  p->bias_smem = 0, p->bias_off = 0, p->bias_rstride = 8, p->bias_nrc = 8, p->bias_ncc = 8;
  p->bias_rslot = p->bias_cslot = p->bias_rcls = p->bias_ccls = 0x76543210u;  // slot = class bits
  uint32_t rset = 0, cset = 0;  // bit b set: class bits b occur
  for (int oy = 0; oy < p->out_h; oy++) rset |= 1u << dw_border_bits(oy, p->stride, p->pad_top, p->in_h);
  for (int ox = 0; ox < p->out_w; ox++) cset |= 1u << dw_border_bits(ox, p->stride, p->pad_left, p->in_w);
  const int nrc = __builtin_popcount(rset), ncc = __builtin_popcount(cset);
  const int bytes = nrc * ncc * p->channels * 4;
  if (getenv("QNNP_CUDA_DW_BIAS_GLOBAL") != nullptr || p->smem_total + bytes > smem_limit) return;
  uint32_t rslot = 0, cslot = 0, rcls = 0, ccls = 0;  // unproduced classes: slot 0
  for (uint32_t b = 0, k = 0; b < 8; b++)
    if (rset & (1u << b)) rslot |= k << (4 * b), rcls |= b << (4 * k), k++;
  for (uint32_t b = 0, k = 0; b < 8; b++)
    if (cset & (1u << b)) cslot |= k << (4 * b), ccls |= b << (4 * k), k++;
  p->bias_smem = 1;
  p->bias_off = p->smem_total - 1024;  // behind everything the plan placed (smem_total includes the 1024-byte alignment slack)
  p->smem_total += bytes;
  p->bias_rstride = ncc, p->bias_nrc = nrc, p->bias_ncc = ncc;
  p->bias_rslot = rslot, p->bias_cslot = cslot, p->bias_rcls = rcls, p->bias_ccls = ccls;
}

// Tiling of the depthwise tensor-core kernel (q8_dwconv_umma_sm100.cu).  Pure function of the geometry, so that the
// CPU test can replay the smem addressing it prescribes.  Returns false when the shape is not eligible.
// pair != 0 plans the channel-pair form (see DwTcParams::pair); it needs a single weight operand (wmode != 2).
bool plan_dw_umma(int C, int batch, int H, int W, int OH, int OW, int s, int pad_top, int pad_left, int wmode, int smem_optin,
                  q8::DwTcParams* p, int pair = 0) {
  if (C <= 0 || (C % 16) != 0 || (s != 1 && s != 2) || (s == 2 && (W % 2) != 0) || pad_top > 2 || pad_left > 2) return false;
  if (batch <= 0 || OH <= 0 || OW <= 0) return false;
  if (pair && (wmode == 2 || C < 32)) return false;
  memset(p, 0, sizeof(*p));
  p->pair = pair ? 1 : 0;
  const int PB = pair ? 32 : 16;  // bytes of a pixel in a shared-memory plane
  p->batch = batch, p->channels = C, p->cgs = C / 16;
  p->in_h = H, p->in_w = W, p->out_h = OH, p->out_w = OW, p->stride = s, p->pad_top = pad_top, p->pad_left = pad_left;
  p->nb_cols = wmode == 2 ? 32 : 16;
  p->b_signed = wmode == 1 ? 0 : 1;
  // rows: either 16-row tiles of one image, or whole (short) images stacked, each padded to Q row groups
  const int rows_needed = s * (OH - 1) + 3;
  const int Qw = (rows_needed + s - 1) / s;
  p->whole = Qw <= 16 ? 1 : 0;
  if (p->whole) {
    // stack as many images as still have ALL their valid rows inside the UMMA's 16 row groups: image i occupies
    // groups [i*Q, i*Q + OH), the Q - OH groups after them are its bottom halo and produce nothing
    p->Q = Qw;
    p->nb = 1 + (16 - OH) / Qw;
    p->box_rows = s * Qw;
    p->yt = 1;
  } else {
    p->Q = 16;
    p->nb = 1;
    p->box_rows = 15 * s + 3;
    p->yt = (OH + 15) / 16;
  }
  p->nt = (batch + p->nb - 1) / p->nb;
  // columns: which plane and which plane-pixel offset each kernel column reads
  int par[3], dx[3], dxmin[2] = {1 << 20, 1 << 20};
  for (int kx = 0; kx < 3; kx++) {
    if (s == 1) {
      par[kx] = 0, dx[kx] = kx - pad_left;
    } else {
      par[kx] = ((kx - pad_left) % 2 + 2) % 2;
      dx[kx] = idiv_floor(kx - pad_left - par[kx], 2);
    }
    if (dx[kx] < dxmin[par[kx]]) dxmin[par[kx]] = dx[kx];
  }
  p->planes = s;
  for (int q = 0; q < 2; q++) p->x_org[q] = dxmin[q] == (1 << 20) ? 0 : dxmin[q];
  int xoff[3], xoff_max = 0;
  for (int kx = 0; kx < 3; kx++) {
    xoff[kx] = dx[kx] - p->x_org[par[kx]];
    if (xoff[kx] > xoff_max) xoff_max = xoff[kx];
  }
  // sub-tiles (mt) and channel groups (G) per item: mt * G units share an accumulator stage (256 TMEM columns) and are
  // what the 16 epilogue warps / 4 UMMA warps split among themselves, so narrow images take more channel groups.
  // G >= 2 whenever possible: the two 16-byte halves of every 32-byte sector are then moved by the same item.
  const int nsub = (OW + 7) / 8;
  const int umax = 256 / p->nb_cols;  // 8 (split operands) or 16 units
  const int smem_max = smem_optin - kCtlReserve - 1024;
  p->b_bytes = pair ? q8::kDwTcTaps32 * 2 * 32 * 16 : q8::kDwTcTaps * 2 * p->nb_cols * 16;
  // QNNP_CUDA_DW_MT / QNNP_CUDA_DW_G: A/B overrides of the tile search (measurement only)
  const int env_mt = getenv("QNNP_CUDA_DW_MT") != nullptr ? atoi(getenv("QNNP_CUDA_DW_MT")) : 0;
  const int env_g = getenv("QNNP_CUDA_DW_G") != nullptr ? atoi(getenv("QNNP_CUDA_DW_G")) : 0;
  // widest tile tried first.  Measured with 16 units per item (single weight operand), batch 4096: four sub-tiles x four
  // channel groups beat seven x two wherever the layer has >= 4 channel groups (56x56x144: 1.69 vs 2.01 ms — with four
  // sub-tiles an epilogue warp's units, 4 apart, all lie in the same sub-tile, so its column class is computed once per
  // item), while a 2-group layer needs the wide tile to fill the accumulator stage at all (112x112x32: 1.03 vs 1.19 ms)
  int cap0 = umax / 2 < 8 ? umax / 2 : 8;
  if (umax == 16 && p->cgs >= 4) cap0 = 4;
  // ... except, in the pair form, an ODD number of channel groups on a wide image: whole rows x one pair per item beat
  // 4 x 4 with its half-empty last block (56x56x144: 1.52 vs 1.63 ms)
  if (pair && umax == 16 && (p->cgs & 1) && p->cgs >= 5 && nsub > 4) cap0 = 8;
  if (env_mt >= 1 && env_mt <= cap0) cap0 = env_mt;
  for (int cap = cap0; cap >= 1 && p->mt == 0; cap--) {
    const int xt = (nsub + cap - 1) / cap;
    const int mt = (nsub + xt - 1) / xt;
    const int box_px = 8 * mt + xoff_max;
    if (box_px > 256 || p->box_rows > 256) continue;
    const int plane_tx = p->nb * p->box_rows * box_px * PB;
    // (pair mode: planes start on whole 256-byte swizzle atoms, so that the TMA's and the UMMA's pattern — both functions of
    // the absolute shared-memory address — agree wherever the box is placed)
    const int plane_bytes = (int) round_up(plane_tx, pair ? 256 : 128);
    const int a_bytes = p->planes * plane_bytes;
    const int cg_bytes = (int) round_up(a_bytes + p->b_bytes, pair ? 256 : 128);
    int G = umax / mt;
    if (env_g >= 1 && env_g < G) G = env_g;
    if (G > q8::kDwTcMaxG) G = q8::kDwTcMaxG;
    if (G > p->cgs) G = p->cgs + (pair ? (p->cgs & 1) : 0);
    if (pair) G &= ~1;  // whole channel pairs (an odd group count leaves the last pair half empty)
    for (; G >= 1; G -= (pair ? 2 : 1)) {
      const int stage_bytes = pair ? (G / 2) * cg_bytes : G * cg_bytes;
      int stages = smem_max / stage_bytes;
      if (stages > q8::kDwTcMaxStages) stages = q8::kDwTcMaxStages;
      if (stages < 3 && !(cap == 1 && G == 1 && stages >= 2)) continue;
      // prefer two channel groups per item over wider tiles (both 16-byte halves of every 32-byte sector move together,
      // and the units of an item occupy all four UMMA-issuing warps): a single group is accepted only at the narrowest tile
      if (G == 1 && p->cgs > 1 && cap > 1) continue;
      p->G = G, p->mt = mt, p->xt = xt, p->box_px = box_px, p->plane_tx = plane_tx, p->plane_bytes = plane_bytes;
      p->a_bytes = a_bytes, p->cg_bytes = cg_bytes, p->stage_bytes = stage_bytes, p->num_stages = stages;
      break;
    }
  }
  if (p->mt == 0) return false;
  p->cblocks = (p->cgs + p->G - 1) / p->G;
  p->smem_total = p->num_stages * p->stage_bytes + 1024;
  {
    // Resident weights: a channel block's B operands are the same for every spatial tile, yet they travelled with every
    // item's stage — 15 % of the bytes the kernel pulls from the L2 on the large images, 35-50 % on the 14x14 and 7x7 ones.
    // When the whole layer's blocks fit beside >= 3 ring stages they are loaded once per CTA instead.
    // (QNNP_CUDA_DW_B_STREAM=1 keeps them in the stages.)
    const int blocks_total = pair ? (p->cgs + 1) / 2 : p->cgs, blocks_item = pair ? p->G / 2 : p->G;
    const long long total_b = (long long) blocks_total * p->b_bytes;
    const int cg2 = p->a_bytes;  // (already a multiple of the plane alignment)
    const int stage2 = blocks_item * cg2;
    int stages2 = (int) ((smem_max - total_b) / (stage2 > 0 ? stage2 : 1));
    if (stages2 > q8::kDwTcMaxStages) stages2 = q8::kDwTcMaxStages;
    // Measured (batch 4096): a win wherever the blocks are >= 20 % of an item's bytes (14x14x384: 0.302 -> 0.272 ms) and in
    // the pair form (112x112x96 stride 2: 1.204 -> 1.163); with small blocks beside large tiles it LOSES 6 % (112x112x32,
    // 16-channel form: 0.909 -> 0.966), so it is not used there.
    const bool worth = pair || 4 * p->b_bytes >= p->a_bytes;
    if (total_b <= 160 * 1024 && stages2 >= 3 && worth && getenv("QNNP_CUDA_DW_B_STREAM") == nullptr) {
      p->b_resident = 1;
      p->cg_bytes = cg2, p->stage_bytes = stage2, p->num_stages = stages2;
      p->b_res_off = (int) round_up((size_t) stages2 * stage2, 256);
      p->smem_total = p->b_res_off + (int) total_b + 1024;
    }
  }
  p->sbo = s * p->box_px * PB;
  if ((p->sbo >> 4) > 0x3FFF) return false;
  if (pair)
    for (int ky = 0; ky < 3; ky++)
      for (int kx = 0; kx < 3; kx++) p->a_off9[ky * 3 + kx] = par[kx] * p->plane_bytes + (ky * p->box_px + xoff[kx]) * 32;
  // UMMA u multiplies two taps (K = 2 x 16 channels): (u,0)+(u,2) for kernel rows u = 0..2, (0,1)+(1,1), (2,1)+nothing
  const int t0[q8::kDwTcTaps][2] = {{0, 0}, {1, 0}, {2, 0}, {0, 1}, {2, 1}};
  const int t1[q8::kDwTcTaps][2] = {{0, 2}, {1, 2}, {2, 2}, {1, 1}, {2, 1}};
  for (int u = 0; u < q8::kDwTcTaps; u++) {
    const int a0 = par[t0[u][1]] * p->plane_bytes + (t0[u][0] * p->box_px + xoff[t0[u][1]]) * 16;
    const int a1 = par[t1[u][1]] * p->plane_bytes + (t1[u][0] * p->box_px + xoff[t1[u][1]]) * 16;
    if (a1 < a0 || ((a1 - a0) >> 4) > 0x3FFF) return false;
    p->a_off[u] = a0;
    p->a_lbo[u] = a1 - a0;
  }
  p->acc_stride = p->mt * p->G * p->nb_cols;
  p->acc_stages = 2;
  p->total_items = (long long) p->nt * p->yt * p->xt * p->cblocks;
  if (p->total_items >= (1ll << 31)) return false;
  plan_dw_bias_classes(p, smem_optin - kCtlReserve);
  return true;
}

// CTAs of a persistent kernel: one per SM, never more than there are work items.  QNNP_CUDA_MAX_CTAS=n shrinks the grid
// so that small test shapes still give every CTA many consecutive items (ring wrap-around, accumulator-stage parity,
// item stepping) — the parity tests run selected cases that way.
long long persistent_grid(long long total_items) {
  long long grid = total_items < g_lib.num_sms ? total_items : g_lib.num_sms;
  if (const char* e = getenv("QNNP_CUDA_MAX_CTAS")) {
    const long long v = atoll(e);
    if (v >= 1 && v < grid) grid = v;
  }
  return grid;
}

bool is_device_pointer(const void* ptr) {
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, ptr) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return attr.type == cudaMemoryTypeDevice || attr.type == cudaMemoryTypeManaged;
}


int pow2_align(uintptr_t v, int cap) {  // largest power of two <= cap dividing v (v == 0 -> cap)
  int a = cap;
  while (a > 1 && (v % (uintptr_t) a) != 0) a >>= 1;
  return a;
}

enum KernelKind {
  kKindNone = 0, kKindIgemmGemm, kKindIgemmConv, kKindDw3x3, kKindDirect,
  // operators beside the convolution path (q8_eltwise_sm100.cu)
  kKindAdd, kKindGavgPool, kKindAvgPool, kKindMaxPool, kKindClamp, kKindLut, kKindSoftargmax, kKindShuffle
};

}  // namespace

// ------------------------------------------------------------------------------------------------
// operator object (opaque to users; reference src/qnnpack/operator.h:39-102)
// ------------------------------------------------------------------------------------------------
struct qnnp_launch_plan;
void delete_plan(qnnp_launch_plan* p);

struct qnnp_operator {
  KernelKind kind = kKindNone;
  bool is_fc = false;

  // create-time
  uint32_t pad_top = 0, pad_right = 0, pad_bottom = 0, pad_left = 0;
  uint32_t kh = 1, kw = 1, stride_h = 1, stride_w = 1, dil_h = 1, dil_w = 1;
  uint32_t groups = 1;
  size_t gic = 0, goc = 0;
  uint8_t izp = 0, kzp = 0;
  Q8Requant rq{};
  int rq_mode = 3;

  // device-resident packed parameters
  void* d_weights = nullptr;   // igemm: UMMA blob; dw: int32 [9][c_pad]; direct: original kernel bytes
  size_t weights_bytes = 0;
  int32_t* d_bias = nullptr;   // folded bias
  size_t bias_count = 0;

  // igemm tiling
  int K = 0, nkc = 0, skc = 0, k_stages = 0, mt = 1, n_tiles = 0, n_tile = 0, n_mma = 0, has_corr = 1;
  int folded = 0, b_signed = 0, has_b2 = 0, bias_steps = 0, blk_chunks = 0, k_tail_pad = 0, smem_aconst_off = 0;
  int b_resident = 0, num_stages = 0, stage_bytes = 0;
  int smem_b_off = 0, smem_bias_off = 0, smem_a_off = 0, smem_stage_off = 0, staging_bytes = 0, smem_total = 0;
  bool bulk_capable = false;
  // CTA-pair GEMM (large weights): packed copy [n_tiles2][256 rows][K] (240 channels, ones row, zero rows) + folded biases
  uint8_t* d_w2 = nullptr;
  int32_t* d_bias2 = nullptr;
  int n_tiles2 = 0;
  int c_pad = 0;  // dw
  uint32_t* d_dw_wa = nullptr;  // dw streaming kernel: packed taps, operands A and B
  uint32_t* d_dw_wb = nullptr;
  int dw_wmode = 0;    // streaming depthwise kernel: 0 one s8 operand, 1 u8 (kzp == 0), 2 two s8 operands
  int dwtc_wmode = 0;  // tensor-core depthwise kernel: dw_tc_wmode()
  uint8_t* d_dwtc_w32 = nullptr;  // ... its channel-pair operands (pack_dw_umma32_host), when the single-operand form applies
  uint8_t* d_dwtc_w = nullptr;     // dw tensor-core kernel: block-diagonal B operands (null if channels % 16 != 0)
  int32_t* d_dwtc_bias = nullptr;  // dw tensor-core kernel: [64 border classes][channels]

  // setup-time
  size_t batch = 0, in_h = 0, in_w = 0, out_h = 0, out_w = 0;
  const uint8_t* input = nullptr;
  uint8_t* output = nullptr;
  size_t in_stride = 0, out_stride = 0;
  bool in_on_device = false, out_on_device = false;
  // element-wise / pooling operators
  bool is_deconv = false;        // kKindDirect: transposed convolution (src/deconvolution.c)
  uint32_t adj_h = 0, adj_w = 0; // deconvolution output adjustment
  size_t channels = 0;           // nc / nwc operators
  const uint8_t* input2 = nullptr;
  size_t in2_stride = 0;
  bool in2_on_device = false;
  uint8_t* d_in2 = nullptr;
  size_t d_in2_cap = 0;
  q8::AddParams add{};           // quantisation fields filled at create
  q8::AvgQuant avgq{};
  float in_scale = 0.f, out_scale = 0.f;
  uint8_t ozp = 0, omin = 0, omax = 255;
  uint8_t* d_lut = nullptr;      // 256-entry table (sigmoid, leaky ReLU)
  uint32_t* d_table32 = nullptr; // softargmax: 511 entries
  size_t in_span = 0, in2_span = 0, out_span = 0;  // bytes the operator reads / writes (host staging)
  bool out_dense = true;         // the output has no gaps between pixels / rows (else staging must preserve them)
  struct qnnp_launch_plan* plan = nullptr;  // cached launch state (built in setup / first run; see build_plan)
  // staging for host pointers
  uint8_t* d_in = nullptr;
  uint8_t* d_out = nullptr;
  size_t d_in_cap = 0, d_out_cap = 0;
};

namespace {

void free_operator(qnnp_operator* op) {
  if (op == nullptr) return;
  cudaFree(op->d_weights);
  cudaFree(op->d_bias);
  cudaFree(op->d_w2);
  cudaFree(op->d_bias2);
  cudaFree(op->d_dw_wa);
  cudaFree(op->d_dw_wb);
  cudaFree(op->d_dwtc_w);
  cudaFree(op->d_dwtc_w32);
  cudaFree(op->d_dwtc_bias);
  cudaFree(op->d_in);
  cudaFree(op->d_out);
  cudaFree(op->d_in2);
  cudaFree(op->d_lut);
  cudaFree(op->d_table32);
  delete_plan(op->plan);
  delete op;
}

int select_rq_mode(const Q8Requant& rq) { return q8_requant_mode(rq); }

// Every accumulator of the operator obeys |n| <= max|bias| + K * 255 * 255 (n = bias + sum (a - izp)(w - kzp)); with
// that bound the cheapest exact requantisation form ("U", requant_math.h) can be proven safe at create time.
void enable_bounded_requant(qnnp_operator* op, const int32_t* bias, size_t count, size_t K) {
  if (getenv("QNNP_CUDA_NO_URQ") != nullptr) return;
  int64_t bmax = 0;
  for (size_t i = 0; i < count; i++) {
    const int64_t b = bias[i] < 0 ? -(int64_t) bias[i] : (int64_t) bias[i];
    bmax = b > bmax ? b : bmax;
  }
  q8_requant_enable_u(op->rq, bmax + (int64_t) K * 255 * 255);
}

bool scale_ok(float s) { return s > 0.0f && isnormal(s); }

uint32_t f32_bits(float f) {
  uint32_t u;
  memcpy(&u, &f, sizeof u);
  return u;
}

// Folded bias: b + K*izp*kzp - izp*sum_k w   (src/qnnpack/pack.h:24,29,43 / :63,84 / :146,159), int32 wrap-around.
int32_t fold_bias(int32_t b, size_t k_total, uint8_t izp, uint8_t kzp, const uint8_t* w) {
  uint32_t wsum = 0;
  for (size_t i = 0; i < k_total; i++) wsum += w[i];
  return (int32_t) ((uint32_t) b + (uint32_t) k_total * (uint32_t) izp * (uint32_t) kzp - wsum * (uint32_t) izp);
}

// ------------------------------------------------------------------------------------------------
// igemm planning + packing
// ------------------------------------------------------------------------------------------------

// Tiling + shared-memory plan of the tensor-core kernel; pure function of the operator shape (testable on a CPU box).
struct IgemmPlan {
  int K, nkc, skc, k_stages, mt, n_tiles, n_tile, n_mma, has_corr;
  int folded, bias_steps, blk_chunks, k_tail_pad;
  int b_resident, num_stages, stage_bytes, staging_bytes, bias_bytes;
  int smem_b_off, smem_bias_off, smem_aconst_off, smem_a_off, smem_stage_off, smem_total;
  int bulk_capable;
  int good;  // 1 if the ring meets the in-flight target (>= 3 stages and >= 64 KB or 3 items' worth of K)
  size_t w_total, bias_count;
};

// folded != 0 requests the mode in which bias and zero-point correction are accumulated by extra UMMAs
// (needs the weights resident in smem; the function reports failure rather than silently changing mode).
bool plan_igemm(size_t K, size_t goc, uint32_t groups, int smem_optin, int folded, int bias_steps, IgemmPlan* pl) {
  memset(pl, 0, sizeof(*pl));
  pl->K = (int) K;
  pl->nkc = (int) round_up(ceil_div(K, 16), 2);
  pl->k_tail_pad = (K < (size_t) pl->nkc * 16) ? 1 : 0;
  pl->folded = folded ? 1 : 0;
  pl->bias_steps = folded ? bias_steps : 0;
  const int ones = folded ? 0 : q8::kOnesCols;
  const int n_tile_max = q8::kMaxNMma - ones;
  const int n_pad = (int) round_up(goc, 16);
  if (n_pad <= n_tile_max) {
    pl->n_tiles = 1;
    pl->n_tile = n_pad;
  } else {
    pl->n_tiles = (int) ceil_div(n_pad, n_tile_max);
    pl->n_tile = (int) round_up(ceil_div(n_pad, pl->n_tiles), 16);
  }
  pl->has_corr = folded ? 0 : 1;
  pl->n_mma = pl->n_tile + ones;
  pl->blk_chunks = pl->nkc + (folded ? 4 + 2 * bias_steps : 0);
  pl->bulk_capable = (groups == 1 && pl->n_tiles == 1 && (goc % 4) == 0) ? 1 : 0;
  pl->w_total = (size_t) groups * pl->n_tiles * pl->blk_chunks * pl->n_mma * 16;
  pl->bias_count = (size_t) groups * pl->n_tiles * pl->n_tile;
  pl->bias_bytes = (int) round_up(pl->bias_count * 4, 128);
  const int aconst_bytes = folded ? 2 * q8::kChunkBytes : 0;

  // Preference: as many 128-row sub-tiles per work item as TMEM allows (amortises per-item synchronisation),
  // subject to >= 3 ring stages and >= 64 KB of loads in flight (or the whole K of 3 items); weights stay
  // resident in smem when they fit beside that.
  const int smem_max = smem_optin - kCtlReserve - 1024;
  // sub-tiles per item: mt * n_mma <= 256 columns (two accumulator stages always fit the 512 TMEM columns; up to four
  // are used when the item is narrower).  Measured: larger items win — per-item hand-over costs dominate small ones.
  int mt_max = q8::kMaxNMma / pl->n_mma;
  if (mt_max < 1) mt_max = 1;
  if (mt_max > q8::kMaxSubTiles) mt_max = q8::kMaxSubTiles;
  if (mt_max < 1) mt_max = 1;
  if (const char* e = getenv("QNNP_CUDA_MAX_SUBTILES")) {
    const int v = atoi(e);
    if (v >= 1 && v < mt_max) mt_max = v;
  }
  // Candidates: every (mt, skc).  Feasible = >= 3 ring stages and >= 64 KB of loads in flight (or 3 whole items).
  // Among feasible plans minimise the synchronisation cost per 128-row tile, (1 + k_stages) / mt  — one item-level
  // hand-over plus one ring hand-over per K stage, amortised over mt sub-tiles — with >= 64 contiguous bytes per row
  // and stage (skc >= 4) so that global reads stay sector-efficient; ties go to the larger stage.
  struct Cand { int mt, skc, resident, stages, stage_bytes, staging; long long inflight; bool ok; double cost; };
  Cand best{0, 0, 0, 0, 0, 0, -1, false, 1e30};
  const int skc_min = pl->nkc < 4 ? pl->nkc : 4;
  for (int mt = mt_max; mt >= 1; mt--) {
    // per epilogue pair: the output tile of an item as column panels of n_tile bytes per row in total (panel epilogue),
    // which also covers the dense goc-pitch image of the 1-D bulk path (goc <= n_tile when there is one n-tile)
    const int staging = mt * q8::kTileM * pl->n_tile;
    for (int skc = pl->nkc; skc >= 2; skc -= 2) {
      if (skc > 16 && skc != pl->nkc && (skc % 8) != 0) continue;  // prune the search
      const int a_stage = mt * skc * q8::kChunkBytes;
      const long long fixed = pl->bias_bytes + aconst_bytes + 2LL * staging + 1024;  // (+ alignment of the staging base)
      const int resident = ((long long) pl->w_total + fixed + 3LL * a_stage <= smem_max) ? 1 : 0;
      if (folded && !resident) continue;
      const int stage_bytes = a_stage + (resident ? 0 : skc * pl->n_mma * 16);
      const long long room = smem_max - fixed - (resident ? (long long) pl->w_total : 0);
      int stages = room > 0 ? (int) (room / stage_bytes) : 0;
      if (stages > q8::kMaxStages) stages = q8::kMaxStages;
      if (stages < 2) continue;
      const long long inflight = (long long) stages * a_stage;
      const int k_stages = (int) ceil_div(pl->nkc, skc);
      const bool ok = stages >= 3 && skc >= skc_min && (inflight >= 64 * 1024 || stages >= 3 * k_stages);
      const double cost = (1.0 + k_stages) / mt - 1e-9 * stage_bytes;
      const bool better = (ok && !best.ok) || (ok == best.ok && (ok ? cost < best.cost : inflight > best.inflight));
      if (better) best = Cand{mt, skc, resident, stages, stage_bytes, staging, inflight, ok, cost};
    }
  }
  if (best.mt == 0) return false;
  pl->good = best.ok ? 1 : 0;
  pl->mt = best.mt;
  pl->skc = best.skc;
  pl->k_stages = (int) ceil_div(pl->nkc, pl->skc);
  pl->b_resident = best.resident;
  pl->num_stages = best.stages;
  pl->stage_bytes = best.stage_bytes;
  pl->staging_bytes = best.staging;
  pl->smem_b_off = 0;
  pl->smem_bias_off = (int) round_up(pl->b_resident ? pl->w_total : 0, 128);
  pl->smem_aconst_off = pl->smem_bias_off + pl->bias_bytes;
  pl->smem_a_off = pl->smem_aconst_off + aconst_bytes;
  pl->smem_stage_off = (int) round_up(pl->smem_a_off + pl->num_stages * pl->stage_bytes, 1024);  // swizzle atoms: 1024 B
  pl->smem_total = pl->smem_stage_off + 2 * pl->staging_bytes + 1024;
  return true;
}

// Folded-mode bias operand: bias' = 255 * Q + e with e in [-127, 127]; Q is spread over 31 signed digits per
// UMMA step (|digit| <= 127), so that  sum_k A[k] * digit[k]  with A = [255 x31, 1]  reproduces bias' exactly.
constexpr int kBiasDigitsPerStep = 31;
constexpr int kMaxBiasSteps = 4;

void bias_split(int32_t b, int64_t* q_out, int* e_out) {
  int64_t r = ((int64_t) b % 255 + 255) % 255;  // [0, 254]
  const int e = r <= 127 ? (int) r : (int) r - 255;
  *e_out = e;
  *q_out = ((int64_t) b - e) / 255;
}

int bias_steps_needed(int32_t b) {
  int64_t q;
  int e;
  bias_split(b, &q, &e);
  const int64_t aq = q < 0 ? -q : q;
  const int64_t per_step = (int64_t) kBiasDigitsPerStep * 127;
  const int64_t steps = (aq + per_step - 1) / per_step;
  return steps < 1 ? 1 : (steps > 1000000 ? 1000000 : (int) steps);
}

// Plans the tensor-core kernel for the operator and builds its packed operands in HOST memory (no CUDA call: the CPU test
// tests/test_igemm_pack.py replays the UMMA algebra on exactly these bytes).
enum qnnp_status pack_igemm_host(qnnp_operator* op, const uint8_t* kernel, const int32_t* bias, std::vector<uint8_t>& blob,
                                 std::vector<int32_t>& fbias) {
  const size_t ks = (size_t) op->kh * op->kw;
  const size_t K = ks * op->gic;
  if (K > (size_t) 1 << 24 || op->goc > (size_t) 1 << 24) {
    log_error("convolution too large for the tensor-core path (K=%zu, N=%zu)", K, op->goc);
    return qnnp_status_unsupported_parameter;
  }
  // folded biases first: their magnitude decides whether the tensor core can absorb them
  const size_t oc_all = (size_t) op->groups * op->goc;
  std::vector<int32_t> fb(oc_all);
  int steps = 1;
  for (size_t oc = 0; oc < oc_all; oc++) {
    fb[oc] = fold_bias(bias[oc], K, op->izp, op->kzp, kernel + oc * K);
    const int s = bias_steps_needed(fb[oc]);
    if (s > steps) steps = s;
  }
  const char* mode_env = getenv("QNNP_CUDA_IGEMM_MODE");
  // Folded mode removes two instructions per output from the (instruction-bound) epilogue at the price of 2-3x the
  // UMMA count; measured on B200 it wins when the layer writes more than it reads (N > K) and loses on the narrow
  // projection layers, where UMMA issue is the longer pole.  QNNP_CUDA_IGEMM_MODE=ones|folded overrides.
  bool want_folded = steps <= kMaxBiasSteps && op->goc > K;
  if (mode_env != nullptr && strcmp(mode_env, "ones") == 0) want_folded = false;
  if (mode_env != nullptr && strcmp(mode_env, "folded") == 0) want_folded = steps <= kMaxBiasSteps;
  IgemmPlan pl;
  // folded mode only when its plan keeps a healthy ring; otherwise the "ones" plan (weights may stream)
  const int optin = g_lib.initialized ? g_lib.max_smem_optin : 232448;  // B200: 227 KB opt-in (CPU-side planning/tests)
  bool planned = want_folded && plan_igemm(K, op->goc, op->groups, optin, 1, steps, &pl) && pl.good;
  if (!planned) planned = plan_igemm(K, op->goc, op->groups, optin, 0, 0, &pl);
  if (!planned) {
    log_error("shared-memory plan failed (K=%zu, N=%zu)", K, op->goc);
    return qnnp_status_unsupported_parameter;
  }
  op->K = pl.K, op->nkc = pl.nkc, op->skc = pl.skc, op->k_stages = pl.k_stages, op->mt = pl.mt;
  op->n_tiles = pl.n_tiles, op->n_tile = pl.n_tile, op->n_mma = pl.n_mma, op->has_corr = pl.has_corr;
  op->folded = pl.folded, op->bias_steps = pl.bias_steps, op->blk_chunks = pl.blk_chunks, op->k_tail_pad = pl.k_tail_pad;
  op->b_signed = (pl.folded && op->kzp != 0) ? 1 : 0;
  op->has_b2 = (pl.folded && op->kzp != 0) ? 1 : 0;
  op->b_resident = pl.b_resident, op->num_stages = pl.num_stages, op->stage_bytes = pl.stage_bytes;
  op->staging_bytes = pl.staging_bytes, op->bulk_capable = pl.bulk_capable != 0;
  op->smem_b_off = pl.smem_b_off, op->smem_bias_off = pl.smem_bias_off, op->smem_aconst_off = pl.smem_aconst_off;
  op->smem_a_off = pl.smem_a_off, op->smem_stage_off = pl.smem_stage_off, op->smem_total = pl.smem_total;
  const size_t w_total = pl.w_total, bias_count = pl.bias_count;

  // ---- pack: per (group, n_tile) block, chunk-major [chunk][row (n_mma)][16 B] -------------------------------
  //   chunks [0, nkc)            weights, K-major; "ones" mode: raw u8 + all-ones row n_tile;
  //                              folded mode: (w - 128) as s8 when kzp != 0, raw u8 when kzp == 0
  //   folded only:
  //   chunks [nkc, nkc+2)        constant (128 - kzp) operand, all 32 k valid
  //   chunks [nkc+2, nkc+4)      same, zero where the last chunk pair is K padding
  //   chunks [nkc+4+2t, +2)      bias digits of step t (k = 0..30: digits of Q, k = 31: e in step 0)
  blob.assign(w_total, 0);
  fbias.assign(bias_count, 0);
  const uint8_t wflip = op->b_signed ? 0x80 : 0x00;
  const uint8_t b2val = (uint8_t) (int8_t) (128 - (int) op->kzp);
  for (uint32_t g = 0; g < op->groups; g++) {
    for (int nt = 0; nt < op->n_tiles; nt++) {
      uint8_t* blk = blob.data() + ((size_t) g * op->n_tiles + nt) * op->blk_chunks * op->n_mma * 16;
      auto at = [&](size_t chunk, size_t row, size_t byte) -> uint8_t& { return blk[(chunk * op->n_mma + row) * 16 + byte]; };
      for (int r = 0; r < op->n_tile; r++) {
        const size_t oc = (size_t) nt * op->n_tile + r;
        if (oc >= op->goc) break;
        const uint8_t* wrow = kernel + ((size_t) g * op->goc + oc) * K;
        for (size_t k = 0; k < K; k++) at(k >> 4, r, k & 15) = wrow[k] ^ wflip;
        const int32_t b = fb[(size_t) g * op->goc + oc];
        fbias[((size_t) g * op->n_tiles + nt) * op->n_tile + r] = b;
        if (op->folded) {
          int64_t q;
          int e;
          bias_split(b, &q, &e);
          for (int t = 0; t < op->bias_steps; t++) {
            for (int k = 0; k < kBiasDigitsPerStep; k++) {
              const int64_t d = q > 127 ? 127 : (q < -127 ? -127 : q);
              q -= d;
              at(op->nkc + 4 + 2 * t + (k >> 4), r, k & 15) = (uint8_t) (int8_t) d;
            }
            at(op->nkc + 4 + 2 * t + 1, r, 15) = (uint8_t) (int8_t) (t == 0 ? e : 0);
          }
        }
      }
      if (op->folded) {
        if (op->has_b2) {
          const size_t k_last = (size_t) (op->nkc - 2) * 16;  // first k of the last chunk pair
          for (int r = 0; r < op->n_tile; r++)
            for (int k = 0; k < 32; k++) {
              at(op->nkc + (k >> 4), r, k & 15) = b2val;
              at(op->nkc + 2 + (k >> 4), r, k & 15) = (k_last + k < K) ? b2val : 0;
            }
        }
      } else {
        for (size_t k = 0; k < K; k++) at(k >> 4, op->n_tile, k & 15) = 1;
      }
    }
  }
  op->weights_bytes = w_total;
  op->bias_count = bias_count;
  return qnnp_status_success;
}

enum qnnp_status plan_and_pack_igemm(qnnp_operator* op, const uint8_t* kernel, const int32_t* bias) {
  std::vector<uint8_t> blob;
  std::vector<int32_t> fbias;
  const enum qnnp_status st = pack_igemm_host(op, kernel, bias, blob, fbias);
  if (st != qnnp_status_success) return st;
  cudaError_t e = cudaMalloc(&op->d_weights, blob.size());
  if (e == cudaSuccess) e = cudaMalloc((void**) &op->d_bias, fbias.size() * sizeof(int32_t));
  if (e == cudaSuccess) e = cudaMemcpy(op->d_weights, blob.data(), blob.size(), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(op->d_bias, fbias.data(), fbias.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
  // Weights that cannot stay resident in shared memory (large GEMMs): a second packing for the CTA-pair kernel
  // (q8_gemm2sm_kernel) — plain K-contiguous rows, so the TMA loads them with the 128-byte swizzle itself.
  if (e == cudaSuccess && !op->b_resident && op->groups == 1 && op->kh * op->kw == 1 && (op->K % 16) == 0 &&
      getenv("QNNP_CUDA_NO_GEMM2SM") == nullptr) {
    const size_t K = (size_t) op->K, N = op->goc;
    const int nt2 = (int) ceil_div(N, 240);
    std::vector<uint8_t> w2((size_t) nt2 * 256 * K, 0);
    std::vector<int32_t> b2((size_t) nt2 * 240, 0);
    for (size_t n = 0; n < N; n++) {
      const size_t t = n / 240, r = n % 240;
      memcpy(w2.data() + (t * 256 + r) * K, kernel + n * K, K);
      b2[n] = fold_bias(bias[n], K, op->izp, op->kzp, kernel + n * K);
    }
    // ones row (row sums of A) right after the tile's real channels rounded to 16: row 240, or earlier in the ragged last tile
    for (int t = 0; t < nt2; t++) {
      const size_t real = t == nt2 - 1 ? N - (size_t) t * 240 : 240;
      memset(w2.data() + ((size_t) t * 256 + round_up(real, 16)) * K, 1, K);
    }
    e = cudaMalloc((void**) &op->d_w2, w2.size());
    if (e == cudaSuccess) e = cudaMalloc((void**) &op->d_bias2, b2.size() * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMemcpy(op->d_w2, w2.data(), w2.size(), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(op->d_bias2, b2.data(), b2.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
    op->n_tiles2 = nt2;
  }
  return map_cuda(e, "uploading packed weights");
}

// Weight-operand mode of the depthwise tensor-core kernel.  d = w - kzp spans 9 bits in general:
//   1: kzp == 0                  -> raw u8 weights
//   0: every d in [-128, 127]    -> one s8 operand holding d
//   3: every -d in [-128, 127]   -> one s8 operand holding kzp - w; the accumulators are the NEGATED sums and the epilogue
//                                   subtracts them (free: the bias add becomes a multiply-add by -1).  kzp = 127 — the
//                                   reference benchmarks' own choice — always lands here: d in [-127, 128].
//   2: otherwise                 -> two s8 operands d = floor(d/2) + ceil(d/2) side by side (32 accumulator columns per
//                                   16 channels, added in the epilogue)
int dw_tc_wmode(size_t C, const uint8_t* kernel, int kzp) {
  if (kzp == 0) return 1;
  bool fits = true, fits_neg = true;
  for (size_t i = 0; i < C * 9; i++) {
    const int d = (int) kernel[i] - kzp;
    if (d < -128 || d > 127) fits = false;
    if (-d < -128 || -d > 127) fits_neg = false;
  }
  return fits ? 0 : (fits_neg ? 3 : 2);
}

// Operands of the depthwise tensor-core kernel, built in HOST memory (tests/test_dw_umma_plan.py replays the kernel on
// exactly these bytes).  kernel = [C][9] uint8, wmode: see dw_tc_wmode().
//   wp: per 16-channel group and UMMA u the B operand [2 K-chunks][nbc rows][16 B], each K-chunk diag(w_tap - kzp)
//   bc: [64 border classes][C]: bias - izp * (sum of w - kzp over the taps inside the image); uform: XOR 2^31 (the offset
//       of the "U" requantisation rides on the bias add)
void pack_dw_umma_host(size_t C, const uint8_t* kernel, const int32_t* bias, int izp, int kzp, int wmode, bool uform,
                       std::vector<uint8_t>& wp, std::vector<int32_t>& bc) {
  const int nbc = wmode == 2 ? 32 : 16;
  const size_t ub = (size_t) 2 * nbc * 16;  // bytes of one UMMA's B operand
  wp.assign((C / 16) * q8::kDwTcTaps * ub, 0);
  const int t0[q8::kDwTcTaps] = {0, 3, 6, 1, 7}, t1[q8::kDwTcTaps] = {2, 5, 8, 4, -1};  // tap = ky*3 + kx
  for (size_t cg = 0; cg < C / 16; cg++)
    for (int u = 0; u < q8::kDwTcTaps; u++)
      for (int ch = 0; ch < 2; ch++) {
        const int tap = ch == 0 ? t0[u] : t1[u];
        if (tap < 0) continue;
        for (int n = 0; n < 16; n++) {
          const int32_t w = kernel[(cg * 16 + n) * 9 + tap];
          const int32_t d = w - kzp;
          int32_t da = wmode == 1 ? w : (wmode == 3 ? -d : d), db = 0;
          if (wmode == 2) da = d >> 1, db = d - da;
          uint8_t* blk = wp.data() + (cg * q8::kDwTcTaps + u) * ub + (size_t) ch * nbc * 16;
          blk[(size_t) n * 16 + n] = (uint8_t) da;                        // B[n][k = n] of this K-chunk
          if (nbc == 32) blk[(size_t) (16 + n) * 16 + n] = (uint8_t) db;  // second operand half: rows 16..31
        }
      }
  bc.assign((size_t) 64 * C, 0);
  for (int rm = 0; rm < 8; rm++)
    for (int cm = 0; cm < 8; cm++)
      for (size_t c = 0; c < C; c++) {
        int64_t sum = 0;
        for (int ky = 0; ky < 3; ky++)
          for (int kx = 0; kx < 3; kx++)
            if (((rm >> ky) & 1) && ((cm >> kx) & 1)) sum += (int32_t) kernel[c * 9 + ky * 3 + kx] - kzp;
        const int32_t v = (int32_t) ((int64_t) bias[c] - (int64_t) izp * sum);
        bc[((size_t) rm * 8 + cm) * C + c] = uform ? (int32_t) ((uint32_t) v ^ 0x80000000u) : v;
      }
}

// Pair-mode B operands: per channel pair (32 channels) and tap one K-major no-swizzle block [2 K-chunks][32 rows][16 B] =
// diag(w_tap[c] - kzp) over the pair's 32 channels (rows = output channel, K = input channel; chunk = K / 16).  Channels
// beyond C (odd group count) keep zero weights.  wmode as in dw_tc_wmode() (never 2 here).
void pack_dw_umma32_host(size_t C, const uint8_t* kernel, int kzp, int wmode, std::vector<uint8_t>& wp) {
  const size_t pairs = (C + 31) / 32;
  wp.assign(pairs * q8::kDwTcTaps32 * 1024, 0);
  for (size_t pr = 0; pr < pairs; pr++)
    for (int t = 0; t < q8::kDwTcTaps32; t++)
      for (int n = 0; n < 32; n++) {
        const size_t c = pr * 32 + n;
        if (c >= C) continue;
        const int32_t w = kernel[c * 9 + t], d = w - kzp;
        const int32_t v = wmode == 1 ? w : (wmode == 3 ? -d : d);
        wp[(pr * q8::kDwTcTaps32 + t) * 1024 + (size_t) (n / 16) * 512 + (size_t) n * 16 + (n % 16)] = (uint8_t) v;
      }
}

enum qnnp_status pack_dw3x3(qnnp_operator* op, const uint8_t* kernel, const int32_t* bias) {
  const size_t C = op->groups;
  op->c_pad = (int) round_up(C, 4);
  std::vector<int32_t> w32((size_t) 9 * op->c_pad, 0), fbias(op->c_pad, 0);
  bool fits_s8 = true, fits_neg = true;
  for (size_t c = 0; c < C; c++) {
    for (int t = 0; t < 9; t++) {
      const int32_t d = (int32_t) kernel[c * 9 + t] - (int32_t) op->kzp;
      w32[(size_t) t * op->c_pad + c] = d;
      if (d < -128 || d > 127) fits_s8 = false;
      if (d < -127 || d > 128) fits_neg = false;
    }
    fbias[c] = fold_bias(bias[c], 9, op->izp, op->kzp, kernel + c * 9);
  }
  // streaming dp4a kernel: per channel and kernel row one word (tap kx=0, kx=1, kx=2, 0).
  //   kzp == 0            -> u8 weights as they are                      (wmode 1)
  //   every w-kzp in s8   -> one s8 operand                               (wmode 0)
  //   every kzp-w in s8   -> one s8 operand holding kzp - w; the kernel accumulates the negated sums from the negated
  //                          bias and negates once per output (wmode 3; kzp = 127, the reference benchmarks' choice)
  //   otherwise           -> w - kzp = A + B, A = floor(d/2), B = d - A   (wmode 2; both in [-128, 127] since kzp >= 1)
  op->dw_wmode = op->kzp == 0 ? 1 : (fits_s8 ? 0 : (fits_neg ? 3 : 2));
  std::vector<uint32_t> wa((size_t) 3 * op->c_pad, 0), wb((size_t) 3 * op->c_pad, 0);
  for (size_t c = 0; c < C; c++)
    for (int ky = 0; ky < 3; ky++) {
      uint32_t a = 0, b = 0;
      for (int kx = 0; kx < 3; kx++) {
        const int32_t d = w32[(size_t) (ky * 3 + kx) * op->c_pad + c];
        int32_t da = op->dw_wmode == 3 ? -d : d, db = 0;
        if (op->dw_wmode == 2) {
          da = d >> 1;  // floor
          db = d - da;
        }
        a |= (uint32_t) (uint8_t) da << (8 * kx);
        b |= (uint32_t) (uint8_t) db << (8 * kx);
      }
      wa[(size_t) ky * op->c_pad + c] = a;
      wb[(size_t) ky * op->c_pad + c] = b;
    }
  op->weights_bytes = w32.size() * sizeof(int32_t);
  op->bias_count = fbias.size();
  cudaError_t e = cudaMalloc(&op->d_weights, op->weights_bytes);
  if (e == cudaSuccess) e = cudaMalloc((void**) &op->d_bias, fbias.size() * sizeof(int32_t));
  if (e == cudaSuccess) e = cudaMalloc((void**) &op->d_dw_wa, wa.size() * sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaMalloc((void**) &op->d_dw_wb, wb.size() * sizeof(uint32_t));
  if (e == cudaSuccess) e = cudaMemcpy(op->d_weights, w32.data(), op->weights_bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(op->d_bias, fbias.data(), fbias.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(op->d_dw_wa, wa.data(), wa.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(op->d_dw_wb, wb.data(), wb.size() * sizeof(uint32_t), cudaMemcpyHostToDevice);
  // tensor-core kernel operands (q8_dwconv_umma_sm100.cu)
  if (e == cudaSuccess && (C % 16) == 0) {
    std::vector<uint8_t> wp;
    std::vector<int32_t> bc;
    op->dwtc_wmode = dw_tc_wmode(C, kernel, op->kzp);
    pack_dw_umma_host(C, kernel, bias, op->izp, op->kzp, op->dwtc_wmode, op->rq_mode == 5 || op->rq_mode == 6, wp, bc);
    e = cudaMalloc((void**) &op->d_dwtc_w, wp.size());
    if (e == cudaSuccess) e = cudaMalloc((void**) &op->d_dwtc_bias, bc.size() * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMemcpy(op->d_dwtc_w, wp.data(), wp.size(), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(op->d_dwtc_bias, bc.data(), bc.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
    if (e == cudaSuccess && op->dwtc_wmode != 2 && C >= 32) {  // channel-pair operands (DwTcParams::pair)
      std::vector<uint8_t> wp32;
      pack_dw_umma32_host(C, kernel, op->kzp, op->dwtc_wmode, wp32);
      e = cudaMalloc((void**) &op->d_dwtc_w32, wp32.size());
      if (e == cudaSuccess) e = cudaMemcpy(op->d_dwtc_w32, wp32.data(), wp32.size(), cudaMemcpyHostToDevice);
    }
  }
  return map_cuda(e, "uploading depthwise weights");
}

enum qnnp_status pack_direct(qnnp_operator* op, const uint8_t* kernel, const int32_t* bias) {
  const size_t K = (size_t) op->kh * op->kw * op->gic;
  const size_t oc_all = (size_t) op->groups * op->goc;
  std::vector<int32_t> fbias(oc_all);
  for (size_t oc = 0; oc < oc_all; oc++) fbias[oc] = fold_bias(bias[oc], K, op->izp, op->kzp, kernel + oc * K);
  op->weights_bytes = oc_all * K;
  op->bias_count = oc_all;
  cudaError_t e = cudaMalloc(&op->d_weights, op->weights_bytes);
  if (e == cudaSuccess) e = cudaMalloc((void**) &op->d_bias, oc_all * sizeof(int32_t));
  if (e == cudaSuccess) e = cudaMemcpy(op->d_weights, kernel, op->weights_bytes, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(op->d_bias, fbias.data(), oc_all * sizeof(int32_t), cudaMemcpyHostToDevice);
  return map_cuda(e, "uploading weights");
}

// ------------------------------------------------------------------------------------------------
// launch plans
// ------------------------------------------------------------------------------------------------
// Everything a launch needs besides the stream — kernel parameters, tensor maps, grid, loader / store variants, the
// depthwise tiling — is a function of the operator and of the (input, output) pointers it was set up with.  It is
// computed ONCE, in qnnp_setup_* when both pointers are device pointers (else at the first run, when the staging
// buffers exist), and cached in the operator: qnnp_run_operator only launches.  Environment switches are read while
// the plan is built, never on the launch path.  (Round 1 redid all of it, ~10 getenv() calls and a tensor-map encode
// included, on every run: SURVEY.md §3.4 puts this work in setup, like the reference's indirection-buffer setup,
// src/convolution.c:428-492.)
enum PlanPath {
  kPlanNone = 0, kPlanIgemm, kPlanGemm2sm, kPlanDwUmma, kPlanDwStream, kPlanDwGeneric, kPlanDirect,
  kPlanAdd, kPlanGavgPool, kPlanPool2d, kPlanMap, kPlanSoftargmax, kPlanShuffle
};

bool env_set(const char* name) { return getenv(name) != nullptr; }

// Panel epilogue tables (q8_igemm_sm100.cuh: out_mode 2): n_tile is split greedily into panels of 128/64/32/16 bytes.
void fill_panel_tables(q8::IgemmParams& p, bool dense) {
  const int W = p.folded ? 32 : 16;
  if (dense) {  // one dense image of pitch N = n_tile: unit c starts at byte c * W of its row, no swizzle
    p.e2_dense = 1, p.e2_panels = 0, p.e2_box_rows = 128;
    for (int c = 0; c < (p.n_tile + W - 1) / W && c < 16; c++) {
      p.e2_unit[c].x = (uint32_t) (c * W);
      p.e2_unit[c].y = (uint32_t) p.n_tile;  // pitch; lsh = mask = 0
    }
    return;
  }
  p.e2_dense = 0;
  int col = 0, off = 0, k = 0;
  const int widths[4] = {128, 64, 32, 16};
  for (int wi = 0; wi < 4; wi++) {
    const int w = widths[wi];
    while (p.n_tile - col >= w && k < 4) {
      p.e2_col0[k] = col, p.e2_width[k] = w, p.e2_off[k] = off, p.e2_map[k] = 3 - wi;
      off += w * q8::kTileM * p.mt;
      col += w;
      k++;
    }
  }
  p.e2_panels = k;
  p.e2_box_rows = (p.mt % 2 == 0) ? 256 : 128;
  const int per_sub = (p.n_tile + W - 1) / W;
  for (int c = 0; c < per_sub && c < 16; c++) {
    const int ucol = c * W;
    int pk = 0;
    while (pk + 1 < k && ucol >= p.e2_col0[pk] + p.e2_width[pk]) pk++;
    const int w = p.e2_width[pk];
    const uint32_t lsh = w == 128 ? 4 : (w == 64 ? 3 : (w == 32 ? 2 : 0));
    const uint32_t mask = w == 128 ? 0x70 : (w == 64 ? 0x30 : (w == 32 ? 0x10 : 0));
    p.e2_unit[c].x = (uint32_t) (p.e2_off[pk] + (ucol - p.e2_col0[pk]));
    p.e2_unit[c].y = (uint32_t) w | (lsh << 8) | (mask << 16);
  }
}

}  // namespace

struct qnnp_launch_plan {
  bool valid = false;
  PlanPath path = kPlanNone;
  const uint8_t* in = nullptr;
  uint8_t* out = nullptr;
  int grid = 0;
  // igemm
  q8::IgemmParams ig{};
  int ig_mode = 0, ig_vec = 0;
  bool has_tmap_a = false, has_smaps = false;
  alignas(64) CUtensorMap tmap_a;
  alignas(64) CUtensorMap tmap_b;
  q8::IgemmStoreMaps smaps;
  // depthwise
  q8::DwTcParams tp{};
  alignas(64) CUtensorMap dw_tmap;
  q8::DwStreamParams sp{};
  q8::DwParams dp{};
  int dw_cv = 1;
  // direct
  q8::DirectParams dir{};
  // element-wise / pooling
  const uint8_t* in2 = nullptr;
  int vec = 1;
  bool flag = false;  // map: table lookup; pool2d: max
  q8::AddParams add{};
  q8::MapParams map{};
  q8::ShuffleParams shuf{};
  q8::SoftargmaxParams soft{};
  q8::GavgParams gavg{};
  q8::PoolParams pool{};
};

void delete_plan(qnnp_launch_plan* p) { delete p; }

namespace {

// widest piece size in {16, 4, 1} bytes that divides every given address / stride / length
int common_vec(std::initializer_list<uintptr_t> values) {
  int v = 16;
  for (uintptr_t x : values) v = pow2_align(x, v);
  return v >= 16 ? 16 : (v >= 4 ? 4 : 1);
}

enum qnnp_status build_plan(qnnp_operator* op, const uint8_t* in, const uint8_t* in2, uint8_t* out) {
  if (op->plan == nullptr) op->plan = new (std::nothrow) qnnp_launch_plan();
  if (op->plan == nullptr) return qnnp_status_out_of_memory;
  qnnp_launch_plan& pl = *op->plan;
  pl.valid = false;
  pl.in = in, pl.in2 = in2, pl.out = out;
  const size_t M = op->batch * op->out_h * op->out_w;
  switch (op->kind) {
    case kKindIgemmGemm:
    case kKindIgemmConv: {
      q8::IgemmParams p{};
      p.in = in;
      p.out = out;
      p.wpack = (const uint8_t*) op->d_weights;
      p.bias = op->d_bias;
      p.dbg_acc = g_lib.dbg_acc;
      p.M = (long long) M;
      p.m_tiles = (long long) ceil_div(M, q8::kTileM);
      p.m_super = (long long) ceil_div((size_t) p.m_tiles, (size_t) op->mt);
      p.acc_stride = op->mt * op->n_mma;
      p.acc_stages = 512 / p.acc_stride;
      if (p.acc_stages > q8::kMaxAccStages) p.acc_stages = q8::kMaxAccStages;
      if (const char* e = getenv("QNNP_CUDA_ACC_STAGES")) {
        const int v = atoi(e);
        if (v >= 2 && v <= p.acc_stages) p.acc_stages = v;
      }
      p.total_items = (long long) op->groups * p.m_super * op->n_tiles;
      if (M >= (1ull << 31) || p.total_items >= (1ll << 31)) {
        log_error("operator too large for one launch (M = %zu rows)", M);
        return qnnp_status_unsupported_parameter;
      }
      p.in_stride = (long long) op->in_stride;
      p.out_stride = (long long) op->out_stride;
      p.groups = (int) op->groups, p.gic = (int) op->gic, p.goc = (int) op->goc;
      p.in_h = (int) op->in_h, p.in_w = (int) op->in_w, p.out_h = (int) op->out_h, p.out_w = (int) op->out_w;
      p.kh = (int) op->kh, p.kw = (int) op->kw, p.stride_h = (int) op->stride_h, p.stride_w = (int) op->stride_w;
      p.dil_h = (int) op->dil_h, p.dil_w = (int) op->dil_w, p.pad_top = (int) op->pad_top, p.pad_left = (int) op->pad_left;
      p.K = op->K, p.nkc = op->nkc, p.skc = op->skc, p.k_stages = op->k_stages, p.mt = op->mt;
      p.n_tiles = op->n_tiles, p.n_tile = op->n_tile, p.n_mma = op->n_mma, p.has_corr = op->has_corr;
      p.folded = op->folded, p.b_signed = op->b_signed, p.has_b2 = op->has_b2, p.bias_steps = op->bias_steps;
      p.blk_chunks = op->blk_chunks, p.k_tail_pad = op->k_tail_pad, p.smem_aconst_off = op->smem_aconst_off;
      p.b_resident = op->b_resident, p.num_stages = op->num_stages, p.stage_bytes = op->stage_bytes;
      p.bias_count = (int) op->bias_count;
      p.smem_b_off = op->smem_b_off, p.smem_bias_off = op->smem_bias_off, p.smem_a_off = op->smem_a_off;
      p.smem_stage_off = op->smem_stage_off, p.staging_bytes = op->staging_bytes, p.smem_total = op->smem_total;
      p.staging_bufs = 1;
      p.izp = op->izp, p.kzp = op->kzp;
      p.rq = op->rq;
      p.rq_mode = op->rq_mode;
      // output path: 2 = swizzled panels + 2-D tensor stores (any item, any N, pixel-stride gaps); 1 = dense image + one
      // 1-D bulk store per full item; 0 = per-thread global stores
      const bool bulk = op->bulk_capable && op->out_stride == op->goc && ((uintptr_t) out % 16) == 0 &&
          !env_set("QNNP_CUDA_NO_BULK_STORE");
      p.out_mode = bulk ? 1 : 0;
      pl.has_smaps = false;
      if ((op->rq_mode == 5 || op->rq_mode == 6) && op->groups == 1 && ((uintptr_t) out % 16) == 0 && (op->out_stride % 16) == 0 &&
          g_lib.dbg_acc == nullptr && !env_set("QNNP_CUDA_NO_PANEL_STORE")) {
        // narrow dense outputs whose pitch is conflict-free (N / 16 odd: the 8 lanes of a store phase hit 8 different
        // 16-byte bank groups) leave as ONE contiguous bulk copy per item — measured: 16-byte-wide tensor-store boxes
        // cost the N = 16 projection 13 % (0.70 vs 0.62 ms)
        const bool dense = op->n_tiles == 1 && op->out_stride == op->goc && (int) op->goc == op->n_tile && ((op->goc / 16) & 1) == 1 &&
            op->goc <= 112 && !env_set("QNNP_CUDA_NO_DENSE_STORE");
        fill_panel_tables(p, dense);
        bool ok = true;
        bool done[4] = {false, false, false, false};
        for (int k = 0; k < p.e2_panels && ok; k++) {
          const int cls = p.e2_map[k];
          if (done[cls]) continue;
          done[cls] = true;
          ok = make_tmap_out(&pl.smaps.m[cls][0], out, M, op->goc, op->out_stride, p.e2_width[k], p.e2_box_rows);
        }
        if (ok) {
          p.out_mode = 2;
          pl.has_smaps = true;
        }
      }
      int ov = pow2_align((uintptr_t) out, 32);
      ov = pow2_align((uintptr_t) op->out_stride, ov);
      if (op->groups > 1) ov = pow2_align((uintptr_t) op->goc, ov);  // group offset g*goc (tile offsets are multiples of 16)
      p.out_vec = ov;
      p.shift_mul = q8::requant_shift_mul(op->rq);
      // loader vector width
      int vec = pow2_align((uintptr_t) in, 16);
      vec = pow2_align((uintptr_t) op->in_stride, vec);
      vec = pow2_align((uintptr_t) op->gic, vec);
      if (vec < 4) vec = 1;
      const int mode = op->kind == kKindIgemmGemm ? q8::kModeGemm : q8::kModeConv;
      // 3x3 over 3 dense channels (MobileNetV2 stem): the taps of a kernel row are one 9-byte run
      if (mode == q8::kModeConv && vec == 1 && op->kh == 3 && op->kw == 3 && op->gic == 3 && op->dil_w == 1 &&
          op->in_stride == 3 && op->k_stages == 1 && op->in_w >= 3 && ((uintptr_t) in % 4) == 0 &&
          (op->batch * op->in_h * op->in_w * 3) % 4 == 0 && !env_set("QNNP_CUDA_NO_RUN9"))
        vec = 0;
      // ... and those runs are read from bulk-staged raw input rows when the tensor can be bulk-copied (16-byte aligned
      // base and size) and an item never spans more than two images; the A ring gives up stages for the two raw buffers
      if (vec == 0 && ((uintptr_t) in % 16) == 0 && ((size_t) op->batch * op->in_h * op->in_w * 3) % 16 == 0 &&
          (size_t) op->out_h * op->out_w >= (size_t) op->mt * q8::kTileM && !env_set("QNNP_CUDA_NO_RAW9")) {
        const int rows_out = (int) ((op->mt * q8::kTileM + op->out_w - 2) / op->out_w) + 1;
        const int rows_in = (rows_out + 1) * (int) op->stride_h + 2 * (int) ((op->kh - 1) * op->dil_h + 1);
        const int raw_cap = (int) round_up((size_t) rows_in * op->in_w * 3 + 64, 128);
        // split the shared memory that the A ring had: 4 raw buffers if >= 3 A stages remain, else 3, else 2
        int max_bufs = 4;
        if (const char* ev = getenv("QNNP_CUDA_RAW_BUFS")) max_bufs = atoi(ev) < 2 ? 2 : (atoi(ev) > 4 ? 4 : atoi(ev));
        for (int bufs = max_bufs; bufs >= 2 && vec == 0; bufs--) {
          const int fixed = p.smem_a_off + 2 * p.staging_bytes + 2048 + bufs * raw_cap;
          int stages = p.num_stages;
          while (stages > 3 && fixed + stages * p.stage_bytes > g_lib.max_smem_optin - kCtlReserve) stages--;
          if (fixed + stages * p.stage_bytes > g_lib.max_smem_optin - kCtlReserve) continue;
          p.num_stages = stages;
          p.smem_stage_off = (int) round_up(p.smem_a_off + stages * p.stage_bytes, 1024);
          p.smem_raw_off = p.smem_stage_off + 2 * p.staging_bytes;
          p.raw_cap = raw_cap;
          p.raw_bufs = bufs;
          p.raw_batch = (int) op->batch;
          p.smem_total = p.smem_raw_off + bufs * raw_cap + 1024;
          vec = 2;
        }
      }
      // 1x1 / FC with 16-byte aligned rows: the TMA loads the activation tiles
      pl.has_tmap_a = false;
      // 32-byte slabs when K % 32 == 0; when K % 32 == 16 and the whole K is one stage (K = 144), slabs for the first
      // K - 16 bytes plus the last chunk through the 16-byte view (its partner chunk is out of bounds: zero-filled)
      int a_sw32 = 0;
      if (!env_set("QNNP_CUDA_NO_A_SW32") && (op->skc % 2) == 0) {
        if ((op->K % 32) == 0) a_sw32 = 1;
        else if ((op->K % 32) == 16 && op->K > 32 && op->k_stages == 1 && op->skc * 16 == op->K + 16) a_sw32 = 2;
      }
      if (mode == q8::kModeGemm && vec == 16 && op->groups == 1 && (op->K % 16) == 0 && op->skc <= 256 && M < (1ull << 31) &&
          !env_set("QNNP_CUDA_NO_TMA") &&
          (a_sw32 == 2 ? make_tmap_a(&pl.tmap_a, in, M, op->in_stride, op->K - 16, op->skc - 2, 1) &&
                             make_tmap_a(reinterpret_cast<CUtensorMap*>(&pl.smaps.m[4][0]), in, M, op->in_stride, op->K, 2, 0)
                       : make_tmap_a(&pl.tmap_a, in, M, op->in_stride, op->K, op->skc, a_sw32))) {
        vec = 32;
        pl.has_tmap_a = true;
        p.a_sw32 = a_sw32;
        p.a_tail_c = op->skc - 2;
        if (a_sw32 == 2) pl.has_smaps = true;  // (the tail view travels in the store-map block)
      }
      // panel epilogue: a second staging buffer per epilogue pair when shared memory allows — the shallow-K layers (where the
      // epilogue is the long pole) have far more ring stages than they can use, so stages beyond "3 items of K or 64 KB in
      // flight" are traded for it
      if (p.out_mode == 2 && vec != 2 && !env_set("QNNP_CUDA_SINGLE_STAGING")) {
        const int limit = g_lib.max_smem_optin - kCtlReserve;
        const int a_stage = p.mt * p.skc * q8::kChunkBytes;
        auto total = [&](int st) { return (int) round_up((size_t) p.smem_a_off + (size_t) st * p.stage_bytes, 1024) + 4 * p.staging_bytes + 1024; };
        auto enough = [&](int st) { return st >= 3 && ((long long) st * a_stage >= 64 * 1024 || st >= 3 * p.k_stages); };
        int stages = p.num_stages;
        while (total(stages) > limit && enough(stages - 1)) stages--;
        if (total(stages) <= limit && (stages == p.num_stages || enough(stages))) {
          p.num_stages = stages;
          p.smem_stage_off = (int) round_up((size_t) p.smem_a_off + (size_t) stages * p.stage_bytes, 1024);
          p.smem_total = total(stages);
          p.staging_bufs = 2;
        }
      }
      pl.grid = (int) persistent_grid(p.total_items);
      pl.ig = p;
      pl.ig_mode = mode, pl.ig_vec = vec;
      pl.path = kPlanIgemm;
      // large GEMMs (weights not resident): the CTA-pair kernel, when the operands can be described to the TMA
      // (8 epilogue warps per CTA: the pair kernel wins where the tensor pipe / weight streaming is the long pole, i.e. deep
      // K.  Measured on the MobileNetV2 projections with K = 960: 0.064 -> 0.058, 0.113 -> 0.095 ms; at K = 576 the single-CTA
      // kernel is the faster one since it loads its activations as 32-byte slabs: 0.105 vs 0.139 ms.)
      const int g2_min_k = getenv("QNNP_CUDA_GEMM2SM_MIN_K") != nullptr ? atoi(getenv("QNNP_CUDA_GEMM2SM_MIN_K")) : 768;
      if (op->d_w2 != nullptr && op->K >= g2_min_k && mode == q8::kModeGemm && (op->rq_mode == 5 || op->rq_mode == 6) && M >= 256 &&
          ((uintptr_t) in % 16) == 0 && (op->in_stride % 16) == 0 && ((uintptr_t) out % 16) == 0 && (op->out_stride % 16) == 0 &&
          g_lib.dbg_acc == nullptr && !env_set("QNNP_CUDA_NO_GEMM2SM")) {
        q8::IgemmParams q = p;
        q.n_tile = 240, q.n_mma = 256, q.n_tiles = op->n_tiles2, q.mt = 1, q.folded = 0, q.has_corr = 1;
        q.bias = op->d_bias2;
        q.staging_bytes = q8::kTileM * 240;
        q.out_mode = 2;
        q.e2_last_nmma = (int) round_up(op->goc - (size_t) (op->n_tiles2 - 1) * 240, 16) + 16;
        fill_panel_tables(q, false);
        bool ok = make_tmap_kmajor_sw128(&pl.tmap_a, in, M, (size_t) op->K, op->in_stride) &&
            make_tmap_kmajor_sw128(&pl.tmap_b, op->d_w2, (size_t) op->n_tiles2 * 256, (size_t) op->K, (size_t) op->K);
        bool done[4] = {false, false, false, false};
        for (int k = 0; k < q.e2_panels && ok; k++) {
          const int cls = q.e2_map[k];
          if (done[cls]) continue;
          done[cls] = true;
          ok = make_tmap_out(&pl.smaps.m[cls][0], out, M, op->goc, op->out_stride, q.e2_width[k], q.e2_box_rows);
        }
        if (ok) {
          const long long tiles = (long long) ceil_div(M, 256) * op->n_tiles2;
          long long clusters = g_lib.num_sms / 2;
          if (clusters > tiles) clusters = tiles;
          if (const char* ev = getenv("QNNP_CUDA_MAX_CTAS")) {
            const long long v = atoll(ev) / 2;
            if (v >= 1 && v < clusters) clusters = v;
          }
          pl.ig = q;
          pl.grid = (int) clusters;
          pl.path = kPlanGemm2sm;
        }
      }
      break;
    }
    case kKindDw3x3: {
      int cv = pow2_align((uintptr_t) in, 4);
      cv = pow2_align((uintptr_t) out, cv);
      cv = pow2_align((uintptr_t) op->in_stride, cv);
      cv = pow2_align((uintptr_t) op->out_stride, cv);
      cv = pow2_align((uintptr_t) op->groups, cv);
      const bool stream_ok = cv == 4 && op->dil_h == 1 && op->dil_w == 1 && op->stride_h == op->stride_w &&
          (op->stride_h == 1 || op->stride_h == 2) && !env_set("QNNP_CUDA_DW_GENERIC");
      // tensor-core path: channels % 16 == 0 and 16-byte aligned pixels (TMA boxes, 16-byte output stores)
      // (measured on MobileNetV2 at batch 4096: the tcgen05 kernel wins everywhere except — with the TWO-operand weight form
      // only — stride-2 layers tiled by rows, where the CUDA-core streaming kernel is ~8% faster; with a single operand
      // (16 accumulator columns per unit) it wins there too: 112x112x96 stride 2 1.87 vs 2.00 ms.  QNNP_CUDA_DW_UMMA=1 /
      // QNNP_CUDA_DW_S2_UMMA=1 force the tensor-core path, QNNP_CUDA_DW_S2_STREAM=1 / QNNP_CUDA_DW_NO_UMMA=1 the other way)
      const bool force_tc = env_set("QNNP_CUDA_DW_UMMA");
      const bool s2_rows = op->stride_h == 2 && 2 * (op->out_h - 1) + 3 > 32 && !env_set("QNNP_CUDA_DW_S2_UMMA") &&
          (op->dwtc_wmode == 2 || env_set("QNNP_CUDA_DW_S2_STREAM"));
      q8::DwTcParams& tp = pl.tp;
      const bool tc_base = stream_ok && op->d_dwtc_w != nullptr && !env_set("QNNP_CUDA_DW_NO_UMMA") && (force_tc || !s2_rows) &&
          ((uintptr_t) in % 16) == 0 && ((uintptr_t) out % 16) == 0 && (op->in_stride % 16) == 0 && (op->out_stride % 16) == 0;
      // channel-pair form (32-byte granularity on the L2 for the loads as well) where it was measured to win: stride 2, which
      // reads four input bytes per output byte and ran at 74 % of the L2's request rate in the 16-channel form (112x112x96:
      // 1.76 -> 1.20 ms, 14x14x576: 0.194 -> 0.161).  At stride 1 its larger weight blocks (9 KB per channel pair and item
      // instead of 5 KB) cancel the gain (-1 % ... +14 %).  QNNP_CUDA_DW_PAIR=1 / QNNP_CUDA_DW_NO_PAIR=1 force it on / off.
      // ... and at stride 1 where all of the layer's (larger) pair blocks can stay resident and the layer has >= 4 channel
      // groups: 28x28x192 0.509 -> 0.460, 56x56x144 1.668 -> 1.629; not 112x112x32 (0.909 in the 16-channel form vs 0.946).
      const bool pair_allowed = !env_set("QNNP_CUDA_DW_NO_PAIR") && tc_base && op->d_dwtc_w32 != nullptr;
      bool tc_ok = pair_allowed &&
          plan_dw_umma((int) op->groups, (int) op->batch, (int) op->in_h, (int) op->in_w, (int) op->out_h, (int) op->out_w,
                       (int) op->stride_h, (int) op->pad_top, (int) op->pad_left, op->dwtc_wmode, g_lib.max_smem_optin, &tp, 1) &&
          (op->stride_h == 2 || env_set("QNNP_CUDA_DW_PAIR") || (tp.b_resident && tp.cgs >= 4)) &&
          make_tmap_dw(&pl.dw_tmap, in, op->batch, op->in_h, op->in_w, op->groups, op->in_stride, (int) op->stride_h, tp.box_px,
                       tp.box_rows, tp.nb, 1);
      // ... except that at stride 1 the 16-channel form wins where only IT has room for the border-class table in shared
      // memory (DwTcParams::bias_smem; 14x14x384: 0.257 ms in the pair form with the global table, 0.229 in the 16-channel
      // form with the shared one)
      if (tc_ok && op->stride_h == 1 && !tp.bias_smem && !env_set("QNNP_CUDA_DW_PAIR")) {
        q8::DwTcParams t16;
        if (plan_dw_umma((int) op->groups, (int) op->batch, (int) op->in_h, (int) op->in_w, (int) op->out_h, (int) op->out_w,
                         (int) op->stride_h, (int) op->pad_top, (int) op->pad_left, op->dwtc_wmode, g_lib.max_smem_optin, &t16, 0) &&
            t16.bias_smem)
          tc_ok = false;
      }
      if (!tc_ok)
        tc_ok = tc_base &&
            plan_dw_umma((int) op->groups, (int) op->batch, (int) op->in_h, (int) op->in_w, (int) op->out_h, (int) op->out_w,
                         (int) op->stride_h, (int) op->pad_top, (int) op->pad_left, op->dwtc_wmode, g_lib.max_smem_optin, &tp, 0) &&
            make_tmap_dw(&pl.dw_tmap, in, op->batch, op->in_h, op->in_w, op->groups, op->in_stride, (int) op->stride_h, tp.box_px,
                         tp.box_rows, tp.nb, 0);
      if (tc_ok) {
        tp.out = out, tp.wpack = tp.pair ? op->d_dwtc_w32 : op->d_dwtc_w, tp.bias_cls = op->d_dwtc_bias;
        tp.out_stride = (long long) op->out_stride;
        tp.rq = op->rq, tp.rq_mode = op->rq_mode;
        tp.acc_sign = op->dwtc_wmode == 3 ? -1 : 1;
        tp.store32 = tp.pair || ((tp.G % 2) == 0 && !env_set("QNNP_CUDA_DW_STORE16"));
        long long grid = persistent_grid(tp.total_items);
        tp.chunk = (int) ((tp.total_items + grid - 1) / grid);         // contiguous run of items per CTA
        grid = (tp.total_items + tp.chunk - 1) / tp.chunk;             // (CTAs that would start beyond the end are not launched)
        {  // digits of the per-item step (1) in the item schedule's mixed radix (cb fastest), and the unit-split reciprocals
          long long r = 1;
          tp.step_cb = (int) (r % tp.cblocks), r /= tp.cblocks;
          tp.step_x = (int) (r % tp.xt), r /= tp.xt;
          tp.step_y = (int) (r % tp.yt), r /= tp.yt;
          tp.step_n = (int) r;
          const int tail = (tp.out_w + 7) / 8 - (tp.xt - 1) * tp.mt;  // sub-tiles of the last x tile
          tp.inv_g = (65536u + (uint32_t) tp.mt - 1) / (uint32_t) tp.mt;
          tp.inv_tail = (65536u + (uint32_t) tail - 1) / (uint32_t) tail;
        }
        pl.grid = (int) grid;
        pl.path = kPlanDwUmma;
      } else if (stream_ok) {
        q8::DwStreamParams sp{};
        sp.in = in, sp.out = out;
        sp.wa = op->d_dw_wa, sp.wb = op->d_dw_wb, sp.bias = op->d_bias;
        sp.in_stride = (long long) op->in_stride, sp.out_stride = (long long) op->out_stride;
        sp.batch = (int) op->batch, sp.channels = (int) op->groups, sp.c_pad = op->c_pad;
        sp.in_h = (int) op->in_h, sp.in_w = (int) op->in_w, sp.out_h = (int) op->out_h, sp.out_w = (int) op->out_w;
        sp.stride = (int) op->stride_h, sp.pad_top = (int) op->pad_top, sp.pad_left = (int) op->pad_left;
        sp.wmode = op->dw_wmode, sp.izp = op->izp;
        sp.rq = op->rq, sp.rq_mode = op->rq_mode, sp.shift_mul = q8::requant_shift_mul(op->rq);
        pl.sp = sp;
        pl.path = kPlanDwStream;
      } else {
        q8::DwParams p{};
        p.in = in, p.out = out;
        p.w32 = (const int32_t*) op->d_weights;
        p.bias = op->d_bias;
        p.in_stride = (long long) op->in_stride, p.out_stride = (long long) op->out_stride;
        p.batch = (int) op->batch, p.channels = (int) op->groups, p.c_pad = op->c_pad;
        p.in_h = (int) op->in_h, p.in_w = (int) op->in_w, p.out_h = (int) op->out_h, p.out_w = (int) op->out_w;
        p.stride_h = (int) op->stride_h, p.stride_w = (int) op->stride_w, p.dil_h = (int) op->dil_h, p.dil_w = (int) op->dil_w;
        p.pad_top = (int) op->pad_top, p.pad_left = (int) op->pad_left;
        p.izp = op->izp;
        p.rq = op->rq, p.rq_mode = op->rq_mode;
        pl.dp = p;
        pl.dw_cv = cv == 4 ? 4 : 1;
        pl.path = kPlanDwGeneric;
      }
      break;
    }
    case kKindDirect: {
      q8::DirectParams p{};
      p.in = in, p.out = out;
      p.w = (const uint8_t*) op->d_weights;
      p.bias = op->d_bias;
      p.in_stride = (long long) op->in_stride, p.out_stride = (long long) op->out_stride;
      p.total = (long long) M * op->groups * op->goc;
      p.groups = (int) op->groups, p.gic = (int) op->gic, p.goc = (int) op->goc;
      p.in_h = (int) op->in_h, p.in_w = (int) op->in_w, p.out_h = (int) op->out_h, p.out_w = (int) op->out_w;
      p.kh = (int) op->kh, p.kw = (int) op->kw;
      p.stride_h = (int) op->stride_h, p.stride_w = (int) op->stride_w, p.dil_h = (int) op->dil_h, p.dil_w = (int) op->dil_w;
      p.pad_top = (int) op->pad_top, p.pad_left = (int) op->pad_left;
      p.izp = op->izp, p.kzp = op->kzp;
      p.rq = op->rq;
      p.deconv = op->is_deconv ? 1 : 0;
      pl.dir = p;
      pl.path = kPlanDirect;
      break;
    }
    case kKindAdd: {
      q8::AddParams p = op->add;
      p.a = in, p.b = in2, p.y = out;
      p.a_stride = (long long) op->in_stride, p.b_stride = (long long) op->in2_stride, p.y_stride = (long long) op->out_stride;
      const bool dense = op->in_stride == op->channels && op->in2_stride == op->channels && op->out_stride == op->channels;
      // dense rows form one long row: pieces may then straddle row boundaries
      const size_t row_len = dense ? op->batch * op->channels : op->channels;
      pl.vec = common_vec({(uintptr_t) in, (uintptr_t) in2, (uintptr_t) out, (uintptr_t) row_len,
                           dense ? 0 : (uintptr_t) op->in_stride, dense ? 0 : (uintptr_t) op->in2_stride,
                           dense ? 0 : (uintptr_t) op->out_stride});
      p.rows = dense ? 1 : (long long) op->batch;
      if (row_len / pl.vec >= (1ull << 31)) {  // keep the per-row piece count in 32 bits
        p.rows = (long long) op->batch, pl.vec = common_vec({(uintptr_t) in, (uintptr_t) in2, (uintptr_t) out, (uintptr_t) op->channels});
        p.pieces_per_row = (int) (op->channels / pl.vec);
      } else {
        p.pieces_per_row = (int) (row_len / pl.vec);
      }
      pl.add = p;
      pl.path = kPlanAdd;
      break;
    }
    case kKindClamp:
    case kKindLut: {
      q8::MapParams p{};
      p.x = in, p.y = out, p.lut = op->d_lut;
      p.x_stride = (long long) op->in_stride, p.y_stride = (long long) op->out_stride;
      p.lo = op->omin, p.hi = op->omax;
      const bool dense = op->in_stride == op->channels && op->out_stride == op->channels;
      const size_t row_len = dense ? op->batch * op->channels : op->channels;
      pl.vec = common_vec({(uintptr_t) in, (uintptr_t) out, (uintptr_t) row_len, dense ? 0 : (uintptr_t) op->in_stride,
                           dense ? 0 : (uintptr_t) op->out_stride});
      p.rows = dense ? 1 : (long long) op->batch;
      if (row_len / pl.vec >= (1ull << 31)) {
        p.rows = (long long) op->batch, pl.vec = common_vec({(uintptr_t) in, (uintptr_t) out, (uintptr_t) op->channels});
        p.pieces_per_row = (int) (op->channels / pl.vec);
      } else {
        p.pieces_per_row = (int) (row_len / pl.vec);
      }
      pl.map = p;
      pl.flag = op->kind == kKindLut;
      pl.path = kPlanMap;
      break;
    }
    case kKindShuffle: {
      q8::ShuffleParams p{};
      p.x = in, p.y = out;
      p.rows = (long long) op->batch, p.x_stride = (long long) op->in_stride, p.y_stride = (long long) op->out_stride;
      p.groups = (int) op->groups, p.group_channels = (int) op->gic;
      pl.shuf = p;
      pl.path = kPlanShuffle;
      break;
    }
    case kKindSoftargmax: {
      q8::SoftargmaxParams p{};
      p.x = in, p.y = out, p.table = op->d_table32;
      p.rows = (long long) op->batch, p.x_stride = (long long) op->in_stride, p.y_stride = (long long) op->out_stride;
      p.channels = (int) op->channels;
      pl.soft = p;
      pl.path = kPlanSoftargmax;
      break;
    }
    case kKindGavgPool: {
      q8::GavgParams p{};
      p.x = in, p.y = out;
      p.batch = (long long) op->batch, p.width = (long long) op->in_w;
      p.x_stride = (long long) op->in_stride, p.y_stride = (long long) op->out_stride;
      p.channels = (int) op->channels;
      p.bias = (int32_t) (0u - (uint32_t) op->in_w * (uint32_t) op->izp);  // src/global-average-pooling.c:137
      p.q = op->avgq;
      pl.vec = common_vec({(uintptr_t) in, (uintptr_t) out, (uintptr_t) op->channels, (uintptr_t) op->in_stride,
                           (uintptr_t) op->out_stride}) >= 4 ? 4 : 1;
      pl.gavg = p;
      pl.path = kPlanGavgPool;
      break;
    }
    case kKindAvgPool:
    case kKindMaxPool: {
      q8::PoolParams p{};
      p.x = in, p.y = out;
      p.batch = (long long) op->batch, p.x_stride = (long long) op->in_stride, p.y_stride = (long long) op->out_stride;
      p.channels = (int) op->channels;
      p.in_h = (int) op->in_h, p.in_w = (int) op->in_w, p.out_h = (int) op->out_h, p.out_w = (int) op->out_w;
      p.kh = (int) op->kh, p.kw = (int) op->kw, p.stride_h = (int) op->stride_h, p.stride_w = (int) op->stride_w;
      p.dil_h = (int) op->dil_h, p.dil_w = (int) op->dil_w, p.pad_top = (int) op->pad_top, p.pad_left = (int) op->pad_left;
      p.izp = op->izp, p.bias = 0, p.lo = op->omin, p.hi = op->omax;
      p.q = op->avgq;
      pl.vec = common_vec({(uintptr_t) in, (uintptr_t) out, (uintptr_t) op->channels, (uintptr_t) op->in_stride,
                           (uintptr_t) op->out_stride}) >= 4 ? 4 : 1;
      pl.flag = op->kind == kKindMaxPool;
      pl.pool = p;
      pl.path = kPlanPool2d;
      break;
    }
    default:
      return qnnp_status_invalid_parameter;
  }
  pl.valid = true;
  return qnnp_status_success;
}

enum qnnp_status launch(qnnp_operator* op, const uint8_t* in, const uint8_t* in2, uint8_t* out, cudaStream_t stream) {
  if (op->plan == nullptr || !op->plan->valid || op->plan->in != in || op->plan->in2 != in2 || op->plan->out != out) {
    const enum qnnp_status st = build_plan(op, in, in2, out);
    if (st != qnnp_status_success) return st;
  }
  const qnnp_launch_plan& pl = *op->plan;
  cudaError_t e = cudaSuccess;
  switch (pl.path) {
    case kPlanIgemm:
      e = q8::launch_q8_igemm(pl.ig, pl.ig_mode, pl.ig_vec, pl.has_tmap_a ? &pl.tmap_a : nullptr,
                              pl.has_smaps ? &pl.smaps : nullptr, pl.grid, g_lib.max_smem_optin, stream);
      break;
    case kPlanGemm2sm:
      e = q8::launch_q8_gemm2sm(pl.ig, &pl.tmap_a, &pl.tmap_b, pl.smaps, pl.grid, g_lib.max_smem_optin, stream);
      break;
    case kPlanDwUmma:
      e = q8::launch_q8_dwconv3x3_umma(pl.tp, &pl.dw_tmap, pl.grid, g_lib.max_smem_optin, stream);
      if (e == cudaSuccess) g_lib.dw_umma_launches.fetch_add(1);
      break;
    case kPlanDwStream: e = q8::launch_q8_dwconv3x3_stream(pl.sp, stream); break;
    case kPlanDwGeneric: e = q8::launch_q8_dwconv3x3(pl.dp, pl.dw_cv, stream); break;
    case kPlanDirect: e = q8::launch_q8_direct_conv(pl.dir, stream); break;
    case kPlanAdd: e = q8::launch_q8_add(pl.add, pl.vec, stream); break;
    case kPlanMap: e = q8::launch_q8_map(pl.map, pl.vec, pl.flag, stream); break;
    case kPlanShuffle: e = q8::launch_q8_shuffle(pl.shuf, stream); break;
    case kPlanSoftargmax: e = q8::launch_q8_softargmax(pl.soft, stream); break;
    case kPlanGavgPool: e = q8::launch_q8_gavgpool(pl.gavg, pl.vec, stream); break;
    case kPlanPool2d: e = q8::launch_q8_pool2d(pl.pool, pl.vec, pl.flag, stream); break;
    default: return qnnp_status_invalid_parameter;
  }
  g_lib.launches.fetch_add(1);
  return map_cuda(e, "kernel launch");
}

enum qnnp_status ensure_capacity(uint8_t** buf, size_t* cap, size_t need) {
  if (*cap >= need) return qnnp_status_success;
  cudaFree(*buf);
  *buf = nullptr;
  *cap = 0;
  cudaError_t e = cudaMalloc((void**) buf, need);
  if (e != cudaSuccess) return map_cuda(e, "allocating device staging buffer");
  *cap = need;
  return qnnp_status_success;
}

enum qnnp_status run_impl(qnnp_operator* op, bool async) {
  if (op == nullptr) return qnnp_status_invalid_parameter;
  if (op->batch == 0) return qnnp_status_success;  // src/operator-run.c:642
  bind_device();
  cudaStream_t stream = g_lib.stream;
  const bool two_inputs = op->kind == kKindAdd;
  if (op->in_on_device && op->out_on_device && (!two_inputs || op->in2_on_device)) {
    enum qnnp_status st = launch(op, op->input, op->input2, op->output, stream);
    if (st != qnnp_status_success || async) return st;
    return map_cuda(cudaStreamSynchronize(stream), "stream synchronize");
  }
  if (async) return qnnp_status_invalid_parameter;

  // host pointers: stage through device buffers inside the (synchronous) call.  Pinned (page-locked) host memory makes
  // these copies truly asynchronous DMA transfers; pageable memory goes through the driver's bounce buffers.
  const uint8_t* din = op->input;
  const uint8_t* din2 = op->input2;
  uint8_t* dout = op->output;
  enum qnnp_status st;
  if (!op->in_on_device) {
    if ((st = ensure_capacity(&op->d_in, &op->d_in_cap, op->in_span)) != qnnp_status_success) return st;
    if ((st = map_cuda(cudaMemcpyAsync(op->d_in, op->input, op->in_span, cudaMemcpyHostToDevice, stream), "H2D input")) !=
        qnnp_status_success)
      return st;
    din = op->d_in;
  }
  if (two_inputs && !op->in2_on_device) {
    if ((st = ensure_capacity(&op->d_in2, &op->d_in2_cap, op->in2_span)) != qnnp_status_success) return st;
    if ((st = map_cuda(cudaMemcpyAsync(op->d_in2, op->input2, op->in2_span, cudaMemcpyHostToDevice, stream), "H2D input 2")) !=
        qnnp_status_success)
      return st;
    din2 = op->d_in2;
  }
  if (!op->out_on_device) {
    if ((st = ensure_capacity(&op->d_out, &op->d_out_cap, op->out_span)) != qnnp_status_success) return st;
    dout = op->d_out;
    if (!op->out_dense) {
      // bytes between pixels must survive untouched, as in the reference (ukernels store exactly N bytes)
      if ((st = map_cuda(cudaMemcpyAsync(op->d_out, op->output, op->out_span, cudaMemcpyHostToDevice, stream),
                         "H2D output gaps")) != qnnp_status_success)
        return st;
    }
  }
  if ((st = launch(op, din, din2, dout, stream)) != qnnp_status_success) return st;
  if (!op->out_on_device) {
    if ((st = map_cuda(cudaMemcpyAsync(op->output, op->d_out, op->out_span, cudaMemcpyDeviceToHost, stream), "D2H output")) !=
        qnnp_status_success)
      return st;
  }
  return map_cuda(cudaStreamSynchronize(stream), "stream synchronize");
}

// Common tail of qnnp_setup_*: classify the pointers and, when the operator can run zero-copy, build its launch plan now
// (tensor maps, tiling, kernel variant) so that qnnp_run_operator only launches.
enum qnnp_status finish_setup(qnnp_operator* op, size_t in_pixels, size_t in_width, size_t out_pixels, size_t out_width) {
  // spans: (pixels - 1) * stride + bytes used in the last pixel
  op->in_span = (in_pixels - 1) * op->in_stride + in_width;
  op->in2_span = op->kind == kKindAdd ? (in_pixels - 1) * op->in2_stride + in_width : 0;
  op->out_span = (out_pixels - 1) * op->out_stride + out_width;
  op->out_dense = op->out_stride == out_width;
  op->in_on_device = is_device_pointer(op->input);
  op->out_on_device = is_device_pointer(op->output);
  op->in2_on_device = op->kind == kKindAdd ? is_device_pointer(op->input2) : false;
  if (op->plan != nullptr) op->plan->valid = false;
  if (op->in_on_device && op->out_on_device && (op->kind != kKindAdd || op->in2_on_device)) {
    bind_device();
    return build_plan(op, op->input, op->input2, op->output);
  }
  return qnnp_status_success;
}

size_t output_dimension(size_t padded_input, size_t kernel, size_t dilation, size_t subsampling) {
  const size_t effective_kernel = (kernel - 1) * dilation + 1;  // src/convolution.c:29-37
  return (padded_input - effective_kernel) / subsampling + 1;
}

}  // namespace

// ================================================================================================
// C ABI
// ================================================================================================
QNNP_EXPORT enum qnnp_status qnnp_initialize(void) {
  pthread_once(&g_once, init_once);
  return g_lib.init_status;
}

QNNP_EXPORT enum qnnp_status qnnp_deinitialize(void) { return qnnp_status_success; }

QNNP_EXPORT enum qnnp_status qnnp_create_convolution2d_nhwc_q8(
    uint32_t input_padding_top, uint32_t input_padding_right, uint32_t input_padding_bottom, uint32_t input_padding_left,
    uint32_t kernel_height, uint32_t kernel_width, uint32_t subsampling_height, uint32_t subsampling_width,
    uint32_t dilation_height, uint32_t dilation_width, uint32_t groups, size_t group_input_channels,
    size_t group_output_channels, uint8_t input_zero_point, float input_scale, uint8_t kernel_zero_point,
    float kernel_scale, const uint8_t* kernel, const int32_t* bias, uint8_t output_zero_point, float output_scale,
    uint8_t output_min, uint8_t output_max, uint32_t flags, qnnp_operator_t* convolution_out) {
  (void) flags;  // ignored by the reference as well (src/convolution.c:63)
  if (!g_lib.initialized) {
    log_error("qnnp_create_convolution2d_nhwc_q8 failed because QNNPACK is not properly initialized");
    return qnnp_status_uninitialized;
  }
  // validation order: src/convolution.c:74-115
  if (kernel_width == 0 || kernel_height == 0) {
    log_error("failed to create convolution with %ux%u kernel: kernel dimensions must be non-zero", kernel_width, kernel_height);
    return qnnp_status_invalid_parameter;
  }
  if (subsampling_width == 0 || subsampling_height == 0) {
    log_error("failed to create convolution with %ux%u subsampling: subsampling dimensions must be non-zero",
              subsampling_width, subsampling_height);
    return qnnp_status_invalid_parameter;
  }
  if (dilation_width == 0 || dilation_height == 0) {
    log_error("failed to create convolution with %ux%u dilation: dilation dimensions must be non-zero", dilation_width,
              dilation_height);
    return qnnp_status_invalid_parameter;
  }
  if (!scale_ok(input_scale) || !scale_ok(kernel_scale) || !scale_ok(output_scale)) {
    log_error("failed to create convolution with %.7g input, %.7g kernel, %.7g output scale: scales must be finite and positive",
              input_scale, kernel_scale, output_scale);
    return qnnp_status_invalid_parameter;
  }
  // fp32, in this order: src/convolution.c:161
  const float convolution_scale = input_scale * kernel_scale / output_scale;
  if (convolution_scale >= 1.0f) {
    log_error("failed to create convolution with %.7g input scale, %.7g kernel scale, and %.7g output scale: "
              "convolution scale %.7g is greater or equal to 1.0",
              input_scale, kernel_scale, output_scale, convolution_scale);
    return qnnp_status_unsupported_parameter;
  }
  if (!(convolution_scale >= 0x1.0p-32f)) {
    // the reference only asserts this (requantization.h:30); shifts > 31 are undefined there
    log_error("convolution scale %.7g is below 2^-32", convolution_scale);
    return qnnp_status_unsupported_parameter;
  }
  if (groups == 0 || group_input_channels == 0 || group_output_channels == 0) {
    log_error("failed to create convolution with %u groups, %zu/%zu channels per group", groups, group_input_channels,
              group_output_channels);
    return qnnp_status_invalid_parameter;
  }

  bind_device();
  qnnp_operator* op = new (std::nothrow) qnnp_operator();
  if (op == nullptr) return qnnp_status_out_of_memory;
  op->pad_top = input_padding_top, op->pad_right = input_padding_right;
  op->pad_bottom = input_padding_bottom, op->pad_left = input_padding_left;
  op->kh = kernel_height, op->kw = kernel_width;
  op->stride_h = subsampling_height, op->stride_w = subsampling_width;
  op->dil_h = dilation_height, op->dil_w = dilation_width;
  op->groups = groups, op->gic = group_input_channels, op->goc = group_output_channels;
  op->izp = input_zero_point, op->kzp = kernel_zero_point;
  op->rq = q8_make_requant(f32_bits(convolution_scale), output_zero_point, output_min, output_max);
  enable_bounded_requant(op, bias, groups * group_output_channels, (size_t) kernel_height * kernel_width * group_input_channels);
  op->rq_mode = select_rq_mode(op->rq);

  // kernel family (reference: src/convolution.c:180-189)
  const size_t kernel_size = (size_t) kernel_height * kernel_width;
  const bool any_padding = (input_padding_left | input_padding_top | input_padding_right | input_padding_bottom) != 0;
  enum qnnp_status st;
  if (kernel_height == 3 && kernel_width == 3 && group_input_channels == 1 && group_output_channels == 1 && groups > 1) {
    op->kind = kKindDw3x3;
    st = pack_dw3x3(op, kernel, bias);
  } else if (groups == 1) {
    op->kind = (kernel_size == 1 && subsampling_height == 1 && subsampling_width == 1 && !any_padding) ? kKindIgemmGemm
                                                                                                      : kKindIgemmConv;
    st = plan_and_pack_igemm(op, kernel, bias);
  } else {
    op->kind = kKindDirect;
    st = pack_direct(op, kernel, bias);
  }
  if (st != qnnp_status_success) {
    free_operator(op);
    return st;
  }
  *convolution_out = op;
  return qnnp_status_success;
}

QNNP_EXPORT enum qnnp_status qnnp_setup_convolution2d_nhwc_q8(
    qnnp_operator_t op, size_t batch_size, size_t input_height, size_t input_width, const uint8_t* input,
    size_t input_stride, uint8_t* output, size_t output_stride, pthreadpool_t threadpool) {
  (void) threadpool;
  if (!g_lib.initialized) return qnnp_status_uninitialized;
  if (op == nullptr) return qnnp_status_invalid_parameter;
  if (batch_size == 0) {  // src/convolution.c:396-399
    op->batch = 0;
    if (op->plan != nullptr) op->plan->valid = false;
    return qnnp_status_success;
  }
  if (input_width == 0 || input_height == 0) {
    log_error("failed to setup convolution with %zux%zu input: input dimensions must be non-zero", input_width, input_height);
    return qnnp_status_invalid_parameter;
  }
  op->batch = batch_size;
  op->in_h = input_height, op->in_w = input_width;
  op->input = input, op->in_stride = input_stride;
  op->out_h = output_dimension(op->pad_top + input_height + op->pad_bottom, op->kh, op->dil_h, op->stride_h);
  op->out_w = output_dimension(op->pad_left + input_width + op->pad_right, op->kw, op->dil_w, op->stride_w);
  op->output = output, op->out_stride = output_stride;
  return finish_setup(op, op->batch * op->in_h * op->in_w, op->groups * op->gic, op->batch * op->out_h * op->out_w,
                      op->groups * op->goc);
}

QNNP_EXPORT enum qnnp_status qnnp_create_fully_connected_nc_q8(
    size_t input_channels, size_t output_channels, uint8_t input_zero_point, float input_scale,
    uint8_t kernel_zero_point, float kernel_scale, const uint8_t* kernel, const int32_t* bias,
    uint8_t output_zero_point, float output_scale, uint8_t output_min, uint8_t output_max, uint32_t flags,
    qnnp_operator_t* fully_connected_out) {
  (void) flags;
  if (!g_lib.initialized) {
    log_error("qnnp_create_fully_connected_nc_q8 failed because QNNPACK is not properly initialized");
    return qnnp_status_uninitialized;
  }
  if (!scale_ok(input_scale) || !scale_ok(kernel_scale) || !scale_ok(output_scale)) {  // src/fully-connected.c:49-65
    log_error("failed to create fully connected operator with %.7g input, %.7g kernel, %.7g output scale: "
              "scales must be finite and positive", input_scale, kernel_scale, output_scale);
    return qnnp_status_invalid_parameter;
  }
  const float requantization_scale = input_scale * kernel_scale / output_scale;  // src/fully-connected.c:71
  if (requantization_scale >= 1.0f || !(requantization_scale >= 0x1.0p-32f)) {
    log_error("failed to create fully connected operator: requantization scale %.7g is outside [2^-32, 1)",
              requantization_scale);
    return qnnp_status_unsupported_parameter;
  }
  if (input_channels == 0 || output_channels == 0) return qnnp_status_invalid_parameter;
  bind_device();
  qnnp_operator* op = new (std::nothrow) qnnp_operator();
  if (op == nullptr) return qnnp_status_out_of_memory;
  op->is_fc = true;
  op->groups = 1, op->gic = input_channels, op->goc = output_channels;
  op->izp = input_zero_point, op->kzp = kernel_zero_point;
  op->rq = q8_make_requant(f32_bits(requantization_scale), output_zero_point, output_min, output_max);
  enable_bounded_requant(op, bias, output_channels, input_channels);
  op->rq_mode = select_rq_mode(op->rq);
  op->kind = kKindIgemmGemm;
  enum qnnp_status st = plan_and_pack_igemm(op, kernel, bias);
  if (st != qnnp_status_success) {
    free_operator(op);
    return st;
  }
  *fully_connected_out = op;
  return qnnp_status_success;
}

QNNP_EXPORT enum qnnp_status qnnp_setup_fully_connected_nc_q8(
    qnnp_operator_t op, size_t batch_size, const uint8_t* input, size_t input_stride, uint8_t* output,
    size_t output_stride) {
  if (!g_lib.initialized) return qnnp_status_uninitialized;
  if (op == nullptr) return qnnp_status_invalid_parameter;
  if (batch_size == 0) {
    op->batch = 0;
    if (op->plan != nullptr) op->plan->valid = false;
    return qnnp_status_success;
  }
  // src/fully-connected.c:149-158: one "image" of batch_size x 1 pixels
  op->batch = 1;
  op->in_h = batch_size, op->in_w = 1, op->out_h = batch_size, op->out_w = 1;
  op->input = input, op->in_stride = input_stride;
  op->output = output, op->out_stride = output_stride;
  return finish_setup(op, batch_size, op->gic, batch_size, op->goc);
}

QNNP_EXPORT enum qnnp_status qnnp_run_operator(qnnp_operator_t op, pthreadpool_t threadpool) {
  (void) threadpool;
  return run_impl(op, false);
}

QNNP_EXPORT enum qnnp_status qnnp_delete_operator(qnnp_operator_t op) {
  if (op == nullptr) return qnnp_status_invalid_parameter;  // src/operator-delete.c:17
  free_operator(op);
  return qnnp_status_success;
}

// ---- CUDA extensions (include/qnnpack_cuda.h) -----------------------------------------------------
QNNP_EXPORT enum qnnp_status qnnp_cuda_set_stream(void* s) {
  if (!g_lib.initialized) return qnnp_status_uninitialized;
  g_lib.stream = s != nullptr ? (cudaStream_t) s : g_lib.own_stream;
  return qnnp_status_success;
}
QNNP_EXPORT void* qnnp_cuda_get_stream(void) { return (void*) g_lib.stream; }
QNNP_EXPORT int qnnp_cuda_get_device(void) { return g_lib.device; }
QNNP_EXPORT enum qnnp_status qnnp_cuda_run_operator_async(qnnp_operator_t op) { return run_impl(op, true); }
QNNP_EXPORT enum qnnp_status qnnp_cuda_operator_packed_weights(qnnp_operator_t op, void** device_ptr, size_t* size_bytes) {
  if (op == nullptr || device_ptr == nullptr || size_bytes == nullptr) return qnnp_status_invalid_parameter;
  *device_ptr = op->d_weights;
  *size_bytes = op->weights_bytes;
  return qnnp_status_success;
}
QNNP_EXPORT enum qnnp_status qnnp_cuda_operator_packed_bias(qnnp_operator_t op, void** device_ptr, size_t* size_bytes) {
  if (op == nullptr || device_ptr == nullptr || size_bytes == nullptr) return qnnp_status_invalid_parameter;
  *device_ptr = op->d_bias;
  *size_bytes = op->bias_count * sizeof(int32_t);
  return qnnp_status_success;
}
/* Measured dense int8 tensor-core peak (tera-ops/s) of this device: smem-resident tcgen05.mma kind::i8 loop,
 * `reps` timed launches of `iters` x 8 UMMAs per SM (q8_peak_sm100.cu). */
QNNP_EXPORT enum qnnp_status qnnp_cuda_measure_int8_peak(int iters, int reps, double* tops, double* ms_per_launch) {
  if (!g_lib.initialized) return qnnp_status_uninitialized;
  if (iters <= 0 || reps <= 0 || tops == nullptr || ms_per_launch == nullptr) return qnnp_status_invalid_parameter;
  bind_device();
  const cudaError_t e = q8::measure_int8_peak(g_lib.num_sms, iters, reps, g_lib.stream, tops, ms_per_launch);
  if (e == cudaSuccess) g_lib.launches.fetch_add((unsigned long long) reps + 1);
  return map_cuda(e, "qnnp_cuda_measure_int8_peak");
}
QNNP_EXPORT unsigned long long qnnp_cuda_launch_count(void) { return g_lib.launches.load(); }
QNNP_EXPORT unsigned long long qnnp_cuda_debug_dw_umma_launch_count(void) { return g_lib.dw_umma_launches.load(); }
QNNP_EXPORT int qnnp_cuda_debug_plan_igemm(size_t k, size_t n, uint32_t groups, int folded, int bias_steps, int out[24]) {
  IgemmPlan pl;
  const int optin = g_lib.initialized ? g_lib.max_smem_optin : 232448;  // B200: 227 KB opt-in
  if (!plan_igemm(k, n, groups, optin, folded, bias_steps, &pl)) return 0;
  const int v[24] = {pl.K, pl.nkc, pl.skc, pl.k_stages, pl.mt, pl.n_tiles, pl.n_tile, pl.n_mma, pl.has_corr, pl.b_resident,
                     pl.num_stages, pl.stage_bytes, pl.staging_bytes, pl.bias_bytes, pl.smem_b_off, pl.smem_bias_off,
                     pl.smem_a_off, pl.smem_stage_off, pl.smem_total, pl.bulk_capable, pl.folded, pl.bias_steps,
                     pl.blk_chunks, pl.good};
  for (int i = 0; i < 24; i++) out[i] = v[i];
  return 1;
}
/* Panel-epilogue tables for an n-tile of `n_tile` columns, `mt` sub-tiles per item (CPU-callable; tests/test_planner.py
 * replays the staging writes and the swizzled tensor-store reads on them).  out: [0] panels, [1] box_rows,
 * [2+4k..] col0, width, off, map of panel k (4 panels), [18+2c..] x, y of unit c (16 units). */
QNNP_EXPORT void qnnp_cuda_debug_panel_tables(int n_tile, int mt, int folded, int out[50]) {
  q8::IgemmParams p{};
  p.n_tile = n_tile, p.mt = mt, p.folded = folded & 1;
  fill_panel_tables(p, (folded & 2) != 0);  // bit 1 of `folded`: the dense single-image mode
  out[0] = p.e2_panels, out[1] = p.e2_box_rows;
  for (int k = 0; k < 4; k++) out[2 + 4 * k] = p.e2_col0[k], out[3 + 4 * k] = p.e2_width[k], out[4 + 4 * k] = p.e2_off[k], out[5 + 4 * k] = p.e2_map[k];
  for (int c = 0; c < 16; c++) out[18 + 2 * c] = (int) p.e2_unit[c].x, out[19 + 2 * c] = (int) p.e2_unit[c].y;
}
/* Depthwise tensor-core tiling for a geometry (CPU-callable): fills out[40], returns 0 when the shape is not eligible. */
QNNP_EXPORT int qnnp_cuda_debug_plan_dwconv(int channels, int batch, int in_h, int in_w, int out_h, int out_w, int stride,
                                            int pad_top, int pad_left, int wmode, int out[40]) {
  q8::DwTcParams p;
  const int optin = g_lib.initialized ? g_lib.max_smem_optin : 232448;
  if (!plan_dw_umma(channels, batch, in_h, in_w, out_h, out_w, stride, pad_top, pad_left, wmode, optin, &p)) return 0;
  const int v[40] = {p.G, p.mt, p.xt, p.yt, p.nt, p.nb, p.Q, p.whole, p.planes, p.box_rows, p.box_px, p.plane_tx, p.plane_bytes,
                     p.a_bytes, p.b_bytes, p.cg_bytes, p.stage_bytes, p.num_stages, p.smem_total, p.x_org[0], p.x_org[1],
                     p.a_off[0], p.a_off[1], p.a_off[2], p.a_off[3], p.a_off[4], p.a_lbo[0], p.a_lbo[1], p.a_lbo[2], p.a_lbo[3],
                     p.a_lbo[4], p.sbo, p.nb_cols, p.b_signed, p.acc_stride, p.cblocks, p.cgs, (int) p.total_items, 0, 0};
  for (int i = 0; i < 40; i++) out[i] = v[i];
  return 1;
}
/* Channel-pair plan of the depthwise tensor-core kernel (DwTcParams::pair).  out[0..37] as qnnp_cuda_debug_plan_dwconv,
 * out[38] = 1, out[39..47] = a_off9[ky*3+kx]. */
QNNP_EXPORT int qnnp_cuda_debug_plan_dwconv32(int channels, int batch, int in_h, int in_w, int out_h, int out_w, int stride,
                                              int pad_top, int pad_left, int wmode, int out[48]) {
  q8::DwTcParams p;
  const int optin = g_lib.initialized ? g_lib.max_smem_optin : 232448;
  if (!plan_dw_umma(channels, batch, in_h, in_w, out_h, out_w, stride, pad_top, pad_left, wmode, optin, &p, 1)) return 0;
  const int v[48] = {p.G, p.mt, p.xt, p.yt, p.nt, p.nb, p.Q, p.whole, p.planes, p.box_rows, p.box_px, p.plane_tx, p.plane_bytes,
                     p.a_bytes, p.b_bytes, p.cg_bytes, p.stage_bytes, p.num_stages, p.smem_total, p.x_org[0], p.x_org[1],
                     0, 0, 0, 0, 0, 0, 0, 0, 0, 0, p.sbo, p.nb_cols, p.b_signed, p.acc_stride, p.cblocks, p.cgs, (int) p.total_items,
                     1, p.a_off9[0], p.a_off9[1], p.a_off9[2], p.a_off9[3], p.a_off9[4], p.a_off9[5], p.a_off9[6], p.a_off9[7],
                     p.a_off9[8]};
  for (int i = 0; i < 48; i++) out[i] = v[i];
  return 1;
}
/* Border-class bias table of the depthwise plan (either form), see qnnpack_cuda.h. */
QNNP_EXPORT int qnnp_cuda_debug_plan_dwconv_bias(int channels, int batch, int in_h, int in_w, int out_h, int out_w, int stride,
                                                 int pad_top, int pad_left, int wmode, int pair, int out[12]) {
  q8::DwTcParams p;
  const int optin = g_lib.initialized ? g_lib.max_smem_optin : 232448;
  if (!plan_dw_umma(channels, batch, in_h, in_w, out_h, out_w, stride, pad_top, pad_left, wmode, optin, &p, pair)) return 0;
  const int v[12] = {p.bias_smem, p.bias_off, p.bias_rstride, p.bias_nrc, p.bias_ncc, (int) p.bias_rslot, (int) p.bias_cslot,
                     (int) p.bias_rcls, (int) p.bias_ccls, p.smem_total, p.num_stages, p.stage_bytes};
  for (int i = 0; i < 12; i++) out[i] = v[i];
  return 1;
}
/* Channel-pair B operands (pack_dw_umma32_host): wpack must hold ceil(channels / 32) * 9 * 1024 bytes.  Returns the operand
 * mode (dw_tc_wmode), or -1 when the pair form does not apply. */
QNNP_EXPORT int qnnp_cuda_debug_pack_dwconv32(size_t channels, uint8_t kernel_zero_point, const uint8_t* kernel, uint8_t* wpack) {
  if (channels < 32 || (channels % 16) != 0) return -1;
  const int wmode = dw_tc_wmode(channels, kernel, kernel_zero_point);
  if (wmode == 2) return -1;
  std::vector<uint8_t> wp;
  pack_dw_umma32_host(channels, kernel, kernel_zero_point, wmode, wp);
  memcpy(wpack, wp.data(), wp.size());
  return wmode;
}
/* Packed operands of the tensor-core kernel for a K x N fully-connected / 1x1 operator, built on the host (no GPU needed).
 * meta = {folded, nkc, n_tiles, n_tile, n_mma, blk_chunks, bias_steps, b_signed, has_b2, k_tail_pad, has_corr, 0...}.
 * Returns 1 and fills blob / folded_bias (sizes in *blob_bytes / *bias_count; pass capacities in), 0 on failure. */
QNNP_EXPORT int qnnp_cuda_debug_pack_igemm(size_t k, size_t n, uint8_t input_zero_point, uint8_t kernel_zero_point,
                                           const uint8_t* kernel, const int32_t* bias, int meta[16], uint8_t* blob,
                                           size_t* blob_bytes, int32_t* folded_bias, size_t* bias_count) {
  qnnp_operator op;
  op.kind = kKindIgemmGemm;
  op.groups = 1, op.gic = k, op.goc = n;
  op.izp = input_zero_point, op.kzp = kernel_zero_point;
  std::vector<uint8_t> b;
  std::vector<int32_t> fb;
  if (pack_igemm_host(&op, kernel, bias, b, fb) != qnnp_status_success) return 0;
  if (b.size() > *blob_bytes || fb.size() > *bias_count) return 0;
  memcpy(blob, b.data(), b.size());
  memcpy(folded_bias, fb.data(), fb.size() * sizeof(int32_t));
  *blob_bytes = b.size(), *bias_count = fb.size();
  const int v[16] = {op.folded, op.nkc, op.n_tiles, op.n_tile, op.n_mma, op.blk_chunks, op.bias_steps, op.b_signed, op.has_b2,
                     op.k_tail_pad, op.has_corr, 0, 0, 0, 0, 0};
  for (int i = 0; i < 16; i++) meta[i] = v[i];
  return 1;
}
/* Operands of the depthwise tensor-core kernel for C channels (C % 16 == 0), built on the host; needs no GPU.
 * wpack: (C/16) * 5 * 2 * nb_cols * 16 bytes (nb_cols = 32 for wmode 2, else 16); bias_cls: 64 * C int32.
 * Returns the weight-operand mode (0 / 1 / 2) the library would choose, or -1. */
QNNP_EXPORT int qnnp_cuda_debug_pack_dwconv(size_t channels, uint8_t input_zero_point, uint8_t kernel_zero_point,
                                            const uint8_t* kernel, const int32_t* bias, int u_form, uint8_t* wpack,
                                            int32_t* bias_cls) {
  if (channels == 0 || (channels % 16) != 0) return -1;
  const int wmode = dw_tc_wmode(channels, kernel, kernel_zero_point);
  std::vector<uint8_t> wp;
  std::vector<int32_t> bc;
  pack_dw_umma_host(channels, kernel, bias, input_zero_point, kernel_zero_point, wmode, u_form != 0, wp, bc);
  memcpy(wpack, wp.data(), wp.size());
  memcpy(bias_cls, bc.data(), bc.size() * sizeof(int32_t));
  return wmode;
}
/* 1 if the operator runs in folded mode (bias + zero-point correction on the tensor core), 0 otherwise. */
QNNP_EXPORT int qnnp_cuda_debug_operator_is_folded(qnnp_operator_t op) { return op != nullptr && op->folded ? 1 : 0; }
QNNP_EXPORT void qnnp_cuda_debug_set_accumulator_dump(int32_t* device_buffer) { g_lib.dbg_acc = device_buffer; }
QNNP_EXPORT const char* qnnp_cuda_operator_kernel_name(qnnp_operator_t op) {
  if (op == nullptr) return "null";
  switch (op->kind) {
    case kKindIgemmGemm: return "igemm-gemm";
    case kKindIgemmConv: return "igemm-conv";
    case kKindDw3x3: return "dwconv3x3";
    case kKindDirect: return "direct";
    default: return "none";
  }
}

QNNP_EXPORT enum qnnp_status qnnp_cuda_requantize_q31(
    size_t n, const int32_t* input, float scale, uint8_t zero_point, uint8_t qmin, uint8_t qmax, uint8_t* output) {
  if (!g_lib.initialized) return qnnp_status_uninitialized;
  if (!(scale < 1.0f) || !(scale >= 0x1.0p-32f)) return qnnp_status_unsupported_parameter;
  if (n == 0) return qnnp_status_success;
  bind_device();
  const Q8Requant rq = q8_make_requant(f32_bits(scale), zero_point, qmin, qmax);
  cudaStream_t stream = g_lib.stream;
  const bool in_dev = is_device_pointer(input), out_dev = is_device_pointer(output);
  int32_t* din = const_cast<int32_t*>(input);
  uint8_t* dout = output;
  cudaError_t e = cudaSuccess;
  if (!in_dev) {
    e = cudaMalloc((void**) &din, n * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMemcpyAsync(din, input, n * sizeof(int32_t), cudaMemcpyHostToDevice, stream);
  }
  if (e == cudaSuccess && !out_dev) e = cudaMalloc((void**) &dout, n);
  if (e == cudaSuccess) e = q8::launch_q8_requantize(din, dout, (long long) n, rq, stream);
  if (e == cudaSuccess) g_lib.launches.fetch_add(1);
  if (e == cudaSuccess && !out_dev) e = cudaMemcpyAsync(output, dout, n, cudaMemcpyDeviceToHost, stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(stream);
  if (!in_dev) cudaFree(din);
  if (!out_dev) cudaFree(dout);
  return map_cuda(e, "qnnp_cuda_requantize_q31");
}

// ================================================================================================
// operators beside the convolution path (SURVEY.md §8f rows 1, 3, 4): each mirrors the reference's validation order
// and status codes; quantisation parameters restate src/qnnpack/requantization.h with the same fp32 operations.
// ================================================================================================
namespace {

float f32_from_bits(uint32_t u) {
  float f;
  memcpy(&f, &u, sizeof f);
  return f;
}

// qnnp_compute_avgpool_quantization_params, scalar member (src/qnnpack/requantization.h:200-265)
q8::AvgQuant make_avg_quant(float scale, uint8_t ozp, uint8_t omin, uint8_t omax) {
  const uint32_t bits = f32_bits(scale);
  q8::AvgQuant q;
  q.multiplier = (int32_t) ((bits & 0x007FFFFFu) | 0x00800000u);
  const int32_t shift = 127 + 23 - (int32_t) (bits >> 23);
  q.right_shift = (uint32_t) shift;
  q.rounding = (int64_t) 1 << (shift - 1);
  q.min_less_zp = (int32_t) omin - (int32_t) ozp;
  q.max_less_zp = (int32_t) omax - (int32_t) ozp;
  q.zero_point = ozp;
  return q;
}

qnnp_operator* new_operator(KernelKind kind) {
  qnnp_operator* op = new (std::nothrow) qnnp_operator();
  if (op != nullptr) op->kind = kind;
  return op;
}

enum qnnp_status upload(void** dst, const void* src, size_t bytes) {
  cudaError_t e = cudaMalloc(dst, bytes);
  if (e == cudaSuccess) e = cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice);
  return map_cuda(e, "uploading operator table");
}

// nc operators: batch rows of `channels` bytes
enum qnnp_status setup_nc(qnnp_operator* op, size_t batch, const uint8_t* x, size_t x_stride, uint8_t* y, size_t y_stride) {
  if (!g_lib.initialized) return qnnp_status_uninitialized;
  if (op == nullptr) return qnnp_status_invalid_parameter;
  if (batch == 0) {
    op->batch = 0;
    if (op->plan != nullptr) op->plan->valid = false;
    return qnnp_status_success;
  }
  op->batch = batch;
  op->input = x, op->in_stride = x_stride;
  op->output = y, op->out_stride = y_stride;
  return finish_setup(op, batch, op->channels, batch, op->channels);
}

}  // namespace

// ---- deconvolution (src/deconvolution.c:38-277): the direct kernel with the transposed tap mapping ----------------------
QNNP_EXPORT enum qnnp_status qnnp_create_deconvolution2d_nhwc_q8(
    uint32_t input_padding_top, uint32_t input_padding_right, uint32_t input_padding_bottom, uint32_t input_padding_left,
    uint32_t adjustment_height, uint32_t adjustment_width, uint32_t kernel_height, uint32_t kernel_width, uint32_t stride_height,
    uint32_t stride_width, uint32_t dilation_height, uint32_t dilation_width, uint32_t groups, size_t group_input_channels,
    size_t group_output_channels, uint8_t input_zero_point, float input_scale, uint8_t kernel_zero_point, float kernel_scale,
    const uint8_t* kernel, const int32_t* bias, uint8_t output_zero_point, float output_scale, uint8_t output_min,
    uint8_t output_max, uint32_t flags, qnnp_operator_t* deconvolution_out) {
  (void) flags;
  if (!g_lib.initialized) {
    log_error("qnnp_create_deconvolution2d_nhwc_q8 failed because QNNPACK is not properly initialized");
    return qnnp_status_uninitialized;
  }
  if (kernel_width == 0 || kernel_height == 0 || stride_width == 0 || stride_height == 0 || dilation_width == 0 ||
      dilation_height == 0) {  // src/deconvolution.c:77-96
    log_error("failed to create deconvolution: kernel, stride and dilation dimensions must be non-zero");
    return qnnp_status_invalid_parameter;
  }
  if (!scale_ok(input_scale) || !scale_ok(kernel_scale) || !scale_ok(output_scale)) {
    log_error("failed to create deconvolution with %.7g input, %.7g kernel, %.7g output scale: scales must be finite and positive",
              input_scale, kernel_scale, output_scale);
    return qnnp_status_invalid_parameter;
  }
  const float deconvolution_scale = input_scale * kernel_scale / output_scale;  // src/deconvolution.c:118
  if (deconvolution_scale >= 1.0f || !(deconvolution_scale >= 0x1.0p-32f)) {
    log_error("failed to create deconvolution: scale %.7g is outside [2^-32, 1)", deconvolution_scale);
    return qnnp_status_unsupported_parameter;
  }
  if (groups == 0 || group_input_channels == 0 || group_output_channels == 0) return qnnp_status_invalid_parameter;
  bind_device();
  qnnp_operator* op = new_operator(kKindDirect);
  if (op == nullptr) return qnnp_status_out_of_memory;
  op->is_deconv = true;
  op->pad_top = input_padding_top, op->pad_right = input_padding_right;
  op->pad_bottom = input_padding_bottom, op->pad_left = input_padding_left;
  op->adj_h = adjustment_height, op->adj_w = adjustment_width;
  op->kh = kernel_height, op->kw = kernel_width;
  op->stride_h = stride_height, op->stride_w = stride_width;
  op->dil_h = dilation_height, op->dil_w = dilation_width;
  op->groups = groups, op->gic = group_input_channels, op->goc = group_output_channels;
  op->izp = input_zero_point, op->kzp = kernel_zero_point;
  op->rq = q8_make_requant(f32_bits(deconvolution_scale), output_zero_point, output_min, output_max);
  op->rq_mode = select_rq_mode(op->rq);
  // the deconvolution kernel is [group][input channel][ky][kx][output channel] (test/deconvolution-operator-tester.h:411,
  // src/qnnpack/pack.h:93-133); bring it to the convolution layout [group][output channel][ky][kx][input channel]
  const size_t ks = (size_t) kernel_height * kernel_width;
  std::vector<uint8_t> kt((size_t) groups * group_output_channels * ks * group_input_channels);
  for (size_t g = 0; g < groups; g++)
    for (size_t ic = 0; ic < group_input_channels; ic++)
      for (size_t t = 0; t < ks; t++)
        for (size_t oc = 0; oc < group_output_channels; oc++)
          kt[((g * group_output_channels + oc) * ks + t) * group_input_channels + ic] =
              kernel[((g * group_input_channels + ic) * ks + t) * group_output_channels + oc];
  const enum qnnp_status st = pack_direct(op, kt.data(), bias);
  if (st != qnnp_status_success) {
    free_operator(op);
    return st;
  }
  *deconvolution_out = op;
  return qnnp_status_success;
}

QNNP_EXPORT enum qnnp_status qnnp_setup_deconvolution2d_nhwc_q8(qnnp_operator_t op, size_t batch_size, size_t input_height,
                                                                size_t input_width, const uint8_t* input, size_t input_stride,
                                                                uint8_t* output, size_t output_stride, pthreadpool_t threadpool) {
  (void) threadpool;
  if (!g_lib.initialized) return qnnp_status_uninitialized;
  if (op == nullptr || !op->is_deconv) return qnnp_status_invalid_parameter;
  if (batch_size == 0) {
    op->batch = 0;
    if (op->plan != nullptr) op->plan->valid = false;
    return qnnp_status_success;
  }
  if (input_width == 0 || input_height == 0) return qnnp_status_invalid_parameter;
  op->batch = batch_size;
  op->in_h = input_height, op->in_w = input_width;
  op->input = input, op->in_stride = input_stride;
  // src/deconvolution.c:25-36: stride * (in - 1) + adjustment + effective kernel - total padding
  op->out_h = op->stride_h * (input_height - 1) + op->adj_h + ((op->kh - 1) * op->dil_h + 1) - (op->pad_top + op->pad_bottom);
  op->out_w = op->stride_w * (input_width - 1) + op->adj_w + ((op->kw - 1) * op->dil_w + 1) - (op->pad_left + op->pad_right);
  op->output = output, op->out_stride = output_stride;
  return finish_setup(op, batch_size * input_height * input_width, op->groups * op->gic, batch_size * op->out_h * op->out_w,
                      op->groups * op->goc);
}

// ---- add (src/add.c:22-149) ---------------------------------------------------------------------------------------------
QNNP_EXPORT enum qnnp_status qnnp_create_add_nc_q8(size_t channels, uint8_t a_zero_point, float a_scale, uint8_t b_zero_point,
                                                   float b_scale, uint8_t sum_zero_point, float sum_scale, uint8_t sum_min,
                                                   uint8_t sum_max, uint32_t flags, qnnp_operator_t* add_out) {
  (void) flags;
  if (!g_lib.initialized) {
    log_error("qnnp_create_add_nc_q8 failed because QNNPACK is not properly initialized");
    return qnnp_status_uninitialized;
  }
  if (channels == 0) {
    log_error("failed to create add operator with %zu channels: number of channels must be non-zero", channels);
    return qnnp_status_invalid_parameter;
  }
  if (!scale_ok(a_scale) || !scale_ok(b_scale) || !scale_ok(sum_scale)) {
    log_error("failed to create add operator with %.7g A, %.7g B, %.7g output scale: scales must be finite and positive", a_scale,
              b_scale, sum_scale);
    return qnnp_status_invalid_parameter;
  }
  if (sum_min >= sum_max) {
    log_error("failed to create add operator with [%u, %u] output range: range min must be below range max", sum_min, sum_max);
    return qnnp_status_invalid_parameter;
  }
  const float a_output_scale = a_scale / sum_scale, b_output_scale = b_scale / sum_scale;
  if (a_output_scale < 0x1.0p-14f || a_output_scale >= 0x1.0p+8f || b_output_scale < 0x1.0p-14f || b_output_scale >= 0x1.0p+8f) {
    log_error("failed to create add operator: scale ratios %.7g / %.7g must be in [2**-14, 2**8)", a_output_scale, b_output_scale);
    return qnnp_status_unsupported_parameter;
  }
  qnnp_operator* op = new_operator(kKindAdd);
  if (op == nullptr) return qnnp_status_out_of_memory;
  op->channels = channels;
  // qnnp_compute_add_quantization_params (src/qnnpack/requantization.h:327-414), same fp32 operations in the same order
  const float max_output_scale = a_output_scale > b_output_scale ? a_output_scale : b_output_scale;
  const int32_t max_scale_exponent = (int32_t) (f32_bits(max_output_scale) >> 23) - 127;
  const uint32_t shift = (uint32_t) (21 - max_scale_exponent);
  const float scale_multiplier = f32_from_bits((uint32_t) (21 - max_scale_exponent + 127) << 23);
  const uint32_t a_multiplier = (uint32_t) (int32_t) lrintf(a_output_scale * scale_multiplier);
  const uint32_t b_multiplier = (uint32_t) (int32_t) lrintf(b_output_scale * scale_multiplier);
  q8::AddParams& q = op->add;
  q.a_multiplier = a_multiplier, q.b_multiplier = b_multiplier;
  q.shift = (int32_t) shift;
  q.remainder_mask = (int32_t) ((1u << shift) - 1u);
  q.remainder_threshold = (int32_t) (((1u << shift) - 1u) >> 1);
  q.zero_point_product = (int32_t) (0u - (a_multiplier * (uint32_t) a_zero_point + b_multiplier * (uint32_t) b_zero_point));
  q.y_zero_point = sum_zero_point, q.y_min = sum_min, q.y_max = sum_max;
  *add_out = op;
  return qnnp_status_success;
}

QNNP_EXPORT enum qnnp_status qnnp_setup_add_nc_q8(qnnp_operator_t op, size_t batch_size, const uint8_t* a, size_t a_stride,
                                                  const uint8_t* b, size_t b_stride, uint8_t* sum, size_t sum_stride) {
  if (!g_lib.initialized) return qnnp_status_uninitialized;
  if (op == nullptr || op->kind != kKindAdd) return qnnp_status_invalid_parameter;
  op->input2 = b, op->in2_stride = b_stride;
  return setup_nc(op, batch_size, a, a_stride, sum, sum_stride);
}

// ---- global average pooling (src/global-average-pooling.c:22-147) ---------------------------------------------------------
QNNP_EXPORT enum qnnp_status qnnp_create_global_average_pooling_nwc_q8(size_t channels, uint8_t input_zero_point, float input_scale,
                                                                       uint8_t output_zero_point, float output_scale,
                                                                       uint8_t output_min, uint8_t output_max, uint32_t flags,
                                                                       qnnp_operator_t* global_average_pooling_out) {
  (void) flags;
  if (!g_lib.initialized) {
    log_error("qnnp_create_global_average_pooling_nwc_q8 failed because QNNPACK is not properly initialized");
    return qnnp_status_uninitialized;
  }
  if (channels == 0 || !scale_ok(input_scale) || !scale_ok(output_scale)) {
    log_error("failed to create global average pooling operator: channels must be non-zero, scales finite and positive");
    return qnnp_status_invalid_parameter;
  }
  const float input_output_scale = input_scale / output_scale;
  if (input_output_scale < 0x1.0p-8f || input_output_scale >= 0x1.0p+8f) {
    log_error("failed to create global average pooling operator with %.7g input-to-output scale ratio: must be in [2**-8, 2**8)",
              input_output_scale);
    return qnnp_status_unsupported_parameter;
  }
  qnnp_operator* op = new_operator(kKindGavgPool);
  if (op == nullptr) return qnnp_status_out_of_memory;
  op->channels = channels;
  op->izp = input_zero_point, op->ozp = output_zero_point, op->omin = output_min, op->omax = output_max;
  op->in_scale = input_scale, op->out_scale = output_scale;
  *global_average_pooling_out = op;
  return qnnp_status_success;
}

QNNP_EXPORT enum qnnp_status qnnp_setup_global_average_pooling_nwc_q8(qnnp_operator_t op, size_t batch_size, size_t width,
                                                                      const uint8_t* input, size_t input_stride, uint8_t* output,
                                                                      size_t output_stride) {
  if (!g_lib.initialized) return qnnp_status_uninitialized;
  if (op == nullptr || op->kind != kKindGavgPool) return qnnp_status_invalid_parameter;
  if (batch_size == 0) {
    op->batch = 0;
    if (op->plan != nullptr) op->plan->valid = false;
    return qnnp_status_success;
  }
  if (width == 0) {
    log_error("failed to setup global average pooling operator with width %zu: width must be non-zero", width);
    return qnnp_status_invalid_parameter;
  }
  op->batch = batch_size, op->in_w = width, op->in_h = 1;
  op->input = input, op->in_stride = input_stride;
  op->output = output, op->out_stride = output_stride;
  // src/global-average-pooling.c:135-141: scale = input_scale / (output_scale * width), fp32 in this order
  op->avgq = make_avg_quant(op->in_scale / (op->out_scale * (float) width), op->ozp, op->omin, op->omax);
  return finish_setup(op, batch_size * width, op->channels, batch_size, op->channels);
}

// ---- average / max pooling (src/average-pooling.c:36-275, src/max-pooling.c:36-223) --------------------------------------
QNNP_EXPORT enum qnnp_status qnnp_create_average_pooling2d_nhwc_q8(
    uint32_t input_padding_top, uint32_t input_padding_right, uint32_t input_padding_bottom, uint32_t input_padding_left,
    uint32_t pooling_height, uint32_t pooling_width, uint32_t stride_height, uint32_t stride_width, size_t channels,
    uint8_t input_zero_point, float input_scale, uint8_t output_zero_point, float output_scale, uint8_t output_min,
    uint8_t output_max, uint32_t flags, qnnp_operator_t* average_pooling_out) {
  (void) flags;
  if (!g_lib.initialized) {
    log_error("qnnp_create_average_pooling2d_nhwc_q8 failed because QNNPACK is not properly initialized");
    return qnnp_status_uninitialized;
  }
  const uint32_t pooling_size = pooling_height * pooling_width;
  if (pooling_size == 0 || pooling_size == 1 || stride_height == 0 || stride_width == 0 || channels == 0 ||
      !scale_ok(input_scale) || !scale_ok(output_scale)) {  // src/average-pooling.c:66-113 (1x1 pooling is rejected there too)
    log_error("failed to create average pooling with %ux%u pooling, %ux%u stride, %zu channels", pooling_width, pooling_height,
              stride_width, stride_height, channels);
    return qnnp_status_invalid_parameter;
  }
  const float input_output_scale = input_scale / output_scale;
  if (input_output_scale < 0x1.0p-8f || input_output_scale >= 0x1.0p+8f || pooling_size >= 16777216) {
    log_error("failed to create average pooling: scale ratio %.7g must be in [2**-8, 2**8), pooling size below 2**24",
              input_output_scale);
    return qnnp_status_unsupported_parameter;
  }
  qnnp_operator* op = new_operator(kKindAvgPool);
  if (op == nullptr) return qnnp_status_out_of_memory;
  op->pad_top = input_padding_top, op->pad_right = input_padding_right;
  op->pad_bottom = input_padding_bottom, op->pad_left = input_padding_left;
  op->kh = pooling_height, op->kw = pooling_width, op->stride_h = stride_height, op->stride_w = stride_width;
  op->channels = channels;
  op->izp = input_zero_point, op->omin = output_min, op->omax = output_max, op->ozp = output_zero_point;
  // src/average-pooling.c:158-163: scale = input_scale / (output_scale * pooling_size); padded taps count (they read izp)
  op->avgq = make_avg_quant(input_scale / (output_scale * (float) pooling_size), output_zero_point, output_min, output_max);
  *average_pooling_out = op;
  return qnnp_status_success;
}

QNNP_EXPORT enum qnnp_status qnnp_create_max_pooling2d_nhwc_u8(
    uint32_t input_padding_top, uint32_t input_padding_right, uint32_t input_padding_bottom, uint32_t input_padding_left,
    uint32_t pooling_height, uint32_t pooling_width, uint32_t stride_height, uint32_t stride_width, uint32_t dilation_height,
    uint32_t dilation_width, size_t channels, uint8_t output_min, uint8_t output_max, uint32_t flags,
    qnnp_operator_t* max_pooling_out) {
  (void) flags;
  if (!g_lib.initialized) {
    log_error("qnnp_create_max_pooling2d_nhwc_u8 failed because QNNPACK is not properly initialized");
    return qnnp_status_uninitialized;
  }
  const uint32_t pooling_size = pooling_height * pooling_width;
  if (pooling_size == 0 || pooling_size == 1 || stride_height == 0 || stride_width == 0 || dilation_height == 0 ||
      dilation_width == 0 || channels == 0) {  // src/max-pooling.c:64-105
    log_error("failed to create max pooling with %ux%u pooling, %ux%u stride, %ux%u dilation, %zu channels", pooling_width,
              pooling_height, stride_width, stride_height, dilation_width, dilation_height, channels);
    return qnnp_status_invalid_parameter;
  }
  qnnp_operator* op = new_operator(kKindMaxPool);
  if (op == nullptr) return qnnp_status_out_of_memory;
  op->pad_top = input_padding_top, op->pad_right = input_padding_right;
  op->pad_bottom = input_padding_bottom, op->pad_left = input_padding_left;
  op->kh = pooling_height, op->kw = pooling_width, op->stride_h = stride_height, op->stride_w = stride_width;
  op->dil_h = dilation_height, op->dil_w = dilation_width;
  op->channels = channels;
  op->omin = output_min, op->omax = output_max;
  *max_pooling_out = op;
  return qnnp_status_success;
}

namespace {
enum qnnp_status setup_pool2d(qnnp_operator* op, KernelKind kind, size_t batch_size, size_t input_height, size_t input_width,
                              const uint8_t* input, size_t input_stride, uint8_t* output, size_t output_stride) {
  if (!g_lib.initialized) return qnnp_status_uninitialized;
  if (op == nullptr || op->kind != kind) return qnnp_status_invalid_parameter;
  if (batch_size == 0) {
    op->batch = 0;
    if (op->plan != nullptr) op->plan->valid = false;
    return qnnp_status_success;
  }
  if (input_width == 0 || input_height == 0) {
    log_error("failed to setup pooling with %zux%zu input: input dimensions must be non-zero", input_width, input_height);
    return qnnp_status_invalid_parameter;
  }
  op->batch = batch_size, op->in_h = input_height, op->in_w = input_width;
  op->input = input, op->in_stride = input_stride;
  op->out_h = output_dimension(op->pad_top + input_height + op->pad_bottom, op->kh, op->dil_h, op->stride_h);
  op->out_w = output_dimension(op->pad_left + input_width + op->pad_right, op->kw, op->dil_w, op->stride_w);
  op->output = output, op->out_stride = output_stride;
  return finish_setup(op, batch_size * input_height * input_width, op->channels, batch_size * op->out_h * op->out_w, op->channels);
}
}  // namespace

QNNP_EXPORT enum qnnp_status qnnp_setup_average_pooling2d_nhwc_q8(qnnp_operator_t op, size_t batch_size, size_t input_height,
                                                                  size_t input_width, const uint8_t* input, size_t input_stride,
                                                                  uint8_t* output, size_t output_stride, pthreadpool_t threadpool) {
  (void) threadpool;
  return setup_pool2d(op, kKindAvgPool, batch_size, input_height, input_width, input, input_stride, output, output_stride);
}

QNNP_EXPORT enum qnnp_status qnnp_setup_max_pooling2d_nhwc_u8(qnnp_operator_t op, size_t batch_size, size_t input_height,
                                                              size_t input_width, const uint8_t* input, size_t input_stride,
                                                              uint8_t* output, size_t output_stride, pthreadpool_t threadpool) {
  (void) threadpool;
  return setup_pool2d(op, kKindMaxPool, batch_size, input_height, input_width, input, input_stride, output, output_stride);
}

// ---- channel shuffle (src/channel-shuffle.c) --------------------------------------------------------------------------------
QNNP_EXPORT enum qnnp_status qnnp_create_channel_shuffle_nc_x8(size_t groups, size_t group_channels, uint32_t flags,
                                                               qnnp_operator_t* channel_shuffle_out) {
  (void) flags;
  if (!g_lib.initialized) {
    log_error("qnnp_create_channel_shuffle_nc_x8 failed because QNNPACK is not properly initialized");
    return qnnp_status_uninitialized;
  }
  if (groups <= 1 || group_channels == 0) {
    log_error("failed to create channel shuffle operator with %zu groups of %zu channels", groups, group_channels);
    return qnnp_status_invalid_parameter;
  }
  qnnp_operator* op = new_operator(kKindShuffle);
  if (op == nullptr) return qnnp_status_out_of_memory;
  op->groups = (uint32_t) groups, op->gic = group_channels;
  op->channels = groups * group_channels;
  *channel_shuffle_out = op;
  return qnnp_status_success;
}

QNNP_EXPORT enum qnnp_status qnnp_setup_channel_shuffle_nc_x8(qnnp_operator_t op, size_t batch_size, const uint8_t* input,
                                                              size_t input_stride, uint8_t* output, size_t output_stride) {
  if (op == nullptr || op->kind != kKindShuffle) return g_lib.initialized ? qnnp_status_invalid_parameter : qnnp_status_uninitialized;
  return setup_nc(op, batch_size, input, input_stride, output, output_stride);
}

// ---- clamp (src/clamp.c) --------------------------------------------------------------------------------------------------
QNNP_EXPORT enum qnnp_status qnnp_create_clamp_nc_u8(size_t channels, uint8_t output_min, uint8_t output_max, uint32_t flags,
                                                     qnnp_operator_t* clamp_out) {
  (void) flags;
  if (!g_lib.initialized) {
    log_error("qnnp_create_clamp_nc_u8 failed because QNNPACK is not properly initialized");
    return qnnp_status_uninitialized;
  }
  if (channels == 0 || output_min > output_max) {
    log_error("failed to create Clamp operator with %zu channels and [%u, %u] output range", channels, output_min, output_max);
    return qnnp_status_invalid_parameter;
  }
  qnnp_operator* op = new_operator(kKindClamp);
  if (op == nullptr) return qnnp_status_out_of_memory;
  op->channels = channels, op->omin = output_min, op->omax = output_max;
  *clamp_out = op;
  return qnnp_status_success;
}

QNNP_EXPORT enum qnnp_status qnnp_setup_clamp_nc_u8(qnnp_operator_t op, size_t batch_size, const uint8_t* input,
                                                    size_t input_stride, uint8_t* output, size_t output_stride) {
  if (op == nullptr || op->kind != kKindClamp) return g_lib.initialized ? qnnp_status_invalid_parameter : qnnp_status_uninitialized;
  return setup_nc(op, batch_size, input, input_stride, output, output_stride);
}

// ---- sigmoid / leaky ReLU: 256-entry tables built exactly as the reference builds them (src/sigmoid.c:96-112,
//      src/leaky-relu.c:110-125), applied by the lookup kernel (src/x8lut/scalar.c) ---------------------------------------
QNNP_EXPORT enum qnnp_status qnnp_create_sigmoid_nc_q8(size_t channels, uint8_t input_zero_point, float input_scale,
                                                       uint8_t output_zero_point, float output_scale, uint8_t output_min,
                                                       uint8_t output_max, uint32_t flags, qnnp_operator_t* sigmoid_out) {
  (void) flags;
  if (!g_lib.initialized) {
    log_error("qnnp_create_sigmoid_nc_q8 failed because QNNPACK is not properly initialized");
    return qnnp_status_uninitialized;
  }
  if (channels == 0 || !scale_ok(input_scale) || !scale_ok(output_scale) || output_min >= output_max) {
    log_error("failed to create Sigmoid operator: channels must be non-zero, scales finite and positive, min below max");
    return qnnp_status_invalid_parameter;
  }
  if (output_scale != 0x1.0p-8f || output_zero_point != 0) {
    log_error("failed to create Sigmoid operator: only output scale 1/256 and output zero point 0 are supported");
    return qnnp_status_unsupported_parameter;
  }
  uint8_t table[256];
  const float scaled_min = (float) (int32_t) output_min, scaled_max = (float) (int32_t) output_max;
  for (int32_t i = 0; i < 256; i++) {
    const float x = input_scale * (float) (i - (int32_t) (uint32_t) input_zero_point);
    float scaled_sigmoid_x = 256.0f / (1.0f + expf(-x));
    if (scaled_sigmoid_x < scaled_min) scaled_sigmoid_x = scaled_min;
    if (scaled_sigmoid_x > scaled_max) scaled_sigmoid_x = scaled_max;
    table[(uint32_t) i] = (uint8_t) lrintf(scaled_sigmoid_x);
  }
  bind_device();
  qnnp_operator* op = new_operator(kKindLut);
  if (op == nullptr) return qnnp_status_out_of_memory;
  op->channels = channels;
  const enum qnnp_status st = upload((void**) &op->d_lut, table, sizeof table);
  if (st != qnnp_status_success) {
    free_operator(op);
    return st;
  }
  *sigmoid_out = op;
  return qnnp_status_success;
}

QNNP_EXPORT enum qnnp_status qnnp_setup_sigmoid_nc_q8(qnnp_operator_t op, size_t batch_size, const uint8_t* input,
                                                      size_t input_stride, uint8_t* output, size_t output_stride) {
  if (op == nullptr || op->kind != kKindLut) return g_lib.initialized ? qnnp_status_invalid_parameter : qnnp_status_uninitialized;
  return setup_nc(op, batch_size, input, input_stride, output, output_stride);
}

QNNP_EXPORT enum qnnp_status qnnp_create_leaky_relu_nc_q8(size_t channels, float negative_slope, uint8_t input_zero_point,
                                                          float input_scale, uint8_t output_zero_point, float output_scale,
                                                          uint8_t output_min, uint8_t output_max, uint32_t flags,
                                                          qnnp_operator_t* leaky_relu_out) {
  (void) flags;
  if (!g_lib.initialized) {
    log_error("qnnp_create_leaky_relu_nc_q8 failed because QNNPACK is not properly initialized");
    return qnnp_status_uninitialized;
  }
  // src/leaky-relu.c:38-76
  if (channels == 0 || negative_slope <= 0.0f || !isnormal(negative_slope) || negative_slope > 1.0f || !scale_ok(input_scale) ||
      !scale_ok(output_scale) || output_min >= output_max) {
    log_error("failed to create Leaky ReLU operator: invalid channels, slope, scales or output range");
    return qnnp_status_invalid_parameter;
  }
  const float input_output_scale = input_scale / output_scale;
  if (input_output_scale < 0x1.0p-8f || input_output_scale >= 0x1.0p+8f) {
    log_error("failed to create Leaky ReLU operator with %.7g input-to-output scale ratio: must be in [2**-8, 2**8)",
              input_output_scale);
    return qnnp_status_unsupported_parameter;
  }
  uint8_t table[256];
  const float scaled_min_less_zero_point = (float) ((int32_t) output_min - (int32_t) output_zero_point);
  const float scaled_max_less_zero_point = (float) ((int32_t) output_max - (int32_t) output_zero_point);
  for (int32_t i = 0; i < 256; i++) {
    const float x = input_output_scale * (float) (i - (int32_t) (uint32_t) input_zero_point);
    float y = x < 0.0f ? x * negative_slope : x;
    if (y < scaled_min_less_zero_point) y = scaled_min_less_zero_point;
    if (y > scaled_max_less_zero_point) y = scaled_max_less_zero_point;
    table[(uint32_t) i] = (uint8_t) (lrintf(y) + (long) output_zero_point);
  }
  bind_device();
  qnnp_operator* op = new_operator(kKindLut);
  if (op == nullptr) return qnnp_status_out_of_memory;
  op->channels = channels;
  const enum qnnp_status st = upload((void**) &op->d_lut, table, sizeof table);
  if (st != qnnp_status_success) {
    free_operator(op);
    return st;
  }
  *leaky_relu_out = op;
  return qnnp_status_success;
}

QNNP_EXPORT enum qnnp_status qnnp_setup_leaky_relu_nc_q8(qnnp_operator_t op, size_t batch_size, const uint8_t* input,
                                                         size_t input_stride, uint8_t* output, size_t output_stride) {
  if (op == nullptr || op->kind != kKindLut) return g_lib.initialized ? qnnp_status_invalid_parameter : qnnp_status_uninitialized;
  return setup_nc(op, batch_size, input, input_stride, output, output_stride);
}

// ---- softargmax (src/softargmax.c; run: src/operator-run.c:625-637) -------------------------------------------------------
QNNP_EXPORT enum qnnp_status qnnp_create_softargmax_nc_q8(size_t channels, float input_scale, uint8_t output_zero_point,
                                                          float output_scale, uint32_t flags, qnnp_operator_t* softargmax_out) {
  (void) flags;
  if (!g_lib.initialized) {
    log_error("qnnp_create_softargmax_nc_q8 failed because QNNPACK is not properly initialized");
    return qnnp_status_uninitialized;
  }
  if (channels == 0 || !scale_ok(input_scale) || !scale_ok(output_scale)) {
    log_error("failed to create Soft ArgMax operator: channels must be non-zero, scales finite and positive");
    return qnnp_status_invalid_parameter;
  }
  if (output_scale != 0x1.0p-8f || output_zero_point != 0) {
    log_error("failed to create Soft ArgMax operator: only output scale 1/256 and output zero point 0 are supported");
    return qnnp_status_unsupported_parameter;
  }
  // 256 entries as the reference builds them (src/softargmax.c:79-83); a row uses table + (255 - max), i.e. indices up to
  // 510 — entries beyond 255 are never reached because x <= max, they are zero here for definiteness
  uint32_t table[511] = {0};
  const double qscale = fmin(((double) UINT32_MAX) / (double) channels, 8388607.0);
  for (int32_t i = 0; i < 256; i++) {
    const double scaled_exp_xi = qscale * exp((double) (i - 255) * (double) input_scale);
    table[(uint32_t) i] = (uint32_t) lrint(scaled_exp_xi);
  }
  bind_device();
  qnnp_operator* op = new_operator(kKindSoftargmax);
  if (op == nullptr) return qnnp_status_out_of_memory;
  op->channels = channels;
  const enum qnnp_status st = upload((void**) &op->d_table32, table, sizeof table);
  if (st != qnnp_status_success) {
    free_operator(op);
    return st;
  }
  *softargmax_out = op;
  return qnnp_status_success;
}

QNNP_EXPORT enum qnnp_status qnnp_setup_softargmax_nc_q8(qnnp_operator_t op, size_t batch_size, const uint8_t* input,
                                                         size_t input_stride, uint8_t* output, size_t output_stride) {
  if (op == nullptr || op->kind != kKindSoftargmax)
    return g_lib.initialized ? qnnp_status_invalid_parameter : qnnp_status_uninitialized;
  return setup_nc(op, batch_size, input, input_stride, output, output_stride);
}
