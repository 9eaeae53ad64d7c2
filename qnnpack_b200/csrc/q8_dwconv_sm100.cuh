// Parameters of the CUDA-core kernels: 3x3 depthwise, generic direct convolution, stand-alone requantizer.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "requant_math.h"

namespace q8 {

struct DwParams {
  const uint8_t* in;
  uint8_t* out;
  const int32_t* w32;   // [9][c_pad]  (w - kzp), tap index = ky*3 + kx
  const int32_t* bias;  // [c_pad] folded bias (reference pack.h:146-159)
  long long in_stride, out_stride;
  long long total_threads;
  int batch, channels, c_pad;
  int in_h, in_w, out_h, out_w;
  int stride_h, stride_w, dil_h, dil_w, pad_top, pad_left;
  int cgroups, xstrips;
  int izp;
  int rq_mode;
  Q8Requant rq;
};

// streaming dp4a kernel (q8_dwconv_stream_sm100.cu)
struct DwStreamParams {
  const uint8_t* in;
  uint8_t* out;
  const uint32_t* wa;   // [3][c_pad]: per channel and kernel row the three taps packed as bytes (operand A)
  const uint32_t* wb;   // [3][c_pad]: operand B when (w - kzp) does not fit 8 bits (wmode 2)
  const int32_t* bias;  // [c_pad] folded bias
  long long in_stride, out_stride;
  long long total_threads;
  int batch, channels, c_pad;
  int in_h, in_w, out_h, out_w;
  int stride, pad_top, pad_left;
  int cgroups, xstrips, ychunks, tyc;
  int wmode;            // 0: one s8 operand, 1: one u8 operand (kzp == 0), 2: two s8 operands (w - kzp = A + B), 3: one s8 operand holding kzp - w
  int izp;
  int rq_mode;
  int shift_mul;        // see requant_dev.cuh
  Q8Requant rq;
};

// tcgen05 depthwise kernel (q8_dwconv_umma_sm100.cu): 3x3 depthwise as block-diagonal UMMAs over TMA-staged tiles
constexpr int kDwTcTaps = 5;
constexpr int kDwTcTaps32 = 9;      // pair mode: one UMMA (K = 32 channels) per tap        // UMMAs (K = 32 = two taps) per (sub-tile, channel group): 9 taps + 1 empty slot
constexpr int kDwTcMaxStages = 8;
constexpr int kDwTcMaxG = 8;        // channel groups (16 channels each) per work item

struct DwTcParams {
  uint8_t* out;
  const uint8_t* wpack;     // [channel group][kDwTcTaps][2 K-chunks][nb_cols rows][16 B]  block-diagonal B operands
  const int32_t* bias_cls;  // [64 border classes][channels]: bias - izp * sum over the VALID taps of (w - kzp)
  long long out_stride;
  long long total_items;
  int batch, channels, cgs, cblocks;     // cgs = channels / 16; cblocks = ceil(cgs / G)
  int in_h, in_w, out_h, out_w, stride, pad_top, pad_left;
  // work item = nb images x 16 row groups x (8 * mt) output columns x G channel groups
  int G, mt, xt, yt, nt;    // x tiles per row, y tiles per image, image blocks
  int nb, Q;                // images per item; row groups per image inside an item (16 when nb == 1)
  int whole;                // 1: the item covers whole images (box rows = stride * Q per image, origin row -pad_top)
  // smem stage: per channel group [planes][nb][box_rows][box_px][16 B] then the group's B block
  int planes, box_rows, box_px, plane_tx, plane_bytes, a_bytes, b_bytes, cg_bytes, stage_bytes, num_stages, smem_total;
                            // plane_tx = bytes one TMA box delivers; plane_bytes = its 128-byte-rounded smem slot
  int x_org[2];             // plane x origin relative to the item's first output column (in plane pixels)
  int a_off[kDwTcTaps], a_lbo[kDwTcTaps];  // byte offset of the first tap of UMMA u inside a group's A block; second-tap offset
  int sbo;                  // bytes between the rows of consecutive row groups (stride * box_px * 16)
  int nb_cols;              // accumulator columns per unit: 16, or 32 when w - kzp is split into two s8 operands
  int b_signed;             // B operand format: 1 = s8, 0 = u8 (kzp == 0)
  int acc_stride, acc_stages;
  int pair;                 // 1: channel PAIR mode — TMA boxes, smem pixels and UMMAs are 32 channels wide (32-byte sector granularity
                            // on the L2, SWIZZLE_32B tiles, one K = 32 UMMA per tap with a 32x32 diagonal B, N = 32); cg_bytes,
                            // plane_* and sbo then describe 32-byte pixels and one block per channel pair
  int a_off9[9];            // pair mode: byte offset of tap (ky, kx) = index ky*3+kx inside a pair's A block
  int b_resident;           // 1: ALL weight blocks of the layer sit in shared memory for the whole launch (at b_res_off from the
  int b_res_off;            // ring's base) instead of travelling with every item's stage; cg_bytes then has no B part
  int store32;              // 1: the epilogue pairs channel groups and writes 32 bytes per pixel with one 256-bit store
                            // (needs 32-byte aligned output pixels and an even number of channel groups per item)
  int acc_sign;             // +1, or -1 when the B operand holds kzp - w (the accumulators are the negated sums)
  // Border-class biases.  The epilogue reads row ((row slot * bias_rstride) + column slot) of a [slots][channels] table; a
  // class's row / column slot is nibble (row / column class bits) of bias_rslot / bias_cslot.  Global table (bias_smem = 0):
  // slot = class bits, bias_rstride = 8, i.e. bias_cls itself.  bias_smem = 1: only the bias_nrc x bias_ncc classes the
  // geometry produces, copied from bias_cls into shared memory at bias_off (from the aligned base) when the CTA starts; slot k's
  // class bits are nibble k of bias_rcls / bias_ccls, and classes the geometry never produces (rows and columns whose outputs
  // are not stored) read slot 0.
  int bias_smem, bias_off, bias_rstride, bias_nrc, bias_ncc;
  uint32_t bias_rslot, bias_cslot, bias_rcls, bias_ccls;
  // item schedule: a CTA's next item is the NEXT item; in (cb, xtile, ytile, nblk) digits that is this step
  int chunk;                // items per CTA: CTA b runs items [b * chunk, min(total, (b + 1) * chunk))
  int step_cb, step_x, step_y, step_n;
  uint32_t inv_g, inv_tail; // ceil(2^16 / m) for m = mt and for the sub-tile count of the last x tile
  int rq_mode;
  Q8Requant rq;
};

struct DirectParams {
  const uint8_t* in;
  uint8_t* out;
  const uint8_t* w;     // original layout [G][GOC][KH][KW][GIC]
  const int32_t* bias;  // [G*GOC] folded bias
  long long in_stride, out_stride;
  long long total;      // batch*out_h*out_w*groups*goc
  int groups, gic, goc;
  int in_h, in_w, out_h, out_w, kh, kw;
  int stride_h, stride_w, dil_h, dil_w, pad_top, pad_left;
  int izp, kzp;
  int deconv;           // 1: transposed convolution — tap (ky, kx) of output (oy, ox) reads input ((oy + pad_top - ky*dil) / stride, ..)
                        // when the division is exact and in range (src/indirection.c:134-190), else it contributes nothing
  Q8Requant rq;
};

cudaError_t launch_q8_dwconv3x3(DwParams p, int cv, cudaStream_t stream);
cudaError_t launch_q8_dwconv3x3_stream(DwStreamParams p, cudaStream_t stream);
cudaError_t launch_q8_dwconv3x3_umma(const DwTcParams& p, const void* tensor_map, int grid, int max_smem_optin,
                                     cudaStream_t stream);
cudaError_t launch_q8_direct_conv(const DirectParams& p, cudaStream_t stream);
cudaError_t launch_q8_requantize(const int32_t* in, uint8_t* out, long long n, const Q8Requant& rq, cudaStream_t stream);

}  // namespace q8
