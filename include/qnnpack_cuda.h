/*
 * qnnpack_cuda.h — additive, non-breaking extensions of the qnnpack.h C ABI for CUDA callers.
 * Nothing here exists in the reference; a caller that only knows qnnpack.h never needs it.
 * Plain C types only (streams are passed as void* == cudaStream_t) so that cgo / JNI / ctypes
 * bindings do not need the CUDA headers.
 */
#pragma once

#include "qnnpack.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Stream every later qnnp_run_operator / qnnp_cuda_run_operator_async enqueues on.
 * NULL restores the library's own non-blocking stream.  Not thread-safe against concurrent runs. */
enum qnnp_status qnnp_cuda_set_stream(void* cuda_stream);
void* qnnp_cuda_get_stream(void);

/* Device ordinal selected by qnnp_initialize(), or -1 before initialisation. */
int qnnp_cuda_get_device(void);

/* Like qnnp_run_operator (reference include/qnnpack.h:327-329, src/operator-run.c:639) but only enqueues:
 * valid only for operators whose input and output given to qnnp_setup_* are DEVICE pointers
 * (host pointers need the synchronous call, which stages the copies); returns
 * qnnp_status_invalid_parameter otherwise.  Completion is observed through the stream. */
enum qnnp_status qnnp_cuda_run_operator_async(qnnp_operator_t op);

/* Packed-weight blob of a convolution / fully-connected operator, resident on the device.
 * Multi-GPU data parallelism replicates weights by broadcasting this blob (e.g. ncclBroadcast /
 * torch.distributed.broadcast over NVLink) into the identically-created operator on every rank;
 * the steady-state run has no collective.  Returns qnnp_status_invalid_parameter for NULL. */
enum qnnp_status qnnp_cuda_operator_packed_weights(qnnp_operator_t op, void** device_ptr, size_t* size_bytes);
/* The folded int32 bias (b + K*izp*kzp - izp*sum w, reference src/qnnpack/pack.h:24-43) that goes with it. */
enum qnnp_status qnnp_cuda_operator_packed_bias(qnnp_operator_t op, void** device_ptr, size_t* size_bytes);

/* Number of kernels the library has launched since qnnp_initialize() (bench.py's gpu_launches). */
unsigned long long qnnp_cuda_launch_count(void);

/* Stand-alone Q31 requantization int32 -> uint8 on the device (the epilogue as its own kernel);
 * the counterpart of the reference's qnnp_requantize_q31__scalar
 * (src/qnnpack/requantization-stubs.h:22-29, src/requantization/q31-scalar.c:17).
 * `input`/`output` may be host or device pointers; synchronous. scale must be in [2^-32, 1). */
enum qnnp_status qnnp_cuda_requantize_q31(
    size_t n, const int32_t* input, float scale, uint8_t zero_point, uint8_t qmin, uint8_t qmax, uint8_t* output);

/* Debug aid for kernel bring-up: when non-NULL, the next runs of tensor-core operators also dump
 * their raw int32 accumulators ([work item][128][n_mma]) to this DEVICE buffer. */
void qnnp_cuda_debug_set_accumulator_dump(int32_t* device_buffer);

/* The tiling / shared-memory plan the tensor-core kernel would use for a K x N (x groups) operator; needs no GPU.
 * folded != 0: plan for the mode in which bias and zero-point correction run as extra UMMAs (bias_steps of them).
 * out = {K, nkc, skc, k_stages, mt, n_tiles, n_tile, n_mma, has_corr, b_resident, num_stages, stage_bytes,
 *        staging_bytes, bias_bytes, smem_b_off, smem_bias_off, smem_a_off, smem_stage_off, smem_total, bulk_capable,
 *        folded, bias_steps, blk_chunks, good}.  Returns 1 on success, 0 if no plan fits. */
int qnnp_cuda_debug_plan_igemm(size_t k, size_t n, uint32_t groups, int folded, int bias_steps, int out[24]);
int qnnp_cuda_debug_operator_is_folded(qnnp_operator_t op);

/* Packed operands of the tensor-core kernel for a K x N fully-connected / 1x1 operator, built on the host; needs no GPU
 * (tests/test_igemm_pack.py replays the UMMA algebra on these bytes).  kernel = [n][k] uint8, bias = [n] int32.
 * meta = {folded, nkc, n_tiles, n_tile, n_mma, blk_chunks, bias_steps, b_signed, has_b2, k_tail_pad, has_corr, 0, ...};
 * blob = per n-tile [blk_chunks][n_mma][16 B]; *blob_bytes / *bias_count: capacity in, size out.  Returns 1 / 0. */
int qnnp_cuda_debug_pack_igemm(size_t k, size_t n, uint8_t input_zero_point, uint8_t kernel_zero_point, const uint8_t* kernel,
                               const int32_t* bias, int meta[16], uint8_t* blob, size_t* blob_bytes, int32_t* folded_bias,
                               size_t* bias_count);

/* Tiling of the depthwise tensor-core kernel (q8_dwconv_umma_sm100.cu) for a geometry; needs no GPU.  wmode: 0 = every
 * w - kzp fits s8, 1 = kzp == 0 (u8 weights), 2 = w - kzp split into two s8 operands, 3 = every kzp - w fits s8 (negated operand).
 * out = {G, mt, xt, yt, nt, nb, Q, whole, planes, box_rows, box_px, plane_tx, plane_bytes, a_bytes, b_bytes, cg_bytes,
 *        stage_bytes, num_stages, smem_total, x_org[2], a_off[5], a_lbo[5], sbo, nb_cols, b_signed, acc_stride, cblocks, cgs,
 *        total_items, 0, 0}.  Returns 1, or 0 when the shape is not eligible (the CUDA-core depthwise kernels run instead). */
int qnnp_cuda_debug_plan_dwconv(int channels, int batch, int in_h, int in_w, int out_h, int out_w, int stride, int pad_top,
                                int pad_left, int wmode, int out[40]);
/* Operands of the depthwise tensor-core kernel for `channels` (% 16 == 0) channels, built on the host; needs no GPU.
 * kernel = [channels][9] uint8, bias = [channels] int32.  wpack receives (channels/16) * 5 * 2 * nb_cols * 16 bytes
 * (nb_cols = 32 when the returned mode is 2, else 16), bias_cls 64 * channels int32 (XOR 2^31 when u_form != 0).
 * Returns the weight-operand mode (0: one s8 operand, 1: u8, 2: two s8 operands) or -1. */
int qnnp_cuda_debug_pack_dwconv(size_t channels, uint8_t input_zero_point, uint8_t kernel_zero_point, const uint8_t* kernel,
                                const int32_t* bias, int u_form, uint8_t* wpack, int32_t* bias_cls);
/* The same for the kernel's channel-PAIR form (32 channels per TMA box / UMMA, SWIZZLE_32B tiles; single weight operand only).
 * plan: out[0..37] as above (a_off / a_lbo zero), out[38] = 1, out[39..47] = byte offset of tap ky*3+kx inside a pair's A block.
 * pack: wpack receives ceil(channels / 32) * 9 * 1024 bytes: per pair and tap a K-major block [2 K-chunks][32 rows][16 B] =
 * diag(w - kzp), or kzp - w when the returned mode is 3, or raw w when it is 1; returns -1 when the weights need two operands.
 * wmode of both calls: 0, 1 as above, 3 = one s8 operand holding kzp - w (accumulators negated). */
int qnnp_cuda_debug_plan_dwconv32(int channels, int batch, int in_h, int in_w, int out_h, int out_w, int stride, int pad_top,
                                  int pad_left, int wmode, int out[48]);
int qnnp_cuda_debug_pack_dwconv32(size_t channels, uint8_t kernel_zero_point, const uint8_t* kernel, uint8_t* wpack);
/* Border-class bias table of either form's plan (pair = 0 / 1): out = {bias_smem, bias_off, bias_rstride, bias_nrc, bias_ncc,
 * bias_rslot, bias_cslot, bias_rcls, bias_ccls, smem_total, num_stages, stage_bytes} (see DwTcParams in
 * qnnpack_b200/csrc/q8_dwconv_sm100.cuh).  Returns 0 when the shape is not eligible. */
int qnnp_cuda_debug_plan_dwconv_bias(int channels, int batch, int in_h, int in_w, int out_h, int out_w, int stride, int pad_top,
                                     int pad_left, int wmode, int pair, int out[12]);
/* Launches of the depthwise tensor-core kernel since qnnp_initialize() (tests use it to prove the routing). */
unsigned long long qnnp_cuda_debug_dw_umma_launch_count(void);

/* Panel-epilogue tables of the tensor-core kernel for an n-tile (CPU-callable; tests/test_planner.py replays them). */
void qnnp_cuda_debug_panel_tables(int n_tile, int mt, int folded, int out[50]);

/* Measured dense int8 tensor-core peak of this device in tera-ops/s: a shared-memory-resident tcgen05.mma kind::i8 loop
 * (148 CTAs x `iters` x 8 UMMAs of 128x256x32), `reps` launches timed with CUDA events on the library's stream.  The
 * denominator of "%-of-peak on q8gemm" (BASELINE.json metric; reference counter bench/q8gemm.cc:108). */
enum qnnp_status qnnp_cuda_measure_int8_peak(int iters, int reps, double* tops, double* ms_per_launch);

/* Name of the kernel family an operator was routed to: "igemm-gemm", "igemm-conv", "dwconv3x3", "direct". */
const char* qnnp_cuda_operator_kernel_name(qnnp_operator_t op);

#ifdef __cplusplus
}
#endif
