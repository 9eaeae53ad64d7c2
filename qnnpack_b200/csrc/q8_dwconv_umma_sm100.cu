// q8dwconv 3x3 for sm_100a on the tensor cores: depthwise convolution as block-diagonal UMMAs over TMA-staged tiles.
//
// Replaces (reference, paths relative to its root):
//   src/operator-run.c:647-710  dwconv case -> q8dwconv_ukernel_up8x9__sse2 (src/q8dwconv/up8x9-sse2.c:14-372)
//   src/indirection.c:81-132    (no pointer table: a tap is an address offset inside the staged tile)
// for 3x3, dilation 1, stride 1 or 2, channels % 16 == 0; other depthwise shapes keep the CUDA-core kernels
// (q8_dwconv_stream_sm100.cu, q8_dwconv_sm100.cu).
//
// Why tensor cores for a depthwise layer: on the CUDA cores the layer costs ~23 instructions per output byte
// (window transposes + dp4a + requantisation) and runs at ~1/4 of the HBM roofline.  A UMMA with a DIAGONAL
// 16x16 weight block per tap wastes 15/16 of its MACs, but B200 has ~60x more int8 MACs per byte of HBM traffic
// than this layer needs, so the waste is free; what remains per output is the requantisation epilogue only.
//
// Data flow of one work item (nb images x 16 row groups x 8*mt output columns x G groups of 16 channels):
//   TMA     : for each channel group ONE tensor-map box {16 B channels, box_px pixels, box_rows rows, nb images}
//             (two boxes, even / odd input columns, when stride == 2: the input is viewed as [N][H][W/2][2][C]).
//             In smem a pixel is 16 contiguous bytes, so 8 consecutive pixels ARE a K-major no-swizzle core matrix
//             and a row group (8 output columns of one output row) is one 8-row slice of the UMMA's M = 128.
//             Out-of-image pixels are zero-filled by the TMA unit (see bias_cls below).
//   UMMA    : M = 128 (16 row groups: descriptor SBO = stride * row pitch), K = 32 = TWO taps (descriptor LBO = byte
//             distance between the two taps' pixels), N = 16 channels.  B is diag(w_tap[c] - kzp) per tap, packed on
//             the host.  9 taps -> 5 UMMAs per (sub-tile, channel group).  When w - kzp needs 9 bits it is split
//             into two s8 operands that sit side by side in N (N = 32, the epilogue adds the halves).
//   epilogue: TMEM -> registers, + bias_cls, Q31 requantisation, 16-byte global store per pixel.
//   bias_cls: the reference pads with the input zero point, TMA pads with 0.  Both agree once the bias carries
//             -izp * (sum of w - kzp over the taps that are INSIDE the image): 64 border classes (3 row bits x 3
//             column bits) x channels, built on the host; interior pixels all use class 63.  The (at most 9, for padding
//             <= 1 on images >= 3 pixels) classes a geometry produces are copied into shared memory when they fit beside
//             the ring (DwTcParams::bias_smem): one LDS instead of one LDG per bias word.
//
// Same integers as the reference:  acc[c] = bias[c] + sum_valid_taps (a_tap[c] - izp) * (w_tap[c] - kzp).
#include <cuda.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>
#include <string.h>

#include "q8_dwconv_sm100.cuh"
#include "requant_dev.cuh"
#include "sm100_ptx.cuh"

namespace q8 {
namespace {

constexpr int kEpiWarps = 16;
constexpr int kMmaWarp = kEpiWarps;            // first of the UMMA-issuing warps (it also owns the TMEM allocation)
constexpr int kMmaWarps = 7;                   // one lane each; they split the units of an item (see below)
constexpr int kTmaWarp = kMmaWarp + kMmaWarps;
constexpr int kThreads = (kTmaWarp + 1) * 32;  // 768 (24 warps: keeps the 80-register budget)
constexpr int kMaxUnitsPerMmaWarp = 3;         // 16 units (mt * G <= 16) over 7 warps
constexpr int kTmemCols = 512;

struct __align__(8) Ctl {
  uint64_t full[kDwTcMaxStages];
  uint64_t empty[kDwTcMaxStages];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint64_t b_full;  // resident weight blocks have landed (DwTcParams::b_resident)
  uint32_t tmem_base;
};

// What every role needs to know about a work item, computed ONCE by the TMA producer thread (which decodes the item
// anyway) and handed to the 7 UMMA-issuing and 16 epilogue warps through a small shared-memory ring.  Round 2: before,
// each of those 23 warps re-derived it per item (mixed-radix stepping, tail clamps, a 64-bit output origin: ~80-140
// instructions per warp and item — a quarter of everything the kernel executed, profiles/r2c_dw_umma_first2).
// Slot of the k-th item of a CTA: k mod kDescSlots.  A slot is rewritten num_stages + 2 items later at the earliest: the
// producer runs at most num_stages items ahead of the UMMAs, which run at most 2 (accumulator stages) ahead of the
// epilogue's last tensor-memory read of an item — and every reader has copied the slot to registers before that.
// Visibility: the producer writes the slot before its arrive.expect_tx on the stage's `full` barrier (release); the UMMA
// warps read it after their wait on `full` (acquire), the epilogue warps after their wait on `tmem_full`, which the UMMA
// warps signal after that.
struct __align__(16) ItemDesc {
  uint64_t tile_base;  // output address of (image n0, row oy0, column ox0, channel 0)
  int32_t n0, oy0;
  int32_t ox0, c0;
  int32_t mt_eff, g_eff;
  uint32_t inv;        // ceil(2^16 / mt_eff): unit index -> (sub-tile, channel group)
  int32_t units;
  int32_t pad[2];
};
constexpr int kDescSlots = kDwTcMaxStages + 2;

__device__ __forceinline__ ItemDesc load_desc(const ItemDesc* d) {
  ItemDesc r;
  const uint4* s4 = reinterpret_cast<const uint4*>(d);
  uint4* r4 = reinterpret_cast<uint4*>(&r);
  r4[0] = s4[0], r4[1] = s4[1], r4[2] = s4[2];
  return r;
}

__device__ __forceinline__ uint64_t pack_u64(uint32_t lo, uint32_t hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(lo), "r"(hi));
  return r;
}

struct DwItem {
  int cb;       // channel block (G groups of 16 channels)
  int n0;       // first image
  int oy0;      // first output row (0 in whole-image mode)
  int ox0;      // first output column
  int mt_eff;   // sub-tiles (8 columns) that contain at least one valid column
  int g_eff;    // channel groups present in this block
};

// item = ((nblk * yt + ytile) * xt + xtile) * cblocks + cb: the channel blocks of one spatial tile are neighbours in
// the schedule, so the CTAs that run them touch the same DRAM lines at about the same time.
// Every role walks the same item sequence; the position is kept as mixed-radix digits and advanced by the (host-
// computed) digits of the grid size, so the three divisions happen once per CTA instead of once per item and role.
struct ItemPos {
  int cb, xt, yt, nb;
};

__device__ __forceinline__ ItemPos first_pos(const DwTcParams& p, uint32_t item) {
  ItemPos q;
  uint32_t r = item / (uint32_t) p.cblocks;
  q.cb = (int) (item - r * (uint32_t) p.cblocks);
  uint32_t s = r / (uint32_t) p.xt;
  q.xt = (int) (r - s * (uint32_t) p.xt);
  r = s / (uint32_t) p.yt;
  q.yt = (int) (s - r * (uint32_t) p.yt);
  q.nb = (int) r;
  return q;
}

__device__ __forceinline__ void advance_pos(const DwTcParams& p, ItemPos& q) {
  q.cb += p.step_cb;
  int carry = q.cb >= p.cblocks;
  q.cb -= carry ? p.cblocks : 0;
  q.xt += p.step_x + carry;
  carry = q.xt >= p.xt;
  q.xt -= carry ? p.xt : 0;
  q.yt += p.step_y + carry;
  carry = q.yt >= p.yt;
  q.yt -= carry ? p.yt : 0;
  q.nb += p.step_n + carry;
}

__device__ __forceinline__ DwItem make_item(const DwTcParams& p, const ItemPos& q) {
  DwItem it;
  it.cb = q.cb;
  it.n0 = q.nb * p.nb;
  it.oy0 = q.yt * 16;
  it.ox0 = q.xt * p.mt * 8;
  const int left = (p.out_w - it.ox0 + 7) >> 3;
  it.mt_eff = left < p.mt ? left : p.mt;
  const int gl = p.cgs - it.cb * p.G;
  it.g_eff = gl < p.G ? gl : p.G;
  return it;
}

// unit index -> (sub-tile j, channel group gi) with j fastest; inv = ceil(2^16 / mt_eff) (exact for un < 256).
// A warp takes the units h, h+4, ...: with 4, 2 or 1 sub-tiles per item those all lie in ONE sub-tile, so the
// per-sub-tile work of the epilogue (pixel, border class, addresses) is done once per item.
__device__ __forceinline__ void unit_split(int un, int mt_eff, uint32_t inv, int& j, int& gi) {
  gi = (int) (((uint32_t) un * inv) >> 16);
  j = un - gi * mt_eff;
}

__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(
          dst),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, int c4,
                                            uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], "
      "[%7];" ::"r"(dst),
      "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(bar)
      : "memory");
}

__device__ __forceinline__ int4 lds128(uint32_t addr) {
  int4 r;
  asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
  return r;
}

__device__ __forceinline__ uint32_t nibble(uint32_t packed, uint32_t k) { return (packed >> (4u * k)) & 15u; }

// One unit = 16 channels of one 8-column sub-tile for the warp's 32 TMEM lanes (4 row groups x 8 columns).
// The bias words (element `bias_idx` of the border-class table: in shared memory when SMB = p.bias_smem, else bias_cls) are
// fetched BEFORE the TMEM load is waited for (the wait is a compiler barrier for memory operations).
template <int RQ, int NB, bool SMB>
__device__ __forceinline__ uint4 epilogue_unit(const DwTcParams& p, uint32_t taddr, uint32_t bias_idx, uint32_t bias_smem_base,
                                               bool last, uint32_t tmem_empty_bar) {
  // order: start the (asynchronous) TMEM load, fetch the bias words while it is in flight, then wait — the wait is a
  // compiler barrier for memory operations, so the bias loads must be issued before it
  int32_t v[16];
  int32_t w[NB == 32 ? 32 : 1];
  if constexpr (NB == 32) {
    tmem_ld32(taddr, w);
  } else {
    tmem_ld16(taddr, v);
  }
  int4 b[4];
#pragma unroll
  for (int t = 0; t < 4; t++)
    b[t] = SMB ? lds128(bias_smem_base + bias_idx * 4u + 16u * (uint32_t) t)
                       : __ldg(reinterpret_cast<const int4*>(p.bias_cls + bias_idx) + t);
  tmem_ld_wait();
  if constexpr (NB == 32) {
#pragma unroll
    for (int i = 0; i < 16; i++) v[i] = w[i] + w[16 + i];  // (w - kzp) = A + B: the two operand halves
  }
  if (last) {  // this warp has read everything it needs from the accumulator stage
    tc_fence_before_sync();
    mbar_arrive(tmem_empty_bar);
  }
  uint32_t o[4];
#pragma unroll
  for (int t = 0; t < 4; t++) {
    const int32_t bb[4] = {b[t].x, b[t].y, b[t].z, b[t].w};
    int32_t n[4];
#pragma unroll
    for (int i = 0; i < 4; i++) {  // (for RQ 5/6 the table already carries the 2^31 offset of "U")
      if constexpr (NB == 32) {
        n[i] = v[4 * t + i] + bb[i];
      } else {
        // one multiply-add: the sign of a negated weight operand (acc_sign = -1, see dw_tc_wmode) is free, and the add
        // sits on the FMA pipe instead of the ALU pipe, which is the busier one in this epilogue
        n[i] = v[4 * t + i] * p.acc_sign + bb[i];
      }
    }
    if constexpr (RQ == 5 || RQ == 6) {
      int32_t y[4];
#pragma unroll
      for (int i = 0; i < 4; i++) {
        // the final arithmetic shift alternates between the FMA pipe (IMAD.HI, 4 cycles per warp on the half-rate
        // "heavy" pipe that IMAD.HI.U32 above already loads) and the ALU pipe (SHF, 2 cycles): see q8_igemm_sm100.cu
        const uint32_t nu = (uint32_t) n[i];
        const uint32_t hi = (uint32_t) (((uint64_t) nu * p.rq.u_m2 + p.rq.u_k2) >> 32);
        const int32_t tt = (int32_t) (hi + (nu >> 31));
        y[i] = (i & 1) ? (tt >> p.rq.shift) : __mulhi(tt, p.rq.u_sm);
        if constexpr (RQ == 6) y[i] = min(max(y[i], p.rq.qmin), p.rq.qmax);
      }
      o[t] = pack_sat_u8x4(y[0], y[1], y[2], y[3]);
    } else {
      o[t] = requant_pack4_generic(n[0], n[1], n[2], n[3], p.rq);
    }
  }
  return make_uint4(o[0], o[1], o[2], o[3]);
}

// 32 bytes = both 16-channel groups of a channel pair for one pixel = one full 32-byte sector in one request
__device__ __forceinline__ void store32(uint8_t* dst, const uint4& lo, const uint4& hi) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(dst), "r"(lo.x), "r"(lo.y), "r"(lo.z), "r"(lo.w),
               "r"(hi.x), "r"(hi.y), "r"(hi.z), "r"(hi.w)
               : "memory");
}

// UMMA-issuing role of warp kMmaWarp + w.  The whole warp walks the loop CONVERGED and every operand is warp-uniform by
// construction (kernel parameters, blockIdx, loop counters, values broadcast with __shfl_sync), so descriptors and
// addresses live in uniform registers and a tcgen05.mma costs its operand arithmetic plus one instruction; an elected
// lane issues.  (Round 1 put the loop under `if (lane == 0)`: nvcc then rebuilt every operand in vector registers and
// moved it across with an ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall, ~30 instructions per UMMA — 17 % of all the
// instructions this kernel executed, profiles/r1h_dwconv_umma_first2.)
// Channel-pair form (DwTcParams::pair): a pixel is 32 bytes (two channel groups) in a SWIZZLE_32B tile, one UMMA per tap
// with K = 32 channels and a 32x32 diagonal B (N = 32: both groups' accumulators side by side).  The A descriptor's start
// address is the tap's pixel — any multiple of 32 bytes: the swizzle is a function of the absolute shared-memory address
// on both the TMA's and the tensor core's side (tools/microbench/sw32_probe.cu), base offset 0.
__device__ __forceinline__ void mma_role_pair(const DwTcParams& p, Ctl& ctl, const ItemDesc* descs, uint32_t smem_base_v,
                                              uint32_t tmem_base_v, int w_v, uint32_t first, uint32_t step, uint32_t total) {
  const int w = __shfl_sync(0xffffffffu, w_v, 0);
  const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base_v, 0);
  const uint32_t smem_base = __shfl_sync(0xffffffffu, smem_base_v, 0);
  const uint32_t ctl_u = __shfl_sync(0xffffffffu, smem_u32(&ctl), 0);
  const uint32_t bar_full = ctl_u + (uint32_t) offsetof(Ctl, full), bar_empty = ctl_u + (uint32_t) offsetof(Ctl, empty);
  const uint32_t bar_tfull = ctl_u + (uint32_t) offsetof(Ctl, tmem_full), bar_tempty = ctl_u + (uint32_t) offsetof(Ctl, tmem_empty);
  const uint32_t idesc = umma_idesc_i8(128, 32, false, p.b_signed != 0);
  // A: K-major SWIZZLE_32B (layout type 6), rows of 32 bytes, SBO = one output row down; B: K-major no swizzle,
  // [2 K-chunks][32 rows][16 B] per tap (LBO = 512 between the chunks, SBO = 128 between 8-row groups)
  const uint32_t ahi = (((uint32_t) p.sbo >> 4) & 0x3FFFu) | (1u << 14) | (6u << 29);
  const uint32_t bhi = (uint32_t) (umma_desc_kmajor_noswizzle(0, 0, 128) >> 32);
  uint32_t alo[kDwTcTaps32], blo[kDwTcTaps32];
#pragma unroll
  for (int t = 0; t < kDwTcTaps32; t++) {
    alo[t] = (((smem_base + (uint32_t) p.a_off9[t]) >> 4) & 0x3FFFu) | (1u << 16);
    // resident weights: the blocks of ALL channel pairs sit behind the ring, indexed by the global pair
    blo[t] = (uint32_t) umma_desc_kmajor_noswizzle(smem_base + (uint32_t) (p.b_resident ? p.b_res_off : p.a_bytes) + (uint32_t) t * 1024u,
                                                   512, 0);
  }
  if (p.b_resident) mbar_wait_parked(ctl_u + (uint32_t) offsetof(Ctl, b_full), 0);
  int stage = 0, as = 0, dslot = 0;
  uint32_t phase = 0, as_phase = 0;
  for (uint32_t item = first; item < total; item += step) {
    mbar_wait_parked(bar_full + 8u * (uint32_t) stage, phase);
    const int mt_eff = __shfl_sync(0xffffffffu, descs[dslot].mt_eff, 0);
    const int g_eff = __shfl_sync(0xffffffffu, descs[dslot].g_eff, 0);
    const uint32_t inv = __shfl_sync(0xffffffffu, descs[dslot].inv, 0);
    const uint32_t pair0 = (uint32_t) __shfl_sync(0xffffffffu, descs[dslot].c0, 0) >> 5;  // first channel pair of the item
    if (++dslot == kDescSlots) dslot = 0;
    const int units = mt_eff * ((g_eff + 1) >> 1);  // (sub-tile, channel pair), sub-tile fastest
    const uint32_t st16 = ((uint32_t) stage * p.stage_bytes) >> 4;
    const uint32_t acc0 = tmem_u + (uint32_t) as * p.acc_stride;
    mbar_wait_parked(bar_tempty + 8u * (uint32_t) as, as_phase ^ 1);
    tc_fence_after_sync();
    if (elect_one()) {
#pragma unroll
      for (int i = 0; i < 2; i++) {  // at most 8 units per item over 7 warps
        const int un = w + i * kMmaWarps;
        if (un >= units) break;
        int j, gp;
        unit_split(un, mt_eff, inv, j, gp);
        const uint32_t s16 = st16 + (((uint32_t) gp * p.cg_bytes) >> 4);   // operand offsets in 16-byte units
        const uint32_t a16 = s16 + (uint32_t) j * 16;                      // 8 pixels x 32 bytes per sub-tile
        const uint32_t b16 = p.b_resident ? ((pair0 + (uint32_t) gp) * (uint32_t) p.b_bytes) >> 4 : s16;
        const uint32_t dcol = acc0 + (uint32_t) (gp * p.mt + j) * 32;
#pragma unroll
        for (int t = 0; t < kDwTcTaps32; t++)
          umma_i8(dcol, pack_u64(alo[t] + a16, ahi), pack_u64(blo[t] + b16, bhi), idesc, t > 0 ? 1u : 0u);
      }
      umma_commit(bar_empty + 8u * (uint32_t) stage);
      umma_commit(bar_tfull + 8u * (uint32_t) as);
    }
    __syncwarp();
    if (++stage == p.num_stages) stage = 0, phase ^= 1;
    as ^= 1;
    if (as == 0) as_phase ^= 1;
  }
}

template <int NB>
__device__ __forceinline__ void mma_role(const DwTcParams& p, Ctl& ctl, const ItemDesc* descs, uint32_t smem_base_v,
                                         uint32_t tmem_base_v, int w_v, uint32_t first, uint32_t step, uint32_t total) {
  const int w = __shfl_sync(0xffffffffu, w_v, 0);
  const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base_v, 0);
  const uint32_t smem_base = __shfl_sync(0xffffffffu, smem_base_v, 0);
  const uint32_t ctl_u = __shfl_sync(0xffffffffu, smem_u32(&ctl), 0);
  const uint32_t bar_full = ctl_u + (uint32_t) offsetof(Ctl, full), bar_empty = ctl_u + (uint32_t) offsetof(Ctl, empty);
  const uint32_t bar_tfull = ctl_u + (uint32_t) offsetof(Ctl, tmem_full), bar_tempty = ctl_u + (uint32_t) offsetof(Ctl, tmem_empty);
  const uint32_t idesc = umma_idesc_i8(128, NB, false, p.b_signed != 0);
  // Shared-memory descriptors split into words: a unit's operand offset only ever changes the 14-bit address field of
  // the LOW word (stages end below 228 KB >> 4 = 14592 < 2^14), the high word (stride, version) is one constant per
  // operand — so a descriptor costs one 32-bit add instead of a 64-bit one plus two register-file crossings.
  uint32_t alo[kDwTcTaps], blo[kDwTcTaps];
  const uint32_t ahi = (uint32_t) (umma_desc_kmajor_noswizzle(0, 0, (uint32_t) p.sbo) >> 32);
  const uint32_t bhi = (uint32_t) (umma_desc_kmajor_noswizzle(0, 0, 128) >> 32);
#pragma unroll
  for (int u = 0; u < kDwTcTaps; u++) {
    alo[u] = (uint32_t) umma_desc_kmajor_noswizzle(smem_base + (uint32_t) p.a_off[u], (uint32_t) p.a_lbo[u], 0);
    blo[u] = (uint32_t) umma_desc_kmajor_noswizzle(smem_base + (uint32_t) (p.b_resident ? p.b_res_off : p.a_bytes) +
                                                       (uint32_t) u * (2 * NB * 16), NB * 16, 0);
  }
  if (p.b_resident) mbar_wait_parked(ctl_u + (uint32_t) offsetof(Ctl, b_full), 0);
  int stage = 0, as = 0, dslot = 0;
  uint32_t phase = 0, as_phase = 0;
  for (uint32_t item = first; item < total; item += step) {
    // the item's operands first — they arrive long before the epilogue frees an accumulator stage (measured: these warps
    // wait 35 % of their time for tmem_empty and never for `full`), so everything that does not need the accumulators is
    // done before that wait and only the UMMA issue itself follows it
    mbar_wait_parked(bar_full + 8u * (uint32_t) stage, phase);
    // mt_eff / units / inv of the item, from the producer's descriptor (same address in every lane: one broadcast load)
    const int mt_eff = __shfl_sync(0xffffffffu, descs[dslot].mt_eff, 0);
    const int units = __shfl_sync(0xffffffffu, descs[dslot].units, 0);
    const uint32_t inv = __shfl_sync(0xffffffffu, descs[dslot].inv, 0);
    const uint32_t group0 = (uint32_t) __shfl_sync(0xffffffffu, descs[dslot].c0, 0) >> 4;  // first channel group of the item
    if (++dslot == kDescSlots) dslot = 0;
    const uint32_t st16 = ((uint32_t) stage * p.stage_bytes) >> 4;
    const uint32_t acc0 = tmem_u + (uint32_t) as * p.acc_stride;
    mbar_wait_parked(bar_tempty + 8u * (uint32_t) as, as_phase ^ 1);
    tc_fence_after_sync();
    if (elect_one()) {
      // this warp's units w, w + 7, ...: a (uniform) early exit instead of predicated-off slots — the straight-line version
      // executed the operand arithmetic of all 15 slots for every item.  The 5 UMMAs of a unit accumulate into the same
      // columns; the other issuing warps' instructions interleave with them in the tensor pipe's queue.
#pragma unroll
      for (int i = 0; i < kMaxUnitsPerMmaWarp; i++) {
        const int un = w + i * kMmaWarps;
        if (un >= units) break;
        int j, gi;
        unit_split(un, mt_eff, inv, j, gi);
        const uint32_t s16 = st16 + (((uint32_t) gi * p.cg_bytes) >> 4);  // operand offsets in 16-byte units
        const uint32_t a16 = s16 + (uint32_t) j * 8;
        const uint32_t b16 = p.b_resident ? ((group0 + (uint32_t) gi) * (uint32_t) p.b_bytes) >> 4 : s16;
        const uint32_t dcol = acc0 + (uint32_t) (gi * p.mt + j) * NB;
#pragma unroll
        for (int u = 0; u < kDwTcTaps; u++)
          umma_i8(dcol, pack_u64(alo[u] + a16, ahi), pack_u64(blo[u] + b16, bhi), idesc, u > 0 ? 1u : 0u);
      }
      umma_commit(bar_empty + 8u * (uint32_t) stage);  // smem stage may be refilled once these UMMAs have read it
      umma_commit(bar_tfull + 8u * (uint32_t) as);     // this warp's share of the accumulators is complete
    }
    __syncwarp();
    if (++stage == p.num_stages) stage = 0, phase ^= 1;
    as ^= 1;
    if (as == 0) as_phase ^= 1;
  }
}

// SMB = DwTcParams::bias_smem (a template parameter, so that the global-table instances are the plain code)
template <int S, int RQ, int NB, bool PAIR, bool SMB>
__global__ void __launch_bounds__(kThreads, 1)
    q8_dwconv3x3_umma_kernel(const __grid_constant__ DwTcParams p, const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ Ctl ctl;
  __shared__ ItemDesc descs[kDescSlots];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;

  if (tid == 0) {
    for (int s = 0; s < p.num_stages; s++) {
      mbar_init(smem_u32(&ctl.full[s]), 1);
      mbar_init(smem_u32(&ctl.empty[s]), kMmaWarps);  // one tcgen05.commit per issuing warp
    }
    for (int s = 0; s < 2; s++) {
      mbar_init(smem_u32(&ctl.tmem_full[s]), kMmaWarps);
      mbar_init(smem_u32(&ctl.tmem_empty[s]), kEpiWarps * 32);
    }
    mbar_init(smem_u32(&ctl.b_full), 1);
    fence_mbar_init();
  }
  if (warp == kMmaWarp) tmem_alloc<kTmemCols>(smem_u32(&ctl.tmem_base));
  if constexpr (SMB) {  // the border classes this geometry produces, all channels (see DwTcParams::bias_smem)
    const uint32_t q4 = (uint32_t) p.channels >> 2;  // 16-byte words per class row
    const uint32_t words = (uint32_t) (p.bias_nrc * p.bias_ncc) * q4;
    int4* dst = reinterpret_cast<int4*>(smem_raw + (smem_base - smem_u32(smem_raw)) + p.bias_off);
    for (uint32_t i = (uint32_t) tid; i < words; i += kThreads) {
      const uint32_t slot = i / q4, r = slot / (uint32_t) p.bias_ncc, c = slot - r * (uint32_t) p.bias_ncc;
      const uint32_t cls = nibble(p.bias_rcls, r) * 8u + nibble(p.bias_ccls, c);
      dst[i] = __ldg(reinterpret_cast<const int4*>(p.bias_cls) + cls * q4 + (i - slot * q4));
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = ctl.tmem_base;
  // Schedule: every CTA owns ONE CONTIGUOUS run of `chunk` items (channel block fastest, then x tile, y tile, image), not
  // every grid-th item.  The channel blocks of a spatial tile — which share 32-byte sectors whenever a pixel's channel
  // block is not sector-aligned (C = 144: every odd pixel) — and the row-halo neighbours are then read and written by the
  // SAME SM within microseconds.  With the round-robin schedule those sector halves came from different CTAs whose skew
  // grew over a launch; measured on b3_dw (C = 144, 56x56): 8.7 GB of DRAM traffic for 3.7 GB of tensors once the
  // kernel's per-item time dropped (L2 hit rate 41 %), against 4.8 GB before.
  const uint32_t first = blockIdx.x * (uint32_t) p.chunk, step = 1u;
  const uint32_t total = min((uint32_t) p.total_items, first + (uint32_t) p.chunk);

  if (warp == kTmaWarp) {
    // ===================================== TMA producer =====================================
    if (lane == 0) {
      int stage = 0, dslot = 0;
      uint32_t phase = 0;
      if (p.b_resident) {  // every weight block of the layer, once
        const uint32_t nbytes = (uint32_t) ((PAIR ? (p.cgs + 1) >> 1 : p.cgs) * p.b_bytes);
        const uint32_t bar = smem_u32(&ctl.b_full);
        mbar_arrive_expect_tx(bar, nbytes);
        for (uint32_t o = 0; o < nbytes; o += 16384u)
          bulk_g2s(smem_base + (uint32_t) p.b_res_off + o, p.wpack + o, nbytes - o < 16384u ? nbytes - o : 16384u, bar);
      }
      ItemPos pos = first_pos(p, first);
      for (uint32_t item = first; item < total; item += step, advance_pos(p, pos)) {
        const DwItem it = make_item(p, pos);
        mbar_wait_relaxed(smem_u32(&ctl.empty[stage]), phase ^ 1, 32);
        {  // the item's descriptor for the other roles (see ItemDesc)
          ItemDesc d;
          d.tile_base = reinterpret_cast<uint64_t>(p.out + ((size_t) ((long long) it.n0 * p.out_h + it.oy0) * p.out_w + it.ox0) * p.out_stride);
          d.n0 = it.n0, d.oy0 = it.oy0, d.ox0 = it.ox0, d.c0 = it.cb * p.G * 16;
          d.mt_eff = it.mt_eff, d.g_eff = it.g_eff;
          d.inv = it.mt_eff == p.mt ? p.inv_g : p.inv_tail;
          d.units = it.mt_eff * it.g_eff;
          d.pad[0] = d.pad[1] = 0;
          const uint4* s4 = reinterpret_cast<const uint4*>(&d);
          uint4* d4 = reinterpret_cast<uint4*>(&descs[dslot]);
          d4[0] = s4[0], d4[1] = s4[1], d4[2] = s4[2];
          if (++dslot == kDescSlots) dslot = 0;
        }
        const uint32_t bar = smem_u32(&ctl.full[stage]);
        const uint32_t dst0 = smem_base + (uint32_t) stage * p.stage_bytes;
        const int y0 = (p.whole ? 0 : it.oy0 * S) - p.pad_top;
        // one box per channel group (16 bytes per pixel) or, in pair mode, per channel PAIR (32 bytes per pixel: every
        // 32-byte sector of the input is requested once instead of twice); channels beyond C are zero-filled by the TMA
        const int blocks = PAIR ? (it.g_eff + 1) >> 1 : it.g_eff;
        const int cbytes = PAIR ? 32 : 16;
        mbar_arrive_expect_tx(bar, (uint32_t) blocks * (uint32_t) (p.planes * p.plane_tx + (p.b_resident ? 0 : p.b_bytes)));
        for (int gi = 0; gi < blocks; gi++) {
          const int cg = (PAIR ? (it.cb * p.G) >> 1 : it.cb * p.G) + gi;
          const uint32_t dst = dst0 + (uint32_t) gi * p.cg_bytes;
          if constexpr (S == 1) {
            tma_load_4d(dst, &tmap, cg * cbytes, it.ox0 + p.x_org[0], y0, it.n0, bar);
          } else {
            tma_load_5d(dst, &tmap, cg * cbytes, 0, it.ox0 + p.x_org[0], y0, it.n0, bar);
            tma_load_5d(dst + p.plane_bytes, &tmap, cg * cbytes, 1, it.ox0 + p.x_org[1], y0, it.n0, bar);
          }
          if (!p.b_resident) bulk_g2s(dst + p.a_bytes, p.wpack + (size_t) cg * p.b_bytes, (uint32_t) p.b_bytes, bar);
        }
        if (++stage == p.num_stages) stage = 0, phase ^= 1;
      }
    }
  } else if (warp >= kMmaWarp && warp < kMmaWarp + kMmaWarps) {
    // ===================================== UMMA issue (7 warps, one lane each) =====================================
    // This layer needs one small UMMA (N = 16/32) per ~400 outputs, i.e. one every ~40 cycles per SM.  nvcc wraps every
    // tcgen05.mma in an elect/broadcast sequence (~27 instructions), and an issuing warp shares its sub-partition with
    // four busy epilogue warps, so one thread manages only one UMMA per ~100 cycles (measured).  Seven warps issue
    // concurrently (1 -> 4 warps: 2x faster; 4 -> 7: another 2-5 %); warp w owns the units w, w+7, ... of every item.
    // (ONE copy of the loop for all of them: per-warp template instances multiply the code and were measured 2.3x slower,
    // presumably instruction-cache misses)
    if constexpr (PAIR) {
      mma_role_pair(p, ctl, descs, smem_base, tmem_base, warp - kMmaWarp, first, step, total);
    } else {
      mma_role<NB>(p, ctl, descs, smem_base, tmem_base, warp - kMmaWarp, first, step, total);
    }
  } else {
    // ===================================== epilogue (16 warps) =====================================
    // Address and border-class arithmetic is split by how often it changes (the round-1 loop redid 64-bit pixel
    // addresses and nine bounds tests per sub-tile and ~70 instructions per item in every warp):
    //   per kernel : the lane's place in an item — image slot, row, column — and its byte offset from the item's origin
    //   per item   : the origin (warp-uniform: item digits and parameters only), the lane's row class, row validity
    //   per sub-tile: column class and validity (a few 32-bit operations)
    //   per unit   : one 32-bit offset each for the bias words and the store
    const int q = warp & 3, h = warp >> 2;
    const int g = 4 * q + (lane >> 3), px = lane & 7;  // row group and column of this thread's TMEM lane
    const int img = g / p.Q, oyl = g - img * p.Q;
    // byte offset of this lane's pixel from the item's first pixel (image n0, row oy0, column ox0); items span at most a
    // few images, so 32 bits suffice (host-checked: nb * out_h * out_w * out_stride < 2^31)
    const uint32_t lane_off = (uint32_t) ((img * p.out_h + oyl) * p.out_w + px) * (uint32_t) p.out_stride;
    const uint32_t sub_step = 8u * (uint32_t) p.out_stride;  // one sub-tile (8 columns) further
    int as = 0, dslot = 0;
    uint32_t as_phase = 0;
    // values that depend on the SPATIAL tile only: with the contiguous schedule (channel block fastest) they change once
    // every `cblocks` items, so they are recomputed only then
    bool row_ok = false;
    uint32_t rm_row = 0;            // index of this lane's row of the bias table (row slot, column slot 0, channel 0)
    const uint32_t bias_sbase = smem_base + (uint32_t) p.bias_off;
    for (uint32_t item = first; item < total; item += step) {
      const uint32_t empty_bar = smem_u32(&ctl.tmem_empty[as]);
      mbar_wait_parked(smem_u32(&ctl.tmem_full[as]), as_phase);
      tc_fence_after_sync();
      const ItemDesc it = load_desc(&descs[dslot]);  // the producer's decode of this item (see ItemDesc)
      if (++dslot == kDescSlots) dslot = 0;
      if (item == first || it.c0 == 0) {
        const int oy = it.oy0 + oyl;
        row_ok = img < p.nb && it.n0 + img < p.batch && oy < p.out_h;
        // row class: bit k set iff input row iy0 + k lies inside the image (taps below 0 / at or above in_h are padding)
        const int iy0 = oy * S - p.pad_top;
        const int rlo = iy0 < 0 ? -iy0 : 0, rhi = iy0 + 3 - p.in_h > 0 ? iy0 + 3 - p.in_h : 0;
        const uint32_t rm = rhi >= 3 ? 0u : (((7u << rlo) & 7u) & (7u >> rhi));
        rm_row = (SMB ? nibble(p.bias_rslot, rm) * (uint32_t) p.bias_rstride : rm * 8u) * (uint32_t) p.channels;
      }
      uint8_t* const obase = reinterpret_cast<uint8_t*>(it.tile_base) + it.c0;
      const uint32_t bias_row = rm_row + (uint32_t) it.c0;
      const uint32_t tbase = tmem_base + (uint32_t) as * p.acc_stride + ((uint32_t) (q * 32) << 16);
      // warp (q, h) takes the units h, h+4, ... (unit = sub-tile j x channel group gi, j fastest); the per-sub-tile
      // values are redone only when j changes
      const int units = it.units;
      const uint32_t inv = it.inv;
      int j_cur = -1;
      uint32_t bias_idx = 0, dst_off = 0;
      bool valid = false;
      auto sub_tile = [&](int j) {  // column class, validity and byte offset of this lane's pixel in sub-tile j
        if (j != j_cur) {
          j_cur = j;
          dst_off = lane_off + (uint32_t) j * sub_step;
          // Sub-tiles that touch neither the left nor the right image border — all but two per image row — have all three
          // tap columns inside the image for every lane: column class 7, every column valid.  The test is warp-uniform
          // (item and sub-tile only); the general form costs ~25 instructions.
          const int ox_first = it.ox0 + 8 * j;
          if (ox_first * S - p.pad_left >= 0 && (ox_first + 7) * S - p.pad_left + 3 <= p.in_w) {
            bias_idx = bias_row + (SMB ? nibble(p.bias_cslot, 7u) : 7u) * (uint32_t) p.channels;
            valid = row_ok;
          } else {
            const int ox = ox_first + px;
            const int ix0 = ox * S - p.pad_left;
            const int clo = ix0 < 0 ? -ix0 : 0, chi = ix0 + 3 - p.in_w > 0 ? ix0 + 3 - p.in_w : 0;
            const uint32_t cm = chi >= 3 ? 0u : (((7u << clo) & 7u) & (7u >> chi));
            bias_idx = bias_row + (SMB ? nibble(p.bias_cslot, cm) : cm) * (uint32_t) p.channels;
            valid = row_ok && ox < p.out_w;
          }
        }
      };
      if (PAIR || p.store32) {
        // Channel groups in PAIRS: the lane requantises groups 2k and 2k+1 of its pixel back to back and writes their
        // 32 bytes with one 256-bit store = one full 32-byte sector per request.  (Per-group 16-byte stores are half-sector
        // writes: twice the requests on the L2, which this kernel loads to 55-75 % of its peak; without any stores it ran
        // 17 % faster.)  Pair p of an item = (sub-tile j, group pair), j fastest; warp (q, h) takes pairs h, h+4, ...
        const int gpairs = (it.g_eff + 1) >> 1;
        const int pairs = it.mt_eff * gpairs;
        if (h >= pairs) {
          tc_fence_before_sync();
          mbar_arrive(empty_bar);
        }
        for (int pu = h; pu < pairs; pu += 4) {
          int j, gp;
          unit_split(pu, it.mt_eff, inv, j, gp);
          sub_tile(j);
          const int gi = 2 * gp;
          const bool two = gi + 1 < it.g_eff, lastp = pu + 4 >= pairs;
          // accumulator columns of (sub-tile j, group gi): pair mode keeps a pair's two groups side by side
          const uint32_t tlo = tbase + (PAIR ? (uint32_t) (gp * p.mt + j) * 32u : (uint32_t) (gi * p.mt + j) * NB);
          const uint32_t thi = PAIR ? tlo + 16u : tbase + (uint32_t) ((gi + 1) * p.mt + j) * NB;
          const uint4 lo = epilogue_unit<RQ, NB, SMB>(p, tlo, bias_idx + (uint32_t) gi * 16u, bias_sbase, lastp && !two, empty_bar);
          uint8_t* const dst = obase + (dst_off + (uint32_t) gi * 16u);
          if (two) {
            const uint4 hi = epilogue_unit<RQ, NB, SMB>(p, thi, bias_idx + (uint32_t) (gi + 1) * 16u, bias_sbase, lastp, empty_bar);
            if (valid) {
              // (pixel strides that are odd multiples of 16 bytes — C = 144 — leave every other pixel 16-byte aligned only:
              // those lanes write their two halves separately, 1.5 instead of 2 requests per 32 bytes on average)
              if ((reinterpret_cast<uintptr_t>(dst) & 31u) == 0) {
                store32(dst, lo, hi);
              } else {
                *reinterpret_cast<uint4*>(dst) = lo;
                *reinterpret_cast<uint4*>(dst + 16) = hi;
              }
            }
          } else {
            if (valid) *reinterpret_cast<uint4*>(dst) = lo;
          }
        }
      } else {
        if (h >= units) {  // nothing to read (narrow tail item)
          tc_fence_before_sync();
          mbar_arrive(empty_bar);
        }
        for (int un = h; un < units; un += 4) {
          int j, gi;
          unit_split(un, it.mt_eff, inv, j, gi);
          sub_tile(j);
          const uint4 o = epilogue_unit<RQ, NB, SMB>(p, tbase + (uint32_t) (gi * p.mt + j) * NB, bias_idx + (uint32_t) gi * 16u, bias_sbase,
                                                un + 4 >= units, empty_bar);
          if (valid) *reinterpret_cast<uint4*>(obase + (dst_off + (uint32_t) gi * 16u)) = o;
        }
      }
      as ^= 1;
      if (as == 0) as_phase ^= 1;
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) {
    __syncwarp();
    tc_fence_after_sync();
    tmem_dealloc<kTmemCols>(tmem_base);
  }
}

// Raises the kernel's dynamic shared-memory limit to everything the device allows beside its static shared memory.
static cudaError_t set_max_dynamic_smem(const void* kern, int max_smem_optin) {
  cudaFuncAttributes fa;
  cudaError_t e = cudaFuncGetAttributes(&fa, kern);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem_optin - (int) fa.sharedSizeBytes);
}

template <int S, int RQ, int NB, bool PAIR, bool SMB>
cudaError_t launch_smb(const DwTcParams& p, const CUtensorMap& tm, int grid, int max_smem_optin, cudaStream_t stream) {
  auto kern = q8_dwconv3x3_umma_kernel<S, RQ, NB, PAIR, SMB>;
  // once per instantiation, to the device maximum (a per-launch value raced between host threads; see the igemm launcher)
  static cudaError_t attr_status = set_max_dynamic_smem(reinterpret_cast<const void*>(kern), max_smem_optin);
  if (attr_status != cudaSuccess) return attr_status;
  kern<<<grid, kThreads, p.smem_total, stream>>>(p, tm);
  return cudaGetLastError();
}

template <int S, int RQ, int NB, bool PAIR = false>
cudaError_t launch_one(const DwTcParams& p, const CUtensorMap& tm, int grid, int max_smem_optin, cudaStream_t stream) {
  return p.bias_smem ? launch_smb<S, RQ, NB, PAIR, true>(p, tm, grid, max_smem_optin, stream)
                     : launch_smb<S, RQ, NB, PAIR, false>(p, tm, grid, max_smem_optin, stream);
}

template <int S, int NB>
cudaError_t launch_rq(const DwTcParams& p, const CUtensorMap& tm, int grid, int max_smem_optin, cudaStream_t stream) {
  if constexpr (NB == 16) {
    if (p.pair) {
      switch (p.rq_mode) {
        case 5: return launch_one<S, 5, 16, true>(p, tm, grid, max_smem_optin, stream);
        case 6: return launch_one<S, 6, 16, true>(p, tm, grid, max_smem_optin, stream);
        default: return launch_one<S, 3, 16, true>(p, tm, grid, max_smem_optin, stream);
      }
    }
  }
  switch (p.rq_mode) {
    case 5: return launch_one<S, 5, NB>(p, tm, grid, max_smem_optin, stream);
    case 6: return launch_one<S, 6, NB>(p, tm, grid, max_smem_optin, stream);
    default: return launch_one<S, 3, NB>(p, tm, grid, max_smem_optin, stream);  // generic q8_requant(): every other mode
  }
}

}  // namespace

cudaError_t launch_q8_dwconv3x3_umma(const DwTcParams& p, const void* tensor_map, int grid, int max_smem_optin,
                                     cudaStream_t stream) {
  alignas(64) CUtensorMap tm;
  memcpy(&tm, tensor_map, sizeof(tm));
  if (p.stride == 1) {
    return p.nb_cols == 32 ? launch_rq<1, 32>(p, tm, grid, max_smem_optin, stream) : launch_rq<1, 16>(p, tm, grid, max_smem_optin, stream);
  }
  return p.nb_cols == 32 ? launch_rq<2, 32>(p, tm, grid, max_smem_optin, stream) : launch_rq<2, 16>(p, tm, grid, max_smem_optin, stream);
}

}  // namespace q8
