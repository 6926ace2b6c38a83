// dvb_cnn.cu — Inception-v3 genotype classifier for sm_100a (B200) + its C ABI.
//
// Replaces the SavedModel call of call_variants.predict_step (deepvariant/call_variants.py:904-932):
//   dv_utils.preprocess_images   deepvariant/dv_utils.py:356-380      (x - 128) / 128
//   keras_modeling.inceptionv3   deepvariant/keras_modeling.py:246-336 (tf_keras InceptionV3 backbone,
//                                                                      pooling='avg')
//   head                         deepvariant/keras_modeling.py:46-67   Dense(3, softmax, float32)
//
// Every convolution (94 of them, BN folded on the host) is an implicit GEMM on the 5th-gen tensor
// cores, written by hand:
//   M = output pixels (batch folded in), N = Cout, K = taps x Cin.
//   A  NHWC fp16 activations, fetched tap by tap with TILED TMA (4-D tensor map {C, W, H, N}): the
//      M tile is a box of Wt x Ht x Nt output pixels, so one cp.async.bulk.tensor per (tap, Cin
//      block) lands a [<=128 rows x BLOCK_K] K-major, hardware-swizzled tile in shared memory;
//      'same' padding and ragged edges are the TMA's out-of-bounds zero fill, stride-2 layers use
//      the tensor map's element strides.
//   B  [Cout][taps][Cin] fp16 weights, 3-D tensor map, one [BLOCK_N x BLOCK_K] tile per K block.
//   D  fp32 accumulators in TMEM (tcgen05.mma.cta_group::1.kind::f16, M=128, N=BLOCK_N, K=16), read back
//      with tcgen05.ld by 4 epilogue warps that add the folded-BN bias, apply ReLU and store fp16
//      straight into the consumer's NHWC tensor at the branch's channel offset (concat = no copy).
//   Warp roles: warp 0 TMA producer, warp 1 TMEM allocator + single-thread MMA issuer, warps 2-5
//   epilogue; a 4-stage mbarrier ring decouples TMA from MMA.
// Pools are small CUDA-core kernels; global-average-pool + Dense(3) + softmax is one fused fp32 tail.

#include <cuda.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "dvb_common.h"

namespace {

constexpr int kMaxStages = 8;
constexpr int kConvThreads = 192;  // warp0 TMA, warp1 MMA, warps 2..5 epilogue
constexpr uint32_t kBlobMagic = 0x31424E4E;    // 'NNB1': one fp16 plane per kernel
constexpr uint32_t kBlobMagic2 = 0x32424E4E;   // 'NNB2': main + residual fp16 planes per kernel (precision 1)

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// Bounded wait: a mis-programmed TMA / MMA must surface as an error, never hang the GPU.
// suspendTimeHint: without it try_wait comes back after a very short system-defined time and the loop below POLLS - ncu's source
// view showed 3.4 M iterations of it in the four epilogue warps of every one-tile-per-CTA kernel (29 % of all stall samples), issue
// slots taken from the MMA / TMA warps of the co-resident CTAs.  With the hint the warp is suspended in hardware until the phase
// completes (wake-up ~60 clocks after the arrive).
constexpr uint32_t kSuspendHintNs = 1000000u;
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  const uint32_t addr = smem_u32(bar);
  uint32_t done = 0;
  unsigned long long t0 = 0;
  for (unsigned it = 0;; ++it) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2, %3;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity), "r"(kSuspendHintNs)
        : "memory");
    if (done) return;
    if ((it & 1023u) == 1023u) {
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > 2000000000ull) {  // 2 s
        printf("dvb_cnn: mbarrier wait timed out (block %d,%d thread %d parity %u)\n", blockIdx.x, blockIdx.y, threadIdx.x, parity);
        __trap();
      }
    }
  }
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// One lane of a CONVERGED warp.  The single-thread instructions of this file (tcgen05.mma / commit, cp.async.bulk.tensor) take their
// operands from uniform registers; when they sit in a branch that ptxas cannot prove single-lane (`if (lane == 0)`), every one of them
// is wrapped in an ELECT / R2UR.BROADCAST / BRA.U.ANY loop (~100-150 clocks per instruction on the issuing thread - measured: 6 MMAs +
// 2 commits took 1000 clocks).  With the whole warp running the loop on uniform values and only the instruction itself under
// elect.sync, ptxas keeps the operands in uniform registers and emits the bare instruction.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile("{\n.reg .pred px;\nelect.sync _|px, 0xffffffff;\n@px mov.s32 %0, 1;\n}\n" : "+r"(pred));
  return pred != 0;
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem];  kind::f16 (fp16 operands, fp32 accumulate)
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on `bar` once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__host__ __device__ __forceinline__ int TmemColsDev(int n) { int c = 32; while (c < n) c <<= 1; return c; }

__device__ __forceinline__ uint4 hmax2x4(const uint4 a, const uint4 b) {
  uint4 r;
  const __half2* x = reinterpret_cast<const __half2*>(&a);
  const __half2* y = reinterpret_cast<const __half2*>(&b);
  __half2* z = reinterpret_cast<__half2*>(&r);
#pragma unroll
  for (int j = 0; j < 4; ++j) z[j] = __hmax2(x[j], y[j]);
  return r;
}

// UMMA shared-memory descriptor, K-major canonical layouts (cute/arch/mma_sm100_desc.hpp SmemDescriptor):
//   [0,14) start>>4  [16,30) LBO>>4  [32,46) SBO>>4  [46,48) version=1  [61,64) layout type
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t sbo_bytes, uint32_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;                          // LBO (unused for swizzled K-major; canonical value 1)
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;                          // descriptor version (Blackwell)
  d |= (uint64_t)(layout_type & 7) << 61;
  return d;
}

// The MMA-issuing thread is ONE thread: every instruction on its dependent chain costs ~4-6 cycles and nothing
// hides it (measured with the clock64 timeline below: 190 cycles per MMA with 64-bit descriptor arithmetic and
// parameter reloads = 3.5k cycles to issue the 18 MMAs of one tile whose tensor work is 0.3k cycles).  So the
// descriptor is kept as two 32-bit halves: `hi` (SBO, version, swizzle) is loop invariant, `lo` (start address >> 4
// plus LBO) advances by plain 32-bit adds, and the 64-bit value is only assembled inside the asm block.
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo_bytes, uint32_t layout_type) {
  return ((sbo_bytes >> 4) & 0x3FFFu) | (1u << 14) | ((layout_type & 7u) << 29);
}
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr) { return ((saddr >> 4) & 0x3FFFu) | (1u << 16); }

__device__ __forceinline__ void umma_f16_lohi(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc,
                                              uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b64 da, db;\n"
      "mov.b64 da, {%1, %3};\n"
      "mov.b64 db, {%2, %3};\n"
      "setp.ne.b32 p, %5, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ void umma_f16_lohi2(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b64 da, db;\n"
      "mov.b64 da, {%1, %2};\n"
      "mov.b64 db, {%3, %4};\n"
      "setp.ne.b32 p, %6, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}

// Epilogue of one accumulator row: TMEM -> registers -> + bias (shared memory, broadcast) -> ReLU -> fp16 -> global.
// All 32 lanes must call it (tcgen05.ld is warp-collective); `valid` masks the stores only.
template <int W>
__device__ __forceinline__ void epilogue_chunk(const uint32_t (&v)[W], const float* s_bias, __half* dst, bool valid, int relu) {
  if (!valid) return;
#pragma unroll
  for (int g = 0; g < W / 8; ++g) {
    const float4 b0 = *reinterpret_cast<const float4*>(s_bias + g * 8);
    const float4 b1 = *reinterpret_cast<const float4*>(s_bias + g * 8 + 4);
    float x[8] = {__uint_as_float(v[g * 8 + 0]) + b0.x, __uint_as_float(v[g * 8 + 1]) + b0.y, __uint_as_float(v[g * 8 + 2]) + b0.z,
                  __uint_as_float(v[g * 8 + 3]) + b0.w, __uint_as_float(v[g * 8 + 4]) + b1.x, __uint_as_float(v[g * 8 + 5]) + b1.y,
                  __uint_as_float(v[g * 8 + 6]) + b1.z, __uint_as_float(v[g * 8 + 7]) + b1.w};
    if (relu) {
#pragma unroll
      for (int j = 0; j < 8; ++j) x[j] = fmaxf(x[j], 0.f);
    }
    uint32_t pk[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      __half2 hh = __floats2half2_rn(x[2 * j], x[2 * j + 1]);
      pk[j] = *reinterpret_cast<uint32_t*>(&hh);
    }
    *reinterpret_cast<uint4*>(dst + g * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
  }
}

__device__ __forceinline__ void epilogue_row(uint32_t taddr, int block_n, const float* s_bias, __half* dst, bool valid, int relu) {
  int c = 0;
  for (; c + 32 <= block_n; c += 32) {
    uint32_t v[32];
    tmem_ld32(taddr + c, v);
    tmem_ld_wait();
    epilogue_chunk<32>(v, s_bias + c, dst + c, valid, relu);
  }
  if (c < block_n) {
    uint32_t v[16];
    tmem_ld16(taddr + c, v);
    tmem_ld_wait();
    epilogue_chunk<16>(v, s_bias + c, dst + c, valid, relu);
  }
}

// ---------------------------------------------------------------------------------------------
// precision = 1: split-fp16 x3 ("fp32-grade" products on the fp16 tensor pipe)
// ---------------------------------------------------------------------------------------------
// Every fp32 value x is carried as two fp16 planes:  x = main + res * 2^-11  with  main = fp16(x),
// res = fp16((x - main) * 2^11).  |x - main| <= 2^-11 |x|, so the scaled residual sits in the same exponent range
// as main (no fp16 underflow for normal x) and the pair holds ~22 significant bits.  A convolution becomes three
// tensor-core products into two TMEM accumulators,
//     D0 += A_main * B_main            D1 += A_main * B_res + A_res * B_main            y = D0 + 2^-11 * D1
// (fp16 x fp16 products are exact in the fp32 accumulator; the dropped A_res * B_res term is 2^-22 relative).
constexpr float kSplitScale = 2048.f;
constexpr float kSplitInv = 1.f / 2048.f;

__device__ __forceinline__ void split_store2(float x0, float x1, uint32_t* main_pk, uint32_t* res_pk) {
  const __half2 m = __floats2half2_rn(x0, x1);
  const float2 mf = __half22float2(m);
  const __half2 r = __floats2half2_rn((x0 - mf.x) * kSplitScale, (x1 - mf.y) * kSplitScale);
  *main_pk = *reinterpret_cast<const uint32_t*>(&m);
  *res_pk = *reinterpret_cast<const uint32_t*>(&r);
}

// Epilogue of one accumulator row in split mode: y = D0 + 2^-11 * D1 + bias -> ReLU -> (main, res) fp16 planes.
__device__ __forceinline__ void epilogue_row_split2(uint32_t taddr, uint32_t taddr1, int block_n, const float* s_bias, __half* dst_main,
                                                    __half* dst_res, bool valid, int relu);
__device__ __forceinline__ void epilogue_row_split(uint32_t taddr, int block_n, const float* s_bias, __half* dst_main, __half* dst_res,
                                                   bool valid, int relu) {
  epilogue_row_split2(taddr, taddr + (uint32_t)block_n, block_n, s_bias, dst_main, dst_res, valid, relu);
}
// D0 columns at taddr, D1 columns at taddr1 (a column range of a wider accumulator pair)
__device__ __forceinline__ void epilogue_row_split2(uint32_t taddr, uint32_t taddr1, int block_n, const float* s_bias, __half* dst_main,
                                                    __half* dst_res, bool valid, int relu) {
  for (int c = 0; c < block_n; c += 16) {
    uint32_t v0[16], v1[16];
    tmem_ld16(taddr + c, v0);
    tmem_ld16(taddr1 + c, v1);
    tmem_ld_wait();
    if (!valid) continue;
#pragma unroll
    for (int g = 0; g < 2; ++g) {
      uint32_t pm[4], pr[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int i = g * 8 + 2 * j;
        float x0 = __uint_as_float(v0[i]) + __uint_as_float(v1[i]) * kSplitInv + s_bias[c + i];
        float x1 = __uint_as_float(v0[i + 1]) + __uint_as_float(v1[i + 1]) * kSplitInv + s_bias[c + i + 1];
        if (relu) { x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); }
        split_store2(x0, x1, &pm[j], &pr[j]);
      }
      *reinterpret_cast<uint4*>(dst_main + c + g * 8) = make_uint4(pm[0], pm[1], pm[2], pm[3]);
      *reinterpret_cast<uint4*>(dst_res + c + g * 8) = make_uint4(pr[0], pr[1], pr[2], pr[3]);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Convolution = implicit GEMM
// ---------------------------------------------------------------------------------------------
constexpr int kMaxSegs = 4;
struct OutSeg { int col_begin, cstride, coff, relu; __half* out; };   // columns [col_begin, next col_begin) of the GEMM

struct ConvArgs {
  int kh, kw, pad_h, pad_w, stride;
  int cin_blocks, block_k;        // K per stage (16 / 32 / 64 fp16 = 32 / 64 / 128-byte swizzle)
  int Wt, Ht, Nt;                 // output-pixel box of one M tile (Wt*Ht*Nt <= 128)
  int tiles_w, tiles_h, tiles_n;
  int Hout, Wout, n_images;
  int block_n, tmem_cols, stages;
  int out_cstride, out_coff, relu;
  uint32_t idesc, layout_type, sbo_bytes;
  uint32_t a_bytes, b_bytes, a_stage, b_stage;  // TMA bytes and shared-memory footprint per stage
  __half* out;
  const float* bias;
  // merged 1x1 convolutions (several layers reading the same tensor run as ONE GEMM over the concatenated filters):
  // column ranges of N go to different tensors.  n_segs == 0: single destination (out / out_cstride / out_coff / relu).
  int n_segs;
  OutSeg segs[kMaxSegs];
  // split mode (precision 1): residual planes; a_stage / b_stage then hold {main, res} tiles back to back
  __half* out_res;
  uint32_t a_res_off, b_res_off;
  int skip_a_res;                 // the A residual plane is identically zero (network input): skip its load and MMA
  uint32_t idesc_cat;             // split mode: N = 2 * block_n over [B_main ; B_res] when the two tiles are contiguous in a stage, else 0
  int dbg;                        // timing probes (DVB_CNN_DBG; results are garbage): 1 = no TMA loads, MMAs do not wait; 2 = TMA loads, no MMAs
  long long* trace;               // optional clock64 timeline of CTA 0's MMA warp: [k block][4] = stage full seen, MMAs issued, commit issued
};
#define GEMM_TRACE(i, ev) do { if (p.trace && blockIdx.x == 0 && lane == 0 && (i) < 96) p.trace[(i) * 4 + (ev)] = clock64(); } while (0)

// Epilogue of one accumulator row of a merged GEMM: 16-column chunks, each routed to the tensor that owns its column
// range (range boundaries are multiples of 16).  `pix` = flat output pixel index, `col0` = first GEMM column of this row piece.
__device__ __forceinline__ void epilogue_row_segs(uint32_t taddr, int n_cols, int col0, const float* s_bias, const ConvArgs& p, size_t pix,
                                                  bool valid) {
  for (int c = 0; c < n_cols; c += 16) {
    uint32_t v[16];
    tmem_ld16(taddr + c, v);
    tmem_ld_wait();
    const int cg = col0 + c;
    int k = 0;
#pragma unroll
    for (int j = 1; j < kMaxSegs; ++j)
      if (j < p.n_segs && cg >= p.segs[j].col_begin) k = j;
    const OutSeg& sg = p.segs[k];
    epilogue_chunk<16>(v, s_bias + c, sg.out + pix * sg.cstride + sg.coff + (cg - sg.col_begin), valid, sg.relu);
  }
}

template <bool kSplit>
__global__ void __launch_bounds__(kConvThreads, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                 const __grid_constant__ CUtensorMap map_a_res, const __grid_constant__ CUtensorMap map_b_res, const ConvArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic (not an integer round trip): ptxas keeps the shared address space -> LDS / STS, not generic LD / ST
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + p.stages * p.a_stage;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + p.stages * p.b_stage);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + kMaxStages;
  uint64_t* tmem_full = bars + 2 * kMaxStages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 1);
  float* s_bias = reinterpret_cast<float*>(bars + 2 * kMaxStages + 2);   // [block_n]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < p.block_n; i += kConvThreads) s_bias[i] = p.bias[blockIdx.y * p.block_n + i];
  // tile coordinates
  int t = blockIdx.x;
  const int tw = t % p.tiles_w; t /= p.tiles_w;
  const int th = t % p.tiles_h; t /= p.tiles_h;
  const int tn = t;
  const int w0 = tw * p.Wt, h0 = th * p.Ht, n0 = tn * p.Nt;
  const int nb = blockIdx.y;
  const int num_kb = p.kh * p.kw * p.cin_blocks;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&map_a);
    prefetch_tmap(&map_b);
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(tmem_full, 1);
    fence_barrier_init();
  } else if (warp == 1) {
    tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    {
      // ===== TMA producer (the whole warp walks the loop, one elected lane issues) =====
      if constexpr (kSplit) { if (elect_one()) { prefetch_tmap(&map_a_res); prefetch_tmap(&map_b_res); } __syncwarp(); }
      int st = 0;
      uint32_t ph = 0;
      for (int r = 0; r < p.kh && !(p.dbg & 1); ++r) {
        for (int s = 0; s < p.kw; ++s) {
          for (int cb = 0; cb < p.cin_blocks; ++cb) {
            mbar_wait(&empty_bar[st], ph ^ 1);
            if (elect_one()) {
              if constexpr (kSplit) {
                mbar_arrive_expect_tx(&full_bar[st], (p.skip_a_res ? 1u : 2u) * p.a_bytes + 2u * p.b_bytes);
                if (!p.skip_a_res)
                  tma_load_4d(smem_a + st * p.a_stage + p.a_res_off, &map_a_res, &full_bar[st], cb * p.block_k, w0 * p.stride + s - p.pad_w,
                              h0 * p.stride + r - p.pad_h, n0);
                tma_load_3d(smem_b + st * p.b_stage + p.b_res_off, &map_b_res, &full_bar[st], cb * p.block_k, r * p.kw + s, nb * p.block_n);
              } else {
                mbar_arrive_expect_tx(&full_bar[st], p.a_bytes + p.b_bytes);
              }
              tma_load_4d(smem_a + st * p.a_stage, &map_a, &full_bar[st], cb * p.block_k, w0 * p.stride + s - p.pad_w,
                          h0 * p.stride + r - p.pad_h, n0);
              tma_load_3d(smem_b + st * p.b_stage, &map_b, &full_bar[st], cb * p.block_k, r * p.kw + s, nb * p.block_n);
            }
            __syncwarp();
            if (++st == p.stages) { st = 0; ph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    {
      // ===== MMA issuer (the whole warp walks the loop, one elected lane issues) =====
      const int mma_per_kb = p.block_k / 16;
      const uint32_t hi = desc_hi(p.sbo_bytes, p.layout_type), idesc = p.idesc;
      const uint32_t a_lo0 = desc_lo(smem_u32(smem_a)), b_lo0 = desc_lo(smem_u32(smem_b));
      const uint32_t a_inc = p.a_stage >> 4, b_inc = p.b_stage >> 4;
      const int stages = p.stages;
      int st = 0;
      uint32_t ph = 0, a_lo = a_lo0, b_lo = b_lo0, acc = 0;
      for (int kb = 0; kb < num_kb; ++kb) {
        if (!(p.dbg & 1)) mbar_wait(&full_bar[st], ph);
        // (non-split mode: a second K block rides in the same elected round when its stage has landed as well - see the persistent kernel)
        int st2 = st + 1;
        uint32_t ph2 = ph, a_lo2 = a_lo + a_inc, b_lo2 = b_lo + b_inc;
        if (st2 == stages) { st2 = 0; ph2 ^= 1; a_lo2 = a_lo0; b_lo2 = b_lo0; }
        const bool two = !kSplit && (p.dbg & 4) && kb + 1 < num_kb && stages > 1;   // off: measured 10 % slower here (2-3 stages: the producer loses its lead)
        if (two && !(p.dbg & 1)) mbar_wait(&full_bar[st2], ph2);
        tc_fence_after();
        if (elect_one()) {
          if (p.dbg & 2) {
          } else if constexpr (kSplit) {
            const uint32_t a_res = a_lo + (p.a_res_off >> 4), b_res = b_lo + (p.b_res_off >> 4), d1 = tmem_base + (uint32_t)p.block_n;
            const bool with_a_res = !p.skip_a_res;
            if (p.idesc_cat) {
              // [D0 | D1] += A_main * [B_main ; B_res] as ONE instruction of N = 2 block_n (the two filter tiles are adjacent rows of the
              // stage and the two accumulators adjacent TMEM columns): 2 MMAs per K step instead of 3, same products, same order
              for (int k = 0; k < mma_per_kb; ++k) {
                umma_f16_lohi(tmem_base, a_lo + 2 * k, b_lo + 2 * k, hi, p.idesc_cat, acc | (uint32_t)(k != 0));
                if (with_a_res) umma_f16_lohi(d1, a_res + 2 * k, b_lo + 2 * k, hi, idesc, 1u);   // D1 += A_res * B_main
              }
            } else {
              for (int k = 0; k < mma_per_kb; ++k) {
                const uint32_t ac = acc | (uint32_t)(k != 0);
                umma_f16_lohi(tmem_base, a_lo + 2 * k, b_lo + 2 * k, hi, idesc, ac);   // D0 += A_main * B_main
                umma_f16_lohi(d1, a_lo + 2 * k, b_res + 2 * k, hi, idesc, ac);         // D1 += A_main * B_res
                if (with_a_res) umma_f16_lohi(d1, a_res + 2 * k, b_lo + 2 * k, hi, idesc, 1u);   // D1 += A_res * B_main
              }
            }
          } else {
#pragma unroll 4
            for (int k = 0; k < mma_per_kb; ++k) umma_f16_lohi(tmem_base, a_lo + 2 * k, b_lo + 2 * k, hi, idesc, acc | (uint32_t)(k != 0));
          }
          umma_commit(&empty_bar[st]);   // frees the stage once these MMAs retire
          if (two) {
            if (!(p.dbg & 2)) {
#pragma unroll 4
              for (int k = 0; k < mma_per_kb; ++k) umma_f16_lohi(tmem_base, a_lo2 + 2 * k, b_lo2 + 2 * k, hi, idesc, 1u);
            }
            umma_commit(&empty_bar[st2]);
          }
        }
        __syncwarp();
        acc = 1;
        if (two) { st = st2; ph = ph2; a_lo = a_lo2; b_lo = b_lo2; ++kb; }
        a_lo += a_inc; b_lo += b_inc;
        if (++st == stages) { st = 0; ph ^= 1; a_lo = a_lo0; b_lo = b_lo0; }
      }
      if (elect_one()) umma_commit(tmem_full);          // accumulator complete
      __syncwarp();
    }
  } else {
    // ===== epilogue: TMEM -> registers -> bias + ReLU -> fp16 -> NHWC global =====
    const int q = warp & 3;                   // TMEM lane quarter this warp may access
    const int row = q * 32 + lane;            // accumulator row = pixel index inside the tile
    const int w = row % p.Wt;
    const int h = (row / p.Wt) % p.Ht;
    const int n = row / (p.Wt * p.Ht);
    const bool valid = (n < p.Nt) && (w0 + w < p.Wout) && (h0 + h < p.Hout) && (n0 + n < p.n_images);
    __half* dst = p.out + ((size_t)((size_t)(n0 + n) * p.Hout + (h0 + h)) * p.Wout + (w0 + w)) * p.out_cstride + p.out_coff +
                  nb * p.block_n;
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    if constexpr (kSplit)
      epilogue_row_split(tmem_base + ((uint32_t)(q * 32) << 16), p.block_n, s_bias, dst, p.out_res + (dst - p.out), valid, p.relu);
    else if (p.n_segs)
      epilogue_row_segs(tmem_base + ((uint32_t)(q * 32) << 16), p.block_n, nb * p.block_n, s_bias, p,
                        (size_t)((size_t)(n0 + n) * p.Hout + (h0 + h)) * p.Wout + (w0 + w), valid);
    else
      epilogue_row(tmem_base + ((uint32_t)(q * 32) << 16), p.block_n, s_bias, dst, valid, p.relu);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

// ---------------------------------------------------------------------------------------------
// Persistent variant of the tap-by-tap implicit GEMM (precision 0)
// ---------------------------------------------------------------------------------------------
// Measured on the one-tile-per-CTA kernel above (ncu, 1x1 768->192 on 4x12 maps): tensor pipe 31 %, L2 32 %, DRAM 35 %,
// 18 % of the warp slots occupied - nothing is saturated.  Each CTA pays TMEM allocation, barrier init and a cold
// 2-stage pipeline for 12 K blocks of work, and only two CTAs fit an SM (TMEM 2 x 256 columns, 2 x 80 KB).  Here ONE
// CTA per SM stays resident and walks (M tile, N block) pairs: a deep TMA ring (as many stages as fit ~200 KB) runs
// ahead across tile boundaries, the accumulator is double buffered in TMEM (2 x BLOCK_N <= 512 columns) and eight
// epilogue warps (two per TMEM lane quarter, splitting the columns) drain tile i while the MMAs of tile i + 1 issue.
constexpr int kPersistEpiWarps = 8;
constexpr int kPersistThreads = 64 + 32 * kPersistEpiWarps;   // warp 0 TMA, warp 1 MMA, warps 2..9 epilogue

__global__ void __launch_bounds__(kPersistThreads, 1)
conv_gemm_persistent_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const ConvArgs p,
                            const int n_blocks, const int cout) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic (not an integer round trip): ptxas keeps the shared address space -> LDS / STS, not generic LD / ST
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + p.stages * p.a_stage;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + p.stages * p.b_stage);
  uint64_t* full_bar = bars;                       // [kMaxStages]
  uint64_t* empty_bar = bars + kMaxStages;         // [kMaxStages]
  uint64_t* tmem_full = bars + 2 * kMaxStages;     // [2]
  uint64_t* tmem_empty = bars + 2 * kMaxStages + 2;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 4);
  float* s_bias = reinterpret_cast<float*>(bars + 2 * kMaxStages + 6);   // [cout], 16-byte aligned

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < cout; i += kPersistThreads) s_bias[i] = p.bias[i];
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int total = m_tiles * n_blocks;             // tile t = nb * m_tiles + m  (neighbouring CTAs share the weight block)
  const int num_kb = p.kh * p.kw * p.cin_blocks;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&map_a);
    prefetch_tmap(&map_b);
    for (int s = 0; s < p.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], 32 * kPersistEpiWarps); }
    fence_barrier_init();
  } else if (warp == 1) {
    tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    {
      // ===== TMA producer (whole warp, one elected lane issues) =====
      int st = 0;
      uint32_t ph = 0;
      for (int t = blockIdx.x; t < total && !(p.dbg & 1); t += gridDim.x) {
        const int nb = t / m_tiles;
        int m = t - nb * m_tiles;
        const int tw = m % p.tiles_w; m /= p.tiles_w;
        const int th = m % p.tiles_h;
        const int tn = m / p.tiles_h;
        const int w0 = tw * p.Wt * p.stride - p.pad_w, h0 = th * p.Ht * p.stride - p.pad_h, n0 = tn * p.Nt;
        for (int r = 0; r < p.kh; ++r) {
          for (int s = 0; s < p.kw; ++s) {
            for (int cb = 0; cb < p.cin_blocks; ++cb) {
              mbar_wait(&empty_bar[st], ph ^ 1);
              if (elect_one()) {
                mbar_arrive_expect_tx(&full_bar[st], p.a_bytes + p.b_bytes);
                tma_load_4d(smem_a + st * p.a_stage, &map_a, &full_bar[st], cb * p.block_k, w0 + s, h0 + r, n0);
                tma_load_3d(smem_b + st * p.b_stage, &map_b, &full_bar[st], cb * p.block_k, r * p.kw + s, nb * p.block_n);
              }
              __syncwarp();
              if (++st == p.stages) { st = 0; ph ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    {
      // ===== MMA issuer (whole warp, one elected lane issues) =====
      const int mma_per_kb = p.block_k / 16;
      const uint32_t hi = desc_hi(p.sbo_bytes, p.layout_type), idesc = p.idesc;
      const uint32_t a_lo0 = desc_lo(smem_u32(smem_a)), b_lo0 = desc_lo(smem_u32(smem_b));
      const uint32_t a_inc = p.a_stage >> 4, b_inc = p.b_stage >> 4;
      const int stages = p.stages;
      int st = 0, buf = 0, tr_i = 0;
      uint32_t ph = 0, buf_ph = 0, a_lo = a_lo0, b_lo = b_lo0;
      for (int t = blockIdx.x; t < total; t += gridDim.x) {
        mbar_wait(&tmem_empty[buf], buf_ph ^ 1);      // the epilogue has drained this accumulator
        tc_fence_after();
        const uint32_t d = tmem_base + (uint32_t)(buf * p.block_n);
        uint32_t acc = 0;
        // two K blocks per elected round: the per-round cost on the issuing warp (barrier observation ~90 clocks, elect + warp
        // synchronisation, loop state: ~280 clocks measured between a commit and the next MMA) is paid once per 8 MMAs instead of per 4
        for (int kb = 0; kb < num_kb; kb += 2) {
          const bool two = kb + 1 < num_kb;
          int st2 = st + 1;
          uint32_t ph2 = ph, a_lo2 = a_lo + a_inc, b_lo2 = b_lo + b_inc;
          if (st2 == stages) { st2 = 0; ph2 ^= 1; a_lo2 = a_lo0; b_lo2 = b_lo0; }
          if (!(p.dbg & 1)) {
            mbar_wait(&full_bar[st], ph);
            if (two) mbar_wait(&full_bar[st2], ph2);
          }
          tc_fence_after();
          GEMM_TRACE(tr_i, 0);
          if (elect_one()) {
            if (!(p.dbg & 2)) {
#pragma unroll 4
              for (int k = 0; k < mma_per_kb; ++k) umma_f16_lohi(d, a_lo + 2 * k, b_lo + 2 * k, hi, idesc, acc | (uint32_t)(k != 0));
            }
            umma_commit(&empty_bar[st]);
            GEMM_TRACE(tr_i, 1);
            if (two) {
              if (!(p.dbg & 2)) {
#pragma unroll 4
                for (int k = 0; k < mma_per_kb; ++k) umma_f16_lohi(d, a_lo2 + 2 * k, b_lo2 + 2 * k, hi, idesc, 1u);
              }
              umma_commit(&empty_bar[st2]);
            }
            GEMM_TRACE(tr_i, 2);
          }
          __syncwarp();
          ++tr_i;
          acc = 1;
          if (two) { st = st2; ph = ph2; a_lo = a_lo2; b_lo = b_lo2; }
          a_lo += a_inc; b_lo += b_inc;
          if (++st == stages) { st = 0; ph ^= 1; a_lo = a_lo0; b_lo = b_lo0; }
        }
        if (elect_one()) umma_commit(&tmem_full[buf]);
        __syncwarp();
        buf ^= 1;
        if (buf == 0) buf_ph ^= 1;
      }
    }
  } else {
    // ===== epilogue: warp e covers TMEM lane quarter (warp & 3) and column half (e >> 2) =====
    const int e = warp - 2;
    const int q = warp & 3;
    const int half = e >> 2;
    const int row = q * 32 + lane;
    const int w = row % p.Wt;
    const int h = (row / p.Wt) % p.Ht;
    const int n = row / (p.Wt * p.Ht);
    // column split in multiples of 16: first half gets ceil
    const int chunks = p.block_n >> 4;
    const int c_lo = half == 0 ? 0 : ((chunks + 1) >> 1) << 4;
    const int c_n = half == 0 ? ((chunks + 1) >> 1) << 4 : p.block_n - c_lo;
    int buf = 0;
    uint32_t buf_ph = 0;
    for (int t = blockIdx.x; t < total; t += gridDim.x) {
      const int nb = t / m_tiles;
      int m = t - nb * m_tiles;
      const int tw = m % p.tiles_w; m /= p.tiles_w;
      const int th = m % p.tiles_h;
      const int tn = m / p.tiles_h;
      const int w0 = tw * p.Wt, h0 = th * p.Ht, n0 = tn * p.Nt;
      const bool valid = (n < p.Nt) && (w0 + w < p.Wout) && (h0 + h < p.Hout) && (n0 + n < p.n_images);
      __half* dst = p.out + ((size_t)((size_t)(n0 + n) * p.Hout + (h0 + h)) * p.Wout + (w0 + w)) * p.out_cstride + p.out_coff +
                    nb * p.block_n + c_lo;
      mbar_wait(&tmem_full[buf], buf_ph);
      tc_fence_after();
      if (c_n > 0) {
        if (p.n_segs)
          epilogue_row_segs(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * p.block_n + c_lo), c_n, nb * p.block_n + c_lo,
                            s_bias + nb * p.block_n + c_lo, p, (size_t)((size_t)(n0 + n) * p.Hout + (h0 + h)) * p.Wout + (w0 + w), valid);
        else
          epilogue_row(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * p.block_n + c_lo), c_n, s_bias + nb * p.block_n + c_lo, dst,
                       valid, p.relu);
      }
      tc_fence_before();
      mbar_arrive(&tmem_empty[buf]);
      buf ^= 1;
      if (buf == 0) buf_ph ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

// ---------------------------------------------------------------------------------------------
// CTA-pair variant of the persistent kernel (tcgen05 cta_group::2, M = 256): DVB_CNN_PAIR=1, off by default until measured
// ---------------------------------------------------------------------------------------------
// Two CTAs of a 2-CTA cluster (one TPC) work on TWO neighbouring M tiles against the SAME N block.  Each CTA stages its own
// 128-row A tile and only HALF of the weight block (block_n / 2 filter rows); the leader CTA (cluster rank 0) issues one
// tcgen05.mma.cta_group::2 per K step with M = 256, N = block_n, which reads both CTAs' shared memory at the same offsets and
// writes rows 0-127 of the accumulator into the leader's TMEM and rows 128-255 into the peer's.  Per SM the operand stream per MMA
// drops from 4 KB + 32 N to 4 KB + 16 N bytes (DESIGN.md section 4: the SS-mode ceiling N / (128 + N) becomes N / (128 + N / 2)).
// Barriers: both CTAs' TMA loads complete on the LEADER's full barrier (cp.async.bulk.tensor ... cta_group::2 with the barrier
// address of the even CTA); tcgen05.commit ... multicast::cluster releases the stage / publishes the accumulator in BOTH CTAs;
// the epilogue threads of both CTAs arrive on the leader's tmem_empty barrier (mapa + remote arrive).
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;    // cute::Sm100MmaPeerBitMask: shared::cluster address of the even CTA of a pair

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_4d_2sm(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d_2sm(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* dst_smem, uint32_t ncols) {   // one warp in EACH CTA, same warp id, same offset
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16_lohi_2cta(uint32_t d_tmem, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc,
                                                   uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      ".reg .b64 da, db;\n"
      "mov.b64 da, {%1, %3};\n"
      "mov.b64 db, {%2, %3};\n"
      "setp.ne.b32 p, %5, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %4, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the barrier at this shared-memory offset in BOTH CTAs of the pair once the issued MMAs have completed
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar) {
  asm volatile(
      "{\n"
      ".reg .b16 mask;\n"
      "mov.b16 mask, 3;\n"
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], mask;\n"
      "}\n" ::"r"(smem_u32(bar))
      : "memory");
}
// arrive on the barrier at this offset in the cluster's rank-0 CTA
__device__ __forceinline__ void mbar_arrive_rank0(uint64_t* bar) {
  asm volatile(
      "{\n"
      ".reg .b32 ra;\n"
      "mapa.shared::cluster.u32 ra, %0, 0;\n"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n"
      "}\n" ::"r"(smem_u32(bar))
      : "memory");
}

struct PairArgs {
  uint32_t idesc;        // M = 256
  uint32_t b_half_bytes, b_half_stage;
  int stages;
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kPersistThreads, 1)
conv_gemm_pair_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b_half, const ConvArgs p,
                      const PairArgs q2, const int n_blocks, const int cout) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic (not an integer round trip): ptxas keeps the shared address space -> LDS / STS, not generic LD / ST
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + q2.stages * p.a_stage;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_b + q2.stages * q2.b_half_stage);
  uint64_t* full_bar = bars;                       // [kMaxStages]   used in the leader
  uint64_t* empty_bar = bars + kMaxStages;         // [kMaxStages]   both CTAs (multicast commit)
  uint64_t* tmem_full = bars + 2 * kMaxStages;     // [2]            both CTAs (multicast commit)
  uint64_t* tmem_empty = bars + 2 * kMaxStages + 2;   // [2]         used in the leader: epilogue threads of both CTAs arrive
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 4);
  float* s_bias = reinterpret_cast<float*>(bars + 2 * kMaxStages + 6);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  for (int i = threadIdx.x; i < cout; i += kPersistThreads) s_bias[i] = p.bias[i];
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  const int m_pairs = (m_tiles + 1) >> 1;
  const int total = m_pairs * n_blocks;             // pair tile t = nb * m_pairs + mp; CTA `rank` takes M tile 2 mp + rank
  const int num_kb = p.kh * p.kw * p.cin_blocks;
  const int pair_id = blockIdx.x >> 1, num_pairs = gridDim.x >> 1;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&map_a);
    prefetch_tmap(&map_b_half);
    for (int s = 0; s < q2.stages; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], 2 * 32 * kPersistEpiWarps); }
    fence_barrier_init();
  } else if (warp == 1) {
    tmem_alloc_2cta(tmem_slot, (uint32_t)p.tmem_cols);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();        // the peer's barriers and TMEM exist before anything remote touches them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    {
      // ===== TMA producer (both CTAs; whole warp, one elected lane issues): own A tile + own half of the weight block, completing on the leader's barrier =====
      int st = 0;
      uint32_t ph = 0;
      for (int t = pair_id; t < total; t += num_pairs) {
        const int nb = t / m_pairs;
        int m = 2 * (t - nb * m_pairs) + (int)rank;       // m >= m_tiles (odd tile count): every coordinate is out of bounds -> zeros
        const int tw = m % p.tiles_w; m /= p.tiles_w;
        const int th = m % p.tiles_h;
        const int tn = m / p.tiles_h;
        const int w0 = tw * p.Wt * p.stride - p.pad_w, h0 = th * p.Ht * p.stride - p.pad_h, n0 = tn * p.Nt;
        for (int r = 0; r < p.kh; ++r) {
          for (int s = 0; s < p.kw; ++s) {
            for (int cb = 0; cb < p.cin_blocks; ++cb) {
              mbar_wait(&empty_bar[st], ph ^ 1);
              if (elect_one()) {
                if (leader) mbar_arrive_expect_tx(&full_bar[st], 2u * (p.a_bytes + q2.b_half_bytes));
                tma_load_4d_2sm(smem_a + st * p.a_stage, &map_a, &full_bar[st], cb * p.block_k, w0 + s, h0 + r, n0);
                tma_load_3d_2sm(smem_b + st * q2.b_half_stage, &map_b_half, &full_bar[st], cb * p.block_k, r * p.kw + s,
                                nb * p.block_n + (int)rank * (p.block_n >> 1));
              }
              __syncwarp();
              if (++st == q2.stages) { st = 0; ph ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (leader) {
      // ===== MMA issuer: warp 1 of the leader CTA, one elected lane issues =====
      const int mma_per_kb = p.block_k / 16;
      const uint32_t hi = desc_hi(p.sbo_bytes, p.layout_type), idesc = q2.idesc;
      const uint32_t a_lo0 = desc_lo(smem_u32(smem_a)), b_lo0 = desc_lo(smem_u32(smem_b));
      const uint32_t a_inc = p.a_stage >> 4, b_inc = q2.b_half_stage >> 4;
      const int stages = q2.stages;
      int st = 0, buf = 0;
      uint32_t ph = 0, buf_ph = 0, a_lo = a_lo0, b_lo = b_lo0;
      for (int t = pair_id; t < total; t += num_pairs) {
        mbar_wait(&tmem_empty[buf], buf_ph ^ 1);      // both CTAs' epilogues have drained this accumulator
        tc_fence_after();
        const uint32_t d = tmem_base + (uint32_t)(buf * p.block_n);
        uint32_t acc = 0;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(&full_bar[st], ph);
          tc_fence_after();
          if (elect_one()) {
#pragma unroll 4
            for (int k = 0; k < mma_per_kb; ++k) umma_f16_lohi_2cta(d, a_lo + 2 * k, b_lo + 2 * k, hi, idesc, acc | (uint32_t)(k != 0));
            umma_commit_2cta(&empty_bar[st]);
          }
          __syncwarp();
          acc = 1;
          a_lo += a_inc; b_lo += b_inc;
          if (++st == stages) { st = 0; ph ^= 1; a_lo = a_lo0; b_lo = b_lo0; }
        }
        if (elect_one()) umma_commit_2cta(&tmem_full[buf]);
        __syncwarp();
        buf ^= 1;
        if (buf == 0) buf_ph ^= 1;
      }
    }
  } else {
    // ===== epilogue (both CTAs): rows of this CTA's own M tile from its own TMEM =====
    const int e = warp - 2;
    const int q = warp & 3;
    const int half = e >> 2;
    const int row = q * 32 + lane;
    const int w = row % p.Wt;
    const int h = (row / p.Wt) % p.Ht;
    const int n = row / (p.Wt * p.Ht);
    const int chunks = p.block_n >> 4;
    const int c_lo = half == 0 ? 0 : ((chunks + 1) >> 1) << 4;
    const int c_n = half == 0 ? ((chunks + 1) >> 1) << 4 : p.block_n - c_lo;
    int buf = 0;
    uint32_t buf_ph = 0;
    for (int t = pair_id; t < total; t += num_pairs) {
      const int nb = t / m_pairs;
      int m = 2 * (t - nb * m_pairs) + (int)rank;
      const bool tile_exists = m < m_tiles;
      const int tw = m % p.tiles_w; m /= p.tiles_w;
      const int th = m % p.tiles_h;
      const int tn = m / p.tiles_h;
      const int w0 = tw * p.Wt, h0 = th * p.Ht, n0 = tn * p.Nt;
      const bool valid = tile_exists && (n < p.Nt) && (w0 + w < p.Wout) && (h0 + h < p.Hout) && (n0 + n < p.n_images);
      const size_t pix = (size_t)((size_t)(n0 + n) * p.Hout + (h0 + h)) * p.Wout + (w0 + w);
      __half* dst = p.out + pix * p.out_cstride + p.out_coff + nb * p.block_n + c_lo;
      mbar_wait(&tmem_full[buf], buf_ph);
      tc_fence_after();
      if (c_n > 0) {
        if (p.n_segs)
          epilogue_row_segs(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * p.block_n + c_lo), c_n, nb * p.block_n + c_lo,
                            s_bias + nb * p.block_n + c_lo, p, pix, valid);
        else
          epilogue_row(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * p.block_n + c_lo), c_n, s_bias + nb * p.block_n + c_lo, dst,
                       valid, p.relu);
      }
      tc_fence_before();
      mbar_arrive_rank0(&tmem_empty[buf]);
      buf ^= 1;
      if (buf == 0) buf_ph ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();        // no CTA leaves (or frees TMEM) while its partner may still read its shared memory
  if (warp == 1) tmem_dealloc_2cta(tmem_base, (uint32_t)p.tmem_cols);
}

// ---------------------------------------------------------------------------------------------
// Stride-1 k x k convolution on large feature maps: persistent, weights-resident, halo-reusing variant
// ---------------------------------------------------------------------------------------------
// What the tap-by-tap kernel above cannot hide on the wide stem layers (measured, B200):
//   * every input pixel is fetched kh*kw times and the weights once per M tile: 55-60 % of L2->SM throughput with
//     the tensor pipe < 35 % busy;
//   * MMAs that accumulate into the SAME TMEM tile form a dependent chain with ~160-250 cycles per link, far more
//     than the 16-48 cycles an M=128, N=32..96 MMA occupies the tensor core (clock64 timeline of one CTA).
// Here one CTA per SM keeps the WHOLE weight slice of its N block in shared memory for its lifetime and walks M
// tiles persistently in groups of T tiles.  An M tile is Ht output rows x P slots (Ht * P = 128).  Per
// (tile, Cin block) ONE TMA box brings the (Ht + kh) x P input halo; every tap (r, s) is the same shared-memory
// block read from a start address shifted by r*P + s pixels (UMMA shared-memory descriptors swizzle on absolute
// address bits: a shifted start needs no "base offset" — measured: setting it is wrong), so each input pixel is
// fetched once per Cin block instead of kh*kw times.  The single MMA-issuing thread round-robins the T tiles of
// a group, i.e. T independent accumulation chains are in flight; two TMEM buffers of T accumulators let the
// epilogue (8 warps) of group i overlap the MMAs of group i+1.
constexpr int kHaloEpiWarps = 16;
constexpr int kHaloThreads = 64 + 32 * kHaloEpiWarps;   // warp 0 TMA, warp 1 MMA, warps 2..17 epilogue
constexpr int kMaxGroup = 8;

struct HaloArgs {
  int kh, kw, pad_h, pad_w;
  int cin_blocks, block_k;
  int P, Ht, Wv;                  // slots per tile row, tile rows (P * Ht == 128), valid slots per row (P - kw + 1)
  int tiles_w, tiles_h;           // per image
  int Hout, Wout, n_images;
  int block_n, n_blocks, tmem_cols, T, nbuf, stages;
  int n_split;                    // epilogue: column ranges per tile (block_n / n_split columns each, a multiple of 16)
  int out_cstride, out_coff, relu;
  uint32_t idesc, layout_type, sbo_bytes;
  uint32_t a_copy_bytes, a_stage, b_tile, b_total_bytes;
  uint32_t a_res_off, idesc_cat;  // precision 1: residual plane of a halo stage; instruction descriptor of N = 2 block_n
  __half* out;
  __half* out_res;
  const float* bias;
  long long* trace;   // optional timeline of CTA 0: [group][8] clock64 stamps (development aid)
};

#define HALO_TRACE(grp_i, ev) do { if (p.trace && blockIdx.x == 0 && (grp_i) < 64) p.trace[(grp_i) * 8 + (ev)] = clock64(); } while (0)

// kSplit (precision 1, split-fp16 x3): every weight tile is followed by its residual tile, every halo stage holds the main and the
// residual plane, a tile's accumulators are the column pair [D0 | D1]:  [D0 | D1] += A_main * [B_main ; B_res]  (one instruction,
// N = 2 block_n) and  D1 += A_res * B_main.
template <bool kSplit>
__global__ void __launch_bounds__(kHaloThreads, 1)
conv_halo_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const __grid_constant__ CUtensorMap map_a_res,
                 const __grid_constant__ CUtensorMap map_b_res, const HaloArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic (not an integer round trip): ptxas keeps the shared address space -> LDS / STS, not generic LD / ST
  const int taps = p.kh * p.kw;
  constexpr uint32_t kPlanes = kSplit ? 2u : 1u;
  const uint32_t b_slot = kPlanes * p.b_tile;                       // one (Cin block, tap): the filter tile [+ its residual tile]
  uint8_t* smem_b = smem;                                           // [cin_blocks][taps][planes][block_n][block_k]
  uint8_t* smem_a = smem + (size_t)p.cin_blocks * taps * b_slot;    // [stages][planes][halo pixels][block_k]
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_a + (size_t)p.stages * p.a_stage);
  uint64_t* a_full = bars;                              // [kMaxStages * 2]
  uint64_t* a_empty = bars + 2 * kMaxStages;
  uint64_t* b_full = bars + 4 * kMaxStages;
  uint64_t* tmem_full = bars + 4 * kMaxStages + 1;    // [2]
  uint64_t* tmem_empty = bars + 4 * kMaxStages + 3;   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4 * kMaxStages + 5);
  float* s_bias = reinterpret_cast<float*>(bars + 4 * kMaxStages + 6);   // [block_n]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nb = blockIdx.x % p.n_blocks;
  const int g = blockIdx.x / p.n_blocks, G = gridDim.x / p.n_blocks;
  for (int i = threadIdx.x; i < p.block_n; i += kHaloThreads) s_bias[i] = p.bias[nb * p.block_n + i];
  const int tiles_per_image = p.tiles_w * p.tiles_h;
  const int total_tiles = p.n_images * tiles_per_image;
  const int T = p.T;
  // CTA g owns tile groups g, g + G, ...; group j holds tiles j*T .. j*T + T-1 (clamped to the last tile: the
  // duplicates recompute and re-store identical values, which keeps every barrier protocol uniform).
  const int total_groups = (total_tiles + T - 1) / T;
  const uint32_t row_bytes = (uint32_t)p.block_k * 2u;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&map_a);
    prefetch_tmap(&map_b);
    if constexpr (kSplit) { prefetch_tmap(&map_a_res); prefetch_tmap(&map_b_res); }
    for (int s = 0; s < p.stages; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
    mbar_init(b_full, 1);
    for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], 32 * kHaloEpiWarps); }
    fence_barrier_init();
  } else if (warp == 1) {
    tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    {
      // ===== TMA producer (whole warp, one elected lane issues): weights once, then one halo per (tile, Cin block) =====
      if (elect_one()) {
        mbar_arrive_expect_tx(b_full, kPlanes * p.b_total_bytes);
        for (int cb = 0; cb < p.cin_blocks; ++cb)
          for (int t = 0; t < taps; ++t) {
            tma_load_3d(smem_b + (size_t)(cb * taps + t) * b_slot, &map_b, b_full, cb * p.block_k, nb * p.block_n, t);
            if constexpr (kSplit) tma_load_3d(smem_b + (size_t)(cb * taps + t) * b_slot + p.b_tile, &map_b_res, b_full, cb * p.block_k, nb * p.block_n, t);
          }
      }
      __syncwarp();
      int st = 0;
      uint32_t ph = 0;
      for (int grp = g; grp < total_groups; grp += G) {
        for (int cb = 0; cb < p.cin_blocks; ++cb) {
          for (int t = 0; t < T; ++t) {
            const int tile = min(grp * T + t, total_tiles - 1);
            const int n = tile / tiles_per_image;
            const int rem = tile - n * tiles_per_image;
            const int th = rem / p.tiles_w, tw = rem - th * p.tiles_w;
            mbar_wait(&a_empty[st], ph ^ 1);
            if (elect_one()) {
              mbar_arrive_expect_tx(&a_full[st], kPlanes * p.a_copy_bytes);
              tma_load_4d(smem_a + (size_t)st * p.a_stage, &map_a, &a_full[st], cb * p.block_k, tw * p.Wv - p.pad_w, th * p.Ht - p.pad_h, n);
              if constexpr (kSplit)
                tma_load_4d(smem_a + (size_t)st * p.a_stage + p.a_res_off, &map_a_res, &a_full[st], cb * p.block_k, tw * p.Wv - p.pad_w, th * p.Ht - p.pad_h, n);
            }
            __syncwarp();
            if (++st == p.stages) { st = 0; ph ^= 1; }
          }
        }
        if (lane == 0) HALO_TRACE((grp - g) / G, 1);
      }
    }
  } else if (warp == 1) {
    {
      // ===== MMA issuer (whole warp, one elected lane issues): T accumulation chains in flight =====
      mbar_wait(b_full, 0);
      tc_fence_after();
      const int mma_per_kb = p.block_k / 16;
      const uint32_t hi = desc_hi(p.sbo_bytes, p.layout_type), idesc = p.idesc;
      const uint32_t a_lo0 = desc_lo(smem_u32(smem_a)), b_lo0 = desc_lo(smem_u32(smem_b));
      const uint32_t a_stage_inc = p.a_stage >> 4, a_row_inc = ((uint32_t)p.P * row_bytes) >> 4, a_px_inc = row_bytes >> 4;
      const uint32_t b_tile_inc = b_slot >> 4, a_res_inc = p.a_res_off >> 4;
      const int stages = p.stages, kh = p.kh, kw = p.kw, cin_blocks = p.cin_blocks;
      const uint32_t block_n = kPlanes * (uint32_t)p.block_n;     // TMEM columns of one tile's accumulator(s)
      const int nbuf = p.nbuf;
      int st = 0, buf = 0;
      uint32_t ph = 0, buf_ph = 0;
      for (int grp = g; grp < total_groups; grp += G) {
        mbar_wait(&tmem_empty[buf], buf_ph ^ 1);   // the epilogue has drained this buffer of T accumulators
        if (lane == 0) HALO_TRACE((grp - g) / G, 2);
        tc_fence_after();
        const uint32_t d0 = tmem_base + (uint32_t)buf * (uint32_t)T * block_n;
        const uint32_t d1 = d0 + block_n, d2 = d1 + block_n, d3 = d2 + block_n, d4 = d3 + block_n, d5 = d4 + block_n, d6 = d5 + block_n,
                       d7 = d6 + block_n;
        uint32_t accum = 0, b_lo = b_lo0;
        for (int cb = 0; cb < cin_blocks; ++cb) {
          uint32_t a_lo_t[kMaxGroup];
          int st_t = st;
          uint32_t ph_t = ph;
#pragma unroll
          for (int t = 0; t < kMaxGroup; ++t) {
            a_lo_t[t] = 0;
            if (t < T) {
              mbar_wait(&a_full[st_t], ph_t);
              a_lo_t[t] = a_lo0 + (uint32_t)st_t * a_stage_inc;
              if (++st_t == stages) { st_t = 0; ph_t ^= 1; }
            }
          }
          if (cb == 0 && lane == 0) HALO_TRACE((grp - g) / G, 3);
          tc_fence_after();
          if (elect_one()) {
          uint32_t off_r = 0, bl = b_lo, acm = accum;     // the elected lane's working copies: the warp's loop state changes below, for all lanes
          for (int r = 0; r < kh; ++r) {
            uint32_t off = off_r;
            for (int s = 0; s < kw; ++s) {
              for (int k = 0; k < mma_per_kb; ++k) {
                const uint32_t ao = off + 2 * k, bo = bl + 2 * k, ac = acm | (uint32_t)(k != 0);
                // straight-line round-robin over the T accumulators: consecutive MMAs never depend on each other
                if constexpr (kSplit) {
#pragma unroll
                  for (int t = 0; t < kMaxGroup; ++t)
                    if (t < T) {
                      umma_f16_lohi(d0 + (uint32_t)t * block_n, a_lo_t[t] + ao, bo, hi, p.idesc_cat, ac);                            // [D0 | D1] += A_main * [B_main ; B_res]
                      umma_f16_lohi(d0 + (uint32_t)t * block_n + (uint32_t)p.block_n, a_lo_t[t] + a_res_inc + ao, bo, hi, idesc, 1u);   // D1 += A_res * B_main
                    }
                } else if (T == 8) {
                  umma_f16_lohi(d0, a_lo_t[0] + ao, bo, hi, idesc, ac);
                  umma_f16_lohi(d1, a_lo_t[1] + ao, bo, hi, idesc, ac);
                  umma_f16_lohi(d2, a_lo_t[2] + ao, bo, hi, idesc, ac);
                  umma_f16_lohi(d3, a_lo_t[3] + ao, bo, hi, idesc, ac);
                  umma_f16_lohi(d4, a_lo_t[4] + ao, bo, hi, idesc, ac);
                  umma_f16_lohi(d5, a_lo_t[5] + ao, bo, hi, idesc, ac);
                  umma_f16_lohi(d6, a_lo_t[6] + ao, bo, hi, idesc, ac);
                  umma_f16_lohi(d7, a_lo_t[7] + ao, bo, hi, idesc, ac);
                } else if (T == 4) {
                  umma_f16_lohi(d0, a_lo_t[0] + ao, bo, hi, idesc, ac);
                  umma_f16_lohi(d1, a_lo_t[1] + ao, bo, hi, idesc, ac);
                  umma_f16_lohi(d2, a_lo_t[2] + ao, bo, hi, idesc, ac);
                  umma_f16_lohi(d3, a_lo_t[3] + ao, bo, hi, idesc, ac);
                } else {
#pragma unroll
                  for (int t = 0; t < kMaxGroup; ++t)
                    if (t < T) umma_f16_lohi(d0 + (uint32_t)t * block_n, a_lo_t[t] + ao, bo, hi, idesc, ac);
                }
              }
              acm = 1;
              off += a_px_inc;
              bl += b_tile_inc;
            }
            off_r += a_row_inc;
          }
          {
            int st_c = st;
            for (int t = 0; t < T; ++t) {
              umma_commit(&a_empty[st_c]);
              if (++st_c == stages) st_c = 0;
            }
          }
          }
          __syncwarp();
          accum = 1;
          b_lo += (uint32_t)(kh * kw) * b_tile_inc;
          for (int t = 0; t < T; ++t)
            if (++st == stages) { st = 0; ph ^= 1; }
        }
        if (elect_one()) umma_commit(&tmem_full[buf]);
        __syncwarp();
        if (lane == 0) HALO_TRACE((grp - g) / G, 4);
        if (nbuf == 2) { buf ^= 1; if (buf == 0) buf_ph ^= 1; }
        else buf_ph ^= 1;
      }
    }
  } else {
    // ===== epilogue: 16 warps; a warp may only touch the TMEM lane quarter (warp % 4); the 4 warps of a quarter split the
    // tiles of the group ((t & 3) == sub).  Many warps because the per-row work is a long dependent chain (TMEM load ->
    // bias -> ReLU -> pack -> store) that only thread-level parallelism hides.
    const int e = warp - 2;
    const int q = warp & 3;
    const int half = e >> 2;   // 0..3
    const int row = q * 32 + lane;
    const int hh = row / p.P, slot = row - hh * p.P;
    int buf = 0;
    uint32_t buf_ph = 0;
    for (int grp = g; grp < total_groups; grp += G) {
      mbar_wait(&tmem_full[buf], buf_ph);
      if (threadIdx.x == 64) HALO_TRACE((grp - g) / G, 5);
      tc_fence_after();
      const int n_split = p.n_split, cols = p.block_n / n_split;
      for (int u = half; u < T * n_split; u += kHaloEpiWarps / 4) {
        const int t = u / n_split, c0 = (u - t * n_split) * cols;
        const int tile = min(grp * T + t, total_tiles - 1);
        const int n = tile / tiles_per_image;
        const int rem = tile - n * tiles_per_image;
        const int th = rem / p.tiles_w, tw = rem - th * p.tiles_w;
        const int w = tw * p.Wv + slot, h = th * p.Ht + hh;
        const bool valid = (slot < p.Wv) && (w < p.Wout) && (h < p.Hout);
        __half* dst = p.out + ((size_t)((size_t)n * p.Hout + h) * p.Wout + w) * p.out_cstride + p.out_coff + nb * p.block_n + c0;
        const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)((buf * T + t) * (int)kPlanes * p.block_n + c0);
        if constexpr (kSplit) epilogue_row_split2(tacc, tacc + (uint32_t)p.block_n, cols, s_bias + c0, dst, p.out_res + (dst - p.out), valid, p.relu);
        else epilogue_row(tacc, cols, s_bias + c0, dst, valid, p.relu);
      }
      tc_fence_before();
      mbar_arrive(&tmem_empty[buf]);
      if (threadIdx.x == 64) HALO_TRACE((grp - g) / G, 6);
      if (p.nbuf == 2) { buf ^= 1; if (buf == 0) buf_ph ^= 1; }
      else buf_ph ^= 1;
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

// ---------------------------------------------------------------------------------------------
// Row-streaming 3x3 convolution with the kernel rows stacked along N  (conv2, conv3 [+ max pool p1] of the stem)
// ---------------------------------------------------------------------------------------------
// What bounds the narrow stem layers on the kernels above: an M = 128 SS-mode MMA keeps the tensor pipe busy for about
// 64 + N/2 clocks (the 4 KB A tile is read from shared memory at 64 B per clock whatever N is), so N = 32 / 64 runs at
// 20 / 33 % of the pipe's rate (measured: conv2 61 % pipe-busy at 12 % of the math rate).  Here N is made 3x wider without
// any extra arithmetic: ONE input row (128 pixel slots x Cin, one TMA box, fetched exactly once) is multiplied by the filters
// of all three kernel rows at once, B = [3 kw taps x Cin] x [3 kernel rows x Cout], and the three column blocks of the result
// accumulate into the TMEM accumulators of three DIFFERENT output rows (input row j adds to output rows j, j-1, j-2).  The
// accumulators of a stream of rows live in a ring of three column slots; which kernel row lands in which slot rotates with
// the step, and the rotation is free: the filter tile is stored as five row blocks [r2 r1 r0 r2 r1] and the B descriptor
// starts at block 2 - (step mod 3).  Per input row: 3 x (Cin / 16) MMAs of N = 3 Cout (conv2: 6 x (64 + 48) = 672 clocks instead
// of 18 x 80 = 1440; conv3: 960 instead of 1728).  An accumulator slot is complete two steps after it was opened; the epilogue
// drains it, stores zeros back (every MMA accumulates) and hands it back.  MMA(t + 1) depends on drain(t), so a CTA runs TWO
// independent streams (two images) that fill each other's bubbles.  One CTA per SM; each stream walks whole images, so rows
// never cross CTAs and the 3x3 / stride-2 max pool that follows conv3 is fused: the epilogue thread that owns pixel column w
// keeps the running vertical maximum in registers (fp16 max is exact), every second row goes through a shared-memory row
// for the horizontal 3-max and leaves as coalesced 16-byte stores - conv3's output (2.7 GB per 4096 images) is never written.
constexpr int kRowsThreads = 320;        // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue of stream 0, warps 6-9 of stream 1
constexpr int kRowsRing = 4;             // input-row buffers per stream

struct RowsArgs {
  int cin, cout;                 // stored input channels (32 or 64), output channels (3 * cout <= 256)
  int J;                         // input rows streamed per image = Hin + 2 * pad
  int pad, Hout, Wout, n_images;
  int pool;                      // 1: out = maxpool3x3/2(relu(conv + b)), [n][Hp][Wp][out_cstride]; 0: [n][Hout][Wout][out_cstride]
  int Hp, Wp;
  int out_cstride, out_coff;
  uint32_t idesc, layout_type, sbo_bytes, row_bytes;
  uint32_t b_blk_bytes, b_tap_bytes, a_buf_bytes;
  __half* out;
  const float* bias;
  long long* trace;              // optional clock64 timeline of CTA 0, stream 0: [step][8] (DVB_CNN_TRACE; development aid)
};
#define ROWS_TRACE(step, ev) do { if (p.trace && blockIdx.x == 0 && (step) < 48) p.trace[(step) * 8 + (ev)] = clock64(); } while (0)

__device__ __forceinline__ void tmem_st32_zero(uint32_t taddr) {
  const uint32_t z = 0u;
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, "
      "%1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1, %1};" ::"r"(taddr), "r"(z)
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {   // immediate barrier ids: a register id makes ptxas reserve all 16 barriers
  (void)nthreads;
  if (id == 1) asm volatile("bar.sync 1, 128;" ::: "memory");
  else asm volatile("bar.sync 2, 128;" ::: "memory");
}

template <bool kPool>      // two instantiations: the plain one (conv2) does not carry the pooling state's registers
__global__ void __launch_bounds__(kRowsThreads, 1)
conv_rows_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b, const RowsArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic (not an integer round trip): ptxas keeps the shared address space -> LDS / STS, not generic LD / ST
  uint8_t* smem_b = smem;                                                  // [3 taps][5 blocks][cout rows][cin]
  uint8_t* smem_a = smem_b + 3 * p.b_tap_bytes;                            // [2 streams][kRowsRing][128 slots][cin]
  uint8_t* smem_row = smem_a + 2 * kRowsRing * p.a_buf_bytes;              // [2 streams][128 pixels][cout] fp16, 16-byte chunks XOR-swizzled
  const uint32_t row_stage_bytes = 128u * (uint32_t)p.cout * 2u;            // exchange slots of the pooled-row emit live here
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem_row + 2 * row_stage_bytes);
  uint64_t* in_full = bars;                          // [2][kRowsRing]
  uint64_t* in_empty = bars + 2 * kRowsRing;         // [2][kRowsRing]
  uint64_t* acc_done = bars + 4 * kRowsRing;         // [2]
  uint64_t* acc_free = bars + 4 * kRowsRing + 2;     // [2]
  uint64_t* b_full = bars + 4 * kRowsRing + 4;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 4 * kRowsRing + 5);
  float* s_bias = reinterpret_cast<float*>(bars + 4 * kRowsRing + 6);      // [cout]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int i = threadIdx.x; i < p.cout; i += kRowsThreads) s_bias[i] = p.bias[i];
  // images of this CTA: blockIdx.x, + gridDim.x, ...; stream st takes every second one of them
  const int G = gridDim.x;
  const int cnt = (p.n_images - (int)blockIdx.x + G - 1) / G;
  const int cnt_st[2] = {(cnt + 1) >> 1, cnt >> 1};
  const int steps_st[2] = {cnt_st[0] * p.J, cnt_st[1] * p.J};
  const int steps_max = steps_st[0];                 // stream 0 never has fewer images than stream 1
  const int ncol = 3 * p.cout;                       // accumulator columns of one stream (ring of three slots)

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&map_a);
    prefetch_tmap(&map_b);
    for (int i = 0; i < 2 * kRowsRing; ++i) { mbar_init(&in_full[i], 1); mbar_init(&in_empty[i], 1); }
    for (int st = 0; st < 2; ++st) { mbar_init(&acc_done[st], 1); mbar_init(&acc_free[st], 128); }
    mbar_init(b_full, 1);
    fence_barrier_init();
  } else if (warp == 1) {
    tmem_alloc(tmem_slot, (uint32_t)TmemColsDev(2 * ncol));
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    {
      // ===== TMA producer (whole warp, one elected lane issues): the filter tile once, then one input row per (stream, step) =====
      if (elect_one()) {
        mbar_arrive_expect_tx(b_full, 15u * p.b_blk_bytes);
        for (int s = 0; s < 3; ++s)
          for (int blk = 0; blk < 5; ++blk)
            tma_load_3d(smem_b + s * p.b_tap_bytes + blk * p.b_blk_bytes, &map_b, b_full, 0, blk * p.cout, s);
      }
      __syncwarp();
      int rb[2] = {0, 0}, j[2] = {0, 0}, img[2] = {(int)blockIdx.x, (int)blockIdx.x + G};
      uint32_t rph[2] = {0, 0};
      for (int t = 0; t < steps_max; ++t) {
#pragma unroll
        for (int st = 0; st < 2; ++st) {
          if (t >= steps_st[st]) continue;
          uint64_t* full = &in_full[st * kRowsRing + rb[st]];
          mbar_wait(&in_empty[st * kRowsRing + rb[st]], rph[st] ^ 1);
          if (elect_one()) {
            mbar_arrive_expect_tx(full, 128u * p.row_bytes);
            tma_load_4d(smem_a + (size_t)(st * kRowsRing + rb[st]) * p.a_buf_bytes, &map_a, full, 0, -p.pad, j[st] - p.pad, img[st]);
          }
          __syncwarp();
          if (++rb[st] == kRowsRing) { rb[st] = 0; rph[st] ^= 1; }
          if (++j[st] == p.J) { j[st] = 0; img[st] += 2 * G; }
        }
      }
    }
  } else if (warp == 1) {
    {
      // ===== MMA issuer (whole warp, one elected lane issues): per (stream, step) 3 taps x cin/16 MMAs of N = 3 cout into the stream's ring =====
      mbar_wait(b_full, 0);
      tc_fence_after();
      const int kper = p.cin >> 4;
      const uint32_t hi = desc_hi(p.sbo_bytes, p.layout_type), idesc = p.idesc;
      const uint32_t a_lo0 = desc_lo(smem_u32(smem_a)), b_lo0 = desc_lo(smem_u32(smem_b));
      const uint32_t a_buf_inc = p.a_buf_bytes >> 4, a_px_inc = p.row_bytes >> 4, b_blk_inc = p.b_blk_bytes >> 4, b_tap_inc = p.b_tap_bytes >> 4;
      int rb[2] = {0, 0};
      uint32_t rph[2] = {0, 0};
      int t3 = 0;                                    // t mod 3
      for (int t = 0; t < steps_max; ++t) {
#pragma unroll
        for (int st = 0; st < 2; ++st) {
          if (t >= steps_st[st]) continue;
          mbar_wait(&acc_free[st], (uint32_t)t & 1u);               // the slot this step opens has been drained and zeroed
          mbar_wait(&in_full[st * kRowsRing + rb[st]], rph[st]);
          tc_fence_after();
          if (st == 0 && lane == 0) ROWS_TRACE(t, 0);
          const uint32_t d = tmem_base + (uint32_t)(st * ncol);
          const uint32_t a_lo = a_lo0 + (uint32_t)(st * kRowsRing + rb[st]) * a_buf_inc;
          const uint32_t b_lo = b_lo0 + (uint32_t)(2 - t3) * b_blk_inc;
          if (elect_one()) {
            if (kper == 2) {
#pragma unroll
              for (int s = 0; s < 3; ++s) {
                umma_f16_lohi(d, a_lo + (uint32_t)s * a_px_inc, b_lo + (uint32_t)s * b_tap_inc, hi, idesc, 1u);
                umma_f16_lohi(d, a_lo + (uint32_t)s * a_px_inc + 2u, b_lo + (uint32_t)s * b_tap_inc + 2u, hi, idesc, 1u);
              }
            } else {
              for (int s = 0; s < 3; ++s)
                for (int k = 0; k < kper; ++k)
                  umma_f16_lohi(d, a_lo + (uint32_t)s * a_px_inc + 2u * k, b_lo + (uint32_t)s * b_tap_inc + 2u * k, hi, idesc, 1u);
            }
            umma_commit(&in_empty[st * kRowsRing + rb[st]]);
            umma_commit(&acc_done[st]);
          }
          __syncwarp();
          if (st == 0 && lane == 0) ROWS_TRACE(t, 1);
          if (++rb[st] == kRowsRing) { rb[st] = 0; rph[st] ^= 1; }
        }
        if (++t3 == 3) t3 = 0;
      }
    }
  } else {
    // ===== epilogue of stream st: 4 warps = 4 TMEM lane quarters; thread = pixel column w of every row of the stream =====
    const int st = (warp - 2) >> 2;
    const int q = warp & 3;
    const int w = q * 32 + lane;
    const int tid = ((warp - 2) & 3) * 32 + lane;     // 0..127 inside the stream's epilogue group
    const int bar_id = 1 + st;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(st * ncol);
    uint8_t* stage = smem_row + st * row_stage_bytes;
    const int nch = p.cout >> 3;                      // 16-byte chunks per pixel: 4 (cout 32) or 8 (cout 64)
    // every accumulator column starts at zero
    for (int c = 0; c < ncol; c += 32) tmem_st32_zero(t_lane + c);
    tmem_st_wait();
    tc_fence_before();
    mbar_arrive(&acc_free[st]);
    uint32_t cur[kPool ? 32 : 1];                     // running vertical maximum (pool mode), packed half2, cout <= 64
#pragma unroll
    for (int i = 0; i < (kPool ? 32 : 1); ++i) cur[i] = 0u;
    int j = 0, img = (int)blockIdx.x + st * G, slot = 1;   // slot drained at step t = (t + 1) mod 3
    for (int t = 0; t < steps_st[st]; ++t) {
      mbar_wait(&acc_done[st], (uint32_t)t & 1u);
      tc_fence_after();
      if (st == 0 && tid == 0) ROWS_TRACE(t, 2);
      const bool row_valid = j >= 2;
      const int o = j - 2;
      uint32_t hv[32];
#pragma unroll
      for (int cc = 0; cc < 2; ++cc) {
        if (cc * 32 < p.cout) {
          uint32_t v[32];
          tmem_ld32(t_lane + slot * p.cout + cc * 32, v);
          tmem_ld_wait();
          tmem_st32_zero(t_lane + slot * p.cout + cc * 32);
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            const float x0 = fmaxf(__uint_as_float(v[2 * i]) + s_bias[cc * 32 + 2 * i], 0.f);
            const float x1 = fmaxf(__uint_as_float(v[2 * i + 1]) + s_bias[cc * 32 + 2 * i + 1], 0.f);
            const __half2 h = __floats2half2_rn(x0, x1);
            hv[cc * 16 + i] = *reinterpret_cast<const uint32_t*>(&h);
          }
        }
      }
      tmem_st_wait();
      tc_fence_before();
      if (st == 0 && tid == 0) ROWS_TRACE(t, 3);
      mbar_arrive(&acc_free[st]);                      // the MMAs of step t + 1 may go ahead while this row is stored
      if (row_valid) {
        const int nh = p.cout >> 1;                    // half2 words per pixel
        if constexpr (!kPool) {
          // every thread owns one pixel: cout * 2 contiguous bytes, written straight from its registers (the staging row + two
          // block barriers + copy-out loop this replaces cost ~1600 clocks per row on the critical path - timeline in profiles/)
          if (w < p.Wout) {
            __half* dst = p.out + (((size_t)img * p.Hout + o) * p.Wout + w) * p.out_cstride + p.out_coff;
#pragma unroll
            for (int c = 0; c < 8; ++c)
              if (c < nch) *reinterpret_cast<uint4*>(dst + c * 8) = make_uint4(hv[4 * c], hv[4 * c + 1], hv[4 * c + 2], hv[4 * c + 3]);
          }
        } else {
          // vertical 3-max over rows 2 ph, 2 ph + 1, 2 ph + 2: an even row closes window ph - 1 and opens window ph
          const bool even = (o & 1) == 0;
          const bool emit = even && o >= 2;
          if (emit) {
            // horizontal 3-max over pixels 2 pw, 2 pw + 1, 2 pw + 2 by the thread of pixel 2 pw: its two right-hand neighbours are
            // lanes + 1 and + 2 (shuffles); lane 30's second neighbour is lane 0 of the NEXT warp, handed over through a 128-byte
            // shared-memory slot (double-buffered by emit parity: one block barrier per pooled row)
            const int par = (o >> 1) & 1;
            uint32_t* exch = reinterpret_cast<uint32_t*>(stage) + (par * 4) * 32;     // [parity][warp quarter][32 words]
#pragma unroll
            for (int i = 0; i < 32; ++i) {
              if (i < nh) {
                const __half2 a = *reinterpret_cast<const __half2*>(&cur[i]), b = *reinterpret_cast<const __half2*>(&hv[i]);
                const __half2 r = __hmax2(a, b);
                cur[i] = *reinterpret_cast<const uint32_t*>(&r);      // cur = the finished vertical maximum of pixel w (re-opened from hv below)
              }
            }
            if (lane == 0 && q > 0) {
#pragma unroll
              for (int i = 0; i < 32; i += 4)
                if (i < nh) *reinterpret_cast<uint4*>(exch + (q - 1) * 32 + i) = make_uint4(cur[i], cur[i + 1], cur[i + 2], cur[i + 3]);
            }
            named_bar_sync(bar_id, 128);
            const int ph = (o >> 1) - 1;
            const int pw = w >> 1;
            const bool writer = (lane & 1) == 0 && pw < p.Wp;
            __half* dst = p.out + (((size_t)img * p.Hp + ph) * p.Wp + pw) * p.out_cstride + p.out_coff;
            // (all 8 shuffles of a 16-byte group are issued before the first one is consumed: the first version consumed each shuffle
            //  right away and ran 64 of them back to back at their full latency - 3000 clocks per pooled row in the timeline)
            const bool edge = lane == 30;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              if (c < nch) {
                uint4 nb = make_uint4(0u, 0u, 0u, 0u);                               // post-ReLU values are >= 0: zero is the identity
                if (edge && q < 3) nb = *reinterpret_cast<const uint4*>(exch + q * 32 + 4 * c);
                uint32_t v1[4], v2[4], mx[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) v1[e] = __shfl_down_sync(0xffffffffu, cur[4 * c + e], 1);
#pragma unroll
                for (int e = 0; e < 4; ++e) v2[e] = __shfl_down_sync(0xffffffffu, cur[4 * c + e], 2);
                if (edge) { v2[0] = nb.x; v2[1] = nb.y; v2[2] = nb.z; v2[3] = nb.w; }
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  const __half2 r = __hmax2(*reinterpret_cast<const __half2*>(&cur[4 * c + e]),
                                            __hmax2(*reinterpret_cast<const __half2*>(&v1[e]), *reinterpret_cast<const __half2*>(&v2[e])));
                  mx[e] = *reinterpret_cast<const uint32_t*>(&r);
                }
                if (writer) *reinterpret_cast<uint4*>(dst + c * 8) = make_uint4(mx[0], mx[1], mx[2], mx[3]);
              }
            }
          }
#pragma unroll
          for (int i = 0; i < 32; ++i) {
            if (i < nh) {
              if (even) cur[i] = hv[i];
              else {
                const __half2 a = *reinterpret_cast<const __half2*>(&cur[i]), b = *reinterpret_cast<const __half2*>(&hv[i]);
                const __half2 r = __hmax2(a, b);
                cur[i] = *reinterpret_cast<const uint32_t*>(&r);
              }
            }
          }
        }
      }
      if (st == 0 && tid == 0) ROWS_TRACE(t, 4);
      if (++slot == 3) slot = 0;
      if (++j == p.J) { j = 0; img += 2 * G; }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, (uint32_t)TmemColsDev(2 * ncol));
}

// ---------------------------------------------------------------------------------------------
// Small CUDA-core kernels
// ---------------------------------------------------------------------------------------------

// dv_utils.preprocess_images fused with the im2col of the first convolution (3x3, stride 2, valid):
//   out[n][oh][ow][k] = (x[n][2*oh + r][2*ow + s][c] - 128) / 128   with k = (r*3 + s)*C + c,  k >= 9*C -> 0
// so that conv1 becomes a plain GEMM over K = Kp (64 for the 7-channel WGS image): one contiguous, fully
// used 128-byte row per output pixel instead of nine strided 32-byte TMA boxes.  (x - 128) / 128 is exact
// in fp16 (|x - 128| <= 128, power-of-two divisor).  One thread per (output pixel, 8 consecutive k).
constexpr int kPatchRows = 4;  // output rows per block
__global__ void __launch_bounds__(256) stem_patch_kernel(const uint8_t* __restrict__ in, __half* __restrict__ out, int n_images, int H,
                                                         int W, int C, int Ho, int Wo, int Kp) {
  // One block = kPatchRows full output rows of one image: the 2*rows+1 input rows they touch are staged in shared
  // memory with coalesced 4-byte loads, then every thread emits 16-byte chunks of patches (coalesced stores).
  extern __shared__ __align__(16) uint8_t s_in[];  // [(2*kPatchRows + 1)][row_pitch] then short koff[Kp]
  const int groups = (Ho + kPatchRows - 1) / kPatchRows;
  const int n = blockIdx.x / groups;
  const int oh0 = (blockIdx.x - n * groups) * kPatchRows;
  const int rows = min(kPatchRows, Ho - oh0);
  const int in_rows = 2 * rows + 1;
  const int row_bytes = W * C;
  const int row_pitch = (row_bytes + 3 + 15) & ~15;  // +3: the copy below starts at a 4-byte aligned address
  short* koff = reinterpret_cast<short*>(s_in + (2 * kPatchRows + 1) * row_pitch);
  for (int k = threadIdx.x; k < Kp; k += blockDim.x) {
    const int r = k / (3 * C);
    koff[k] = k < 9 * C ? (short)(r * row_pitch + (k - r * 3 * C)) : (short)-1;   // (s, c) is contiguous in the input row
  }
  // rows are contiguous in global memory: copy [first byte, last byte) with aligned 32-bit loads
  const size_t g0 = ((size_t)n * H + 2 * oh0) * row_bytes;
  for (int r = 0; r < in_rows; ++r) {
    const size_t gb = g0 + (size_t)r * row_bytes;
    const int mis = (int)(gb & 3);                       // shared copy keeps the same misalignment
    const uint32_t* src = reinterpret_cast<const uint32_t*>(in + (gb - mis));
    uint32_t* dstw = reinterpret_cast<uint32_t*>(s_in + r * row_pitch);
    const int nw = (mis + row_bytes + 3) >> 2;
    const size_t total_bytes = (size_t)n_images * H * row_bytes;
    for (int i = threadIdx.x; i < nw; i += blockDim.x) {
      const size_t off = (gb - mis) + 4 * (size_t)i;
      uint32_t wv;
      if (off + 4 <= total_bytes) {
        wv = __ldg(src + i);
      } else {  // never read past the end of the caller's buffer
        wv = 0;
        for (int bb = 0; bb < 4; ++bb)
          if (off + bb < total_bytes) wv |= (uint32_t)in[off + bb] << (8 * bb);
      }
      dstw[i] = wv;
    }
  }
  __syncthreads();
  // one thread per output pixel: 3 segments of 3*C contiguous input bytes -> Kp halves = Kp/8 16-byte stores
  const int kvec = Kp / 8;
  const uint4* koff4 = reinterpret_cast<const uint4*>(koff);
  for (int t = threadIdx.x; t < rows * Wo; t += blockDim.x) {
    const int orow = t / Wo, px = t - orow * Wo;
    const size_t gb = g0 + (size_t)(2 * orow) * row_bytes;
    const int mis0 = (int)(gb & 3), mis1 = (int)((gb + row_bytes) & 3), mis2 = (int)((gb + 2 * (size_t)row_bytes) & 3);
    // koff[k] = r * row_pitch + j; the three input rows of this pixel start at different 4-byte phases
    const uint8_t* base = s_in + (2 * orow) * row_pitch + 2 * px * C;
    const int adj[3] = {mis0, mis1, mis2};
    __half* dst = out + (((size_t)n * Ho + oh0 + orow) * Wo + px) * Kp;
    for (int kv = 0; kv < kvec; ++kv) {
      const uint4 o4 = koff4[kv];
      const uint32_t ow[4] = {o4.x, o4.y, o4.z, o4.w};
      uint32_t pk[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float v[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int o = (int)(short)((ow[j] >> (16 * e)) & 0xFFFFu);
          float x = 0.f;
          if (o >= 0) {
            const int r = o >= 2 * row_pitch ? 2 : (o >= row_pitch ? 1 : 0);
            x = ((float)base[o + adj[r]] - 128.f) * (1.f / 128.f);
          }
          v[e] = x;
        }
        __half2 hh = __floats2half2_rn(v[0], v[1]);
        pk[j] = *reinterpret_cast<uint32_t*>(&hh);
      }
      *reinterpret_cast<uint4*>(dst + kv * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Fused stem: preprocess + im2col + conv1 (3x3 stride 2 valid, C = 7) straight from the uint8 image
// ---------------------------------------------------------------------------------------------
// The patch route (stem_patch_kernel -> GEMM) writes and re-reads a [N][Ho][Wo][64] fp16 patch tensor (1.4 GB per 2048
// images) that exists only to make conv1 TMA-loadable.  Here the SM builds the A tile itself: one tile = 128 output
// pixels of one output row.  Phase 1 (all threads) streams the three input rows the tile touches from global memory,
// converts bytes to fp16 with the exact (x - 128) / 128 (magic-number trick: 0x6400 | x = 1024 + x, one HFMA2 per pair)
// and leaves them in shared memory as halves; phase 2 (two threads per pixel) assembles each pixel's 63-element patch
// (3 runs of 21 contiguous halves; the middle run lands on an odd half offset -> one funnel shift per word) and stores
// it as the 128-byte row of a canonical 128B-swizzled K-major tile; one thread issues the 4 MMAs (K = 64, N = 32);
// warps 0-3 run the bias + ReLU epilogue from TMEM.  Persistent CTAs, several per SM, hide each other's phases.
constexpr int kStemThreads = 256;
constexpr int kStemC = 7;
constexpr int kStemSeg = 3 * kStemC;   // 21 contiguous (s, c) values per tap row

struct StemArgs {
  const uint8_t* in; __half* out; const float* bias; const __half* w;   // w: [cout][64], k = (r*3 + s)*7 + c
  int n_images, H, W, Ho, Wo, cout, out_cstride, tiles_w;
  long long total_bytes;
  uint32_t idesc;
  int h_pitch;   // halves per staged input row (multiple of 8)
};

__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src, int src_bytes) {   // zero-fills past src_bytes
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst_smem)), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

constexpr int kStemRawPitch = 1840;   // bytes per staged raw input row segment (>= 15 + 1799 + 4 rounded up to 16)

// kPipe: the tile loop as a software pipeline - the MMAs of tile i run while tile i + 1 is converted, and the epilogue of tile i (all
// eight warps, two per TMEM lane quarter) sits between the conversion and the patch assembly of tile i + 1: two accumulators in TMEM,
// three block barriers per tile instead of four, no warp waits for the tensor pipe's latency.
template <bool kPipe>
#ifndef DVB_STEM_MIN_BLOCKS
#define DVB_STEM_MIN_BLOCKS 4
#endif
__global__ void __launch_bounds__(kStemThreads, DVB_STEM_MIN_BLOCKS) stem_conv1_kernel(const StemArgs p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // pointer arithmetic (not an integer round trip): ptxas keeps the shared address space -> LDS / STS, not generic LD / ST
  uint8_t* sA = smem;                         // 128 rows x 128 B, 128B swizzle
  uint8_t* sB = smem + 16384;                 // cout rows x 128 B, 128B swizzle (cout <= 32 -> 4 KB)
  __half* sH = reinterpret_cast<__half*>(smem + 16384 + 4096);   // [3][h_pitch]
  uint8_t* sRaw = reinterpret_cast<uint8_t*>(sH + 3 * p.h_pitch);   // [2][3][kStemRawPitch] raw uint8 row segments (cp.async ring)
  uint64_t* mma_done = reinterpret_cast<uint64_t*>(sRaw + 2 * 3 * kStemRawPitch);   // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(mma_done + 2);
  float* s_bias = reinterpret_cast<float*>(mma_done + 4);   // 32 bytes on: the epilogue reads the bias as float4
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid < p.cout) s_bias[tid] = p.bias[tid];
  for (int i = tid; i < p.cout * 8; i += kStemThreads) {   // weights -> swizzled K-major tile
    const int n = i >> 3, j = i & 7;
    *reinterpret_cast<uint4*>(sB + n * 128 + ((j ^ (n & 7)) << 4)) = *reinterpret_cast<const uint4*>(p.w + n * 64 + j * 8);
  }
  if (tid == 0) { mbar_init(&mma_done[0], 1); mbar_init(&mma_done[1], 1); fence_barrier_init(); }
  if (warp == 1) tmem_alloc(tmem_slot, kPipe ? 64 : 32);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int row_bytes = p.W * kStemC;
  const long long total_tiles = (long long)p.n_images * p.Ho * p.tiles_w;
  uint32_t phase = 0;
  const __half2 kScale = __floats2half2_rn(1.f / 128.f, 1.f / 128.f), kBias = __floats2half2_rn(-9.f, -9.f);

  // Asynchronous staging of the raw bytes of one tile (3 row segments) into ring slot `slot` with 16-byte cp.async
  // (source aligned down to 16 bytes; the 0-15 byte misalignment is removed when the bytes are converted): the loads
  // of tile i + 1 are in flight while tile i is converted, assembled, multiplied and written out.
  // Tiles are walked with 32-bit (n, oh, tw) counters - no 64-bit divisions in the loop.
  const int tiles_per_image = p.Ho * p.tiles_w;
  auto decode = [&](int tile, int& n, int& oh, int& tw) {
    n = tile / tiles_per_image;
    const int rem = tile - n * tiles_per_image;
    oh = rem / p.tiles_w;
    tw = rem - oh * p.tiles_w;
  };
  auto stage = [&](int n, int oh, int tw, int slot) {
    const int ow0 = tw * 128;
    const int npx = min(128, p.Wo - ow0);
    const int seg_bytes = (2 * (npx - 1) + 3) * kStemC;
    const long long row0 = ((long long)n * p.H + 2 * oh) * row_bytes + (long long)2 * ow0 * kStemC;
    for (int r = 0; r < 3; ++r) {
      const uint8_t* g = p.in + row0 + (long long)r * row_bytes;
      const int mis = (int)(reinterpret_cast<uintptr_t>(g) & 15);   // alignment of the ABSOLUTE address
      const uint8_t* src = g - mis;
      const int nq = (mis + seg_bytes + 4 + 15) >> 4;            // 16-byte chunks (4 spare bytes for the last funnel shift)
      const long long left = (p.in + p.total_bytes) - src;       // bytes the caller's buffer still holds from `src`
      const int full = (int)min((long long)nq, left >> 4);       // chunks that lie completely inside the buffer
      uint8_t* dst = sRaw + (slot * 3 + r) * kStemRawPitch;
      for (int i = tid; i < full; i += kStemThreads) cp_async16(dst + 16 * i, src + 16 * i, 16);
      if (full < nq && tid == 0) {                               // last row of the last image: never read past the buffer
        const int tail = (int)(left - 16LL * full);
        cp_async16(dst + 16 * full, tail > 0 ? src + 16 * full : src, tail > 0 ? tail : 0);
      }
    }
    cp_async_commit();
  };

  // epilogue of one tile: kPipe - all eight warps, two per TMEM lane quarter, half of the filters each (cout = 32) or the first four (cout = 16)
  auto drain = [&](int en, int eoh, int etw, int buf) {
    const int q = warp & 3, hf = warp >> 2;
    const int cw = p.cout >= 32 ? p.cout / 2 : p.cout;
    if (hf == 1 && p.cout < 32) return;
    const int eow0 = etw * 128;
    const int m = q * 32 + lane;
    const bool valid = m < min(128, p.Wo - eow0);
    __half* dst = p.out + (((size_t)en * p.Ho + eoh) * p.Wo + eow0 + m) * p.out_cstride + hf * cw;
    epilogue_row(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * 32 + hf * cw), cw, s_bias + hf * cw, dst, valid, 1);
  };
  const int total = (int)total_tiles;
  int tile = blockIdx.x;
  int slot = 0;
  int n, oh, tw;
  int pn = 0, poh = 0, ptw = 0, pbuf = 0, buf = 0;   // kPipe: the tile whose MMAs are in flight
  bool have_prev = false;
  uint32_t done_ph0 = 0u, done_ph1 = 0u;
  decode(min(tile, total - 1), n, oh, tw);
  if (tile < total) stage(n, oh, tw, 0);
  for (; tile < total; tile += gridDim.x, slot ^= 1) {
    const int ow0 = tw * 128;
    const int npx = min(128, p.Wo - ow0);
    const int seg_bytes = (2 * (npx - 1) + 3) * kStemC;   // input bytes of one row this tile touches
    int n2 = n, oh2 = oh, tw2 = tw;
    if (tile + (int)gridDim.x < total) { decode(tile + gridDim.x, n2, oh2, tw2); stage(n2, oh2, tw2, slot ^ 1); cp_async_wait<1>(); }
    else cp_async_wait<0>();
    __syncthreads();
    // ---- phase 1: raw bytes -> fp16 (x - 128) / 128 in shared memory
    const long long row0 = ((long long)n * p.H + 2 * oh) * row_bytes + (long long)2 * ow0 * kStemC;
    for (int r = 0; r < 3; ++r) {
      const int mis = (int)(reinterpret_cast<uintptr_t>(p.in + row0 + (long long)r * row_bytes) & 15);
      const uint32_t* src = reinterpret_cast<const uint32_t*>(sRaw + (slot * 3 + r) * kStemRawPitch) + (mis >> 2);
      const int sh = 8 * (mis & 3);
      const int nw = (seg_bytes + 3) >> 2;
      uint2* dst = reinterpret_cast<uint2*>(sH + r * p.h_pitch);
      for (int i = tid; i < nw; i += kStemThreads) {
        const uint32_t v = __funnelshift_r(src[i], src[i + 1], sh);     // bytes g0 + 4i .. g0 + 4i + 3
        uint32_t a = __byte_perm(v, 0x64646464u, 0x4140), b = __byte_perm(v, 0x64646464u, 0x4342);
        __half2 ha = __hfma2(*reinterpret_cast<__half2*>(&a), kScale, kBias), hb = __hfma2(*reinterpret_cast<__half2*>(&b), kScale, kBias);
        dst[i] = make_uint2(*reinterpret_cast<uint32_t*>(&ha), *reinterpret_cast<uint32_t*>(&hb));
      }
    }
    if constexpr (kPipe) {
      if (have_prev) {   // the previous tile's MMAs were issued a whole conversion ago: its accumulator is (all but always) complete
        mbar_wait(&mma_done[pbuf], pbuf ? done_ph1 : done_ph0);
        if (pbuf) done_ph1 ^= 1u; else done_ph0 ^= 1u;
        tc_fence_after();
        drain(pn, poh, ptw, pbuf);
        tc_fence_before();
      }
    }
    __syncthreads();   // (kPipe: every warp has seen the previous tile's MMAs retire -> sA may be rewritten)
    // ---- phase 2: patch rows.  Thread (m, hf): output words [16 hf, 16 hf + 16) of row m (lane stride 7 words: conflict-free).
    {
      const int m = tid & 127, hf = tid >> 7;   // warp-uniform halves: warps 0-3 build words 0..15, warps 4-7 words 16..31
      uint32_t ow[16];
      if (m < npx) {
        const uint32_t* W0 = reinterpret_cast<const uint32_t*>(sH) + 7 * m;                       // 14 m halves = 7 m words
        const uint32_t* W1 = reinterpret_cast<const uint32_t*>(sH + p.h_pitch) + 7 * m;
        const uint32_t* W2 = reinterpret_cast<const uint32_t*>(sH + 2 * p.h_pitch) + 7 * m;
        if (hf == 0) {
#pragma unroll
          for (int i = 0; i < 10; ++i) ow[i] = W0[i];
          uint32_t prev = W1[0];
          ow[10] = (W0[10] & 0xFFFFu) | (prev << 16);
#pragma unroll
          for (int i = 11; i < 16; ++i) { const uint32_t nx = W1[i - 10]; ow[i] = __funnelshift_r(prev, nx, 16); prev = nx; }
        } else {
          uint32_t prev = W1[5];
#pragma unroll
          for (int i = 16; i < 21; ++i) { const uint32_t nx = W1[i - 10]; ow[i - 16] = __funnelshift_r(prev, nx, 16); prev = nx; }
#pragma unroll
          for (int i = 21; i < 31; ++i) ow[i - 16] = W2[i - 21];
          ow[15] = W2[10] & 0xFFFFu;
        }
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i) ow[i] = 0u;
      }
      uint8_t* rowp = sA + m * 128;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const int j = hf * 4 + c;
        *reinterpret_cast<uint4*>(rowp + ((j ^ (m & 7)) << 4)) = make_uint4(ow[4 * c], ow[4 * c + 1], ow[4 * c + 2], ow[4 * c + 3]);
      }
    }
    fence_proxy_async();
    __syncthreads();
    // ---- MMA: D[128 x cout] = A[128 x 64] * B[cout x 64]^T
    if (warp == 1) {
      tc_fence_after();
      const uint32_t hi = desc_hi(1024u, 2u), a_lo = desc_lo(smem_u32(sA)), b_lo = desc_lo(smem_u32(sB));
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16_lohi(tmem_base + (uint32_t)(buf * 32), a_lo + 2 * k, b_lo + 2 * k, hi, p.idesc, (uint32_t)(k != 0));
        umma_commit(&mma_done[buf]);
      }
      __syncwarp();
    }
    if constexpr (kPipe) {
      pn = n; poh = oh; ptw = tw; pbuf = buf; have_prev = true;
      buf ^= 1;
      n = n2; oh = oh2; tw = tw2;
      continue;   // no closing barrier: the next iteration's first barrier orders the ring slot, the barrier before its patch assembly orders sA
    }
    // ---- epilogue: warps 0..3 own TMEM lane quarters 0..3
    if (warp < 4) {
      mbar_wait(&mma_done[0], phase);
      tc_fence_after();
      const int m = warp * 32 + lane;
      const bool valid = m < npx;
      __half* dst = p.out + (((size_t)n * p.Ho + oh) * p.Wo + ow0 + m) * p.out_cstride;
      epilogue_row(tmem_base + ((uint32_t)(warp * 32) << 16), p.cout, s_bias, dst, valid, 1);
      tc_fence_before();
    }
    phase ^= 1;
    n = n2; oh = oh2; tw = tw2;
    __syncthreads();   // accumulator drained, sA / sH free for the next tile
  }
  if constexpr (kPipe) {
    if (have_prev) {
      mbar_wait(&mma_done[pbuf], pbuf ? done_ph1 : done_ph0);
      tc_fence_after();
      drain(pn, poh, ptw, pbuf);
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, kPipe ? 64 : 32);
}

// ---------------------------------------------------------------------------------------------
// conv1 as a row-streaming, warp-specialised kernel (WGS geometry: 7 channels, 3x3 stride 2 valid, 32 filters)
// ---------------------------------------------------------------------------------------------
// stem_conv1_kernel above is a bulk-synchronous design: four block barriers per 128-pixel tile (26 % of its stall samples) and
// every input row converted 1.5 times.  Here one CTA per SM streams whole images row by row through a pipeline of warp roles:
//   converters (4 warps, a thread per output pixel)  raw uint8 row (cp.async ring) -> exact (x - 128) / 128 in fp16 -> the K-major
//       A tile of THAT input row: pixel w holds the 21 values (3 kw taps x 7 channels) at bytes [14 w, 14 w + 21) of the row, padded
//       to K = 32 (the three bytes that follow ride along against zero weights); each input row is converted exactly once;
//   MMA warp   input row r adds kernel row r - 2 o to output row o: an even row 2 o' feeds kernel row 0 of output row o' AND kernel
//       row 2 of output row o' - 1 - one MMA pair of N = 64 over both accumulator slots (the filter tile is stored [W0 W2 W0 W1], so the
//       slot order flips with the parity of o' by starting 32 rows later); an odd row feeds kernel row 1 of one slot (N = 32);
//   epilogue (4 warps)  after every even row the finished slot is drained (bias + ReLU -> fp16, 64 contiguous bytes per pixel
//       straight from registers), zeroed and handed back; the odd row in between touches only the other slot, so draining overlaps it.
constexpr int kS1Threads = 32 + 128 + 128;   // warp 0 MMA, warps 1-4 converters, warps 5-8 epilogue
constexpr int kS1RawSlots = 4, kS1RawPitch = 1840, kS1ARing = 4;

struct Stem2Args {
  const uint8_t* in; __half* out; const float* bias; const __half* w;   // w: [128][32] = filter tile rows [W0 | W2 | W0 | W1] x K (s * 7 + c, zero from 21)
  int n_images, H, W, Ho, Wo, out_cstride;
  long long total_bytes;
};

__global__ void __launch_bounds__(kS1Threads, 1) stem_rows_kernel(const Stem2Args p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sA = smem;                                  // [kS1ARing][128 rows x 64 B], 64B swizzle
  uint8_t* sB = smem + kS1ARing * 8192;                // 128 rows x 64 B, 64B swizzle
  uint8_t* sRaw = sB + 8192;                           // [kS1RawSlots][kS1RawPitch]
  uint64_t* bars = reinterpret_cast<uint64_t*>(sRaw + kS1RawSlots * kS1RawPitch);
  uint64_t* a_full = bars;                             // [kS1ARing]  128 converter arrivals
  uint64_t* a_empty = bars + kS1ARing;                 // [kS1ARing]  tcgen05.commit
  uint64_t* acc_done = bars + 2 * kS1ARing;            // commit after every even input row
  uint64_t* acc_free = bars + 2 * kS1ARing + 1;        // 128 epilogue arrivals
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kS1ARing + 2);
  float* s_bias = reinterpret_cast<float*>(bars + 2 * kS1ARing + 4);   // [32], 16-byte aligned (read as float4)
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  if (tid < 32) s_bias[tid] = p.bias[tid];
  for (int i = tid; i < 128 * 4; i += kS1Threads) {    // filter tile -> 64B-swizzled K-major rows
    const int n = i >> 2, j = i & 3;
    *reinterpret_cast<uint4*>(sB + n * 64 + ((j ^ ((n >> 1) & 3)) << 4)) = *reinterpret_cast<const uint4*>(p.w + n * 32 + j * 8);
  }
  if (tid == 0) {
    for (int i = 0; i < kS1ARing; ++i) { mbar_init(&a_full[i], 128); mbar_init(&a_empty[i], 1); }
    mbar_init(acc_done, 1);
    mbar_init(acc_free, 128);
    fence_barrier_init();
  }
  if (warp == 0) tmem_alloc(tmem_slot, 64);
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int G = gridDim.x;
  const int n_img = (p.n_images - (int)blockIdx.x + G - 1) / G;      // images blockIdx.x, + G, ...
  const int rows_per_image = 2 * p.Ho + 1;                           // input rows 0 .. 2 Ho: the last one closes output row Ho - 1
  const int total_rows = n_img * rows_per_image;
  const int row_bytes = p.W * kStemC;

  if (warp == 0) {
    // ===== MMA issuer =====
    const uint32_t hi = desc_hi(512u, 4u);
    const uint32_t a_lo0 = desc_lo(smem_u32(sA)), b_lo0 = desc_lo(smem_u32(sB));
    const uint32_t idesc64 = (1u << 4) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    const uint32_t idesc32 = (1u << 4) | ((uint32_t)(32 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    int slot = 0, r = 0;
    uint32_t ph = 0, even_count = 0;
    for (int R = 0; R < total_rows; ++R) {
      const bool even = (r & 1) == 0;
      const int op = r >> 1;                                        // o' (even rows) / the output row an odd row feeds
      if (even) mbar_wait(acc_free, even_count & 1u);               // completion #even_count: the slot this row opens is drained and zero
      mbar_wait(&a_full[slot], ph);
      tc_fence_after();
      if (elect_one()) {
        const uint32_t a_lo = a_lo0 + (uint32_t)slot * (8192u >> 4);
        if (even) {
          const uint32_t b_lo = b_lo0 + ((op & 1) ? (32u * 64u >> 4) : 0u);            // [W0 W2] or [W2 W0] over slots (0, 1)
          umma_f16_lohi(tmem_base, a_lo, b_lo, hi, idesc64, 1u);
          umma_f16_lohi(tmem_base, a_lo + 2u, b_lo + 2u, hi, idesc64, 1u);
        } else {
          const uint32_t b_lo = b_lo0 + (96u * 64u >> 4);                              // W1
          const uint32_t d = tmem_base + (uint32_t)((op & 1) * 32);
          umma_f16_lohi(d, a_lo, b_lo, hi, idesc32, 1u);
          umma_f16_lohi(d, a_lo + 2u, b_lo + 2u, hi, idesc32, 1u);
        }
        umma_commit(&a_empty[slot]);
        if (even) umma_commit(acc_done);
      }
      __syncwarp();
      if (even) ++even_count;
      if (++slot == kS1ARing) { slot = 0; ph ^= 1; }
      if (++r == rows_per_image) r = 0;
    }
  } else if (warp <= 4) {
    // ===== converters: thread = output pixel w of every input row =====
    const int w = tid - 32;
    const int ctid = w;                                             // 0 .. 127
    const __half2 kScale = __floats2half2_rn(1.f / 128.f, 1.f / 128.f), kBias = __floats2half2_rn(-9.f, -9.f);
    auto stage = [&](int Rr) {                                      // cp.async of input row Rr of this CTA's stream into raw slot Rr & 3
      if (Rr < total_rows) {
        const int li = Rr / rows_per_image, rr = Rr - li * rows_per_image;
        const long long img = (long long)blockIdx.x + (long long)li * G;
        const uint8_t* g = p.in + (img * p.H + rr) * row_bytes;
        const int mis = (int)(reinterpret_cast<uintptr_t>(g) & 15);
        const uint8_t* src = g - mis;
        const int nq = (mis + row_bytes + 15) >> 4;
        const long long left = (p.in + p.total_bytes) - src;
        const int full = (int)min((long long)nq, left >> 4);
        uint8_t* dst = sRaw + (Rr & (kS1RawSlots - 1)) * kS1RawPitch;
        if (ctid < full) cp_async16(dst + 16 * ctid, src + 16 * ctid, 16);
        else if (ctid == full && full < nq) {                       // never read past the caller's buffer
          const int tail = (int)(left - 16LL * full);
          cp_async16(dst + 16 * full, tail > 0 ? src + 16 * full : src, tail > 0 ? tail : 0);
        }
      }
      cp_async_commit();
    };
    stage(0);
    stage(1);
    int slot = 0, r = 0, li = 0;
    uint32_t ph = 0;
    for (int R = 0; R < total_rows; ++R) {
      stage(R + 2);
      cp_async_wait<2>();
      asm volatile("bar.sync 3, 128;" ::: "memory");                // every converter's chunks of row R have landed
      const long long img = (long long)blockIdx.x + (long long)li * G;
      const uint8_t* g = p.in + (img * p.H + r) * row_bytes;
      const int mis = (int)(reinterpret_cast<uintptr_t>(g) & 15);
      const uint8_t* raw = sRaw + (R & (kS1RawSlots - 1)) * kS1RawPitch;
      const int base = mis + 2 * kStemC * w;                       // first byte of pixel w's 21-byte run
      const uint32_t* wp = reinterpret_cast<const uint32_t*>(raw + (base & ~3));
      const int sh = 8 * (base & 3);
      uint32_t wd[7];
#pragma unroll
      for (int i = 0; i < 7; ++i) wd[i] = wp[i];
      uint32_t hw[16];
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        const uint32_t v = __funnelshift_r(wd[i], wd[i + 1], sh);
        uint32_t a = __byte_perm(v, 0x64646464u, 0x4140), b = __byte_perm(v, 0x64646464u, 0x4342);
        const __half2 ha = __hfma2(*reinterpret_cast<__half2*>(&a), kScale, kBias), hb = __hfma2(*reinterpret_cast<__half2*>(&b), kScale, kBias);
        hw[2 * i] = *reinterpret_cast<const uint32_t*>(&ha);
        hw[2 * i + 1] = *reinterpret_cast<const uint32_t*>(&hb);
      }
      hw[10] &= 0x0000FFFFu;                                        // k = 21: zero weight, but keep it a clean zero
      hw[11] = 0u;
      hw[12] = hw[13] = hw[14] = hw[15] = 0u;
      mbar_wait(&a_empty[slot], ph ^ 1);
      uint8_t* rowp = sA + slot * 8192 + w * 64;
      const int sw = (w >> 1) & 3;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        *reinterpret_cast<uint4*>(rowp + ((j ^ sw) << 4)) = make_uint4(hw[4 * j], hw[4 * j + 1], hw[4 * j + 2], hw[4 * j + 3]);
      fence_proxy_async();
      mbar_arrive(&a_full[slot]);
      if (++slot == kS1ARing) { slot = 0; ph ^= 1; }
      if (++r == rows_per_image) { r = 0; ++li; }
    }
  } else {
    // ===== epilogue: after every even input row the slot of output row o' - 1 is complete =====
    const int q = warp & 3;
    const int w = q * 32 + lane;
    const uint32_t t_lane = tmem_base + ((uint32_t)(q * 32) << 16);
    tmem_st32_zero(t_lane);
    tmem_st32_zero(t_lane + 32);
    tmem_st_wait();
    tc_fence_before();
    mbar_arrive(acc_free);                                          // completion #0
    uint32_t n_even = 0;
    for (int li = 0; li < n_img; ++li) {
      const long long img = (long long)blockIdx.x + (long long)li * G;
      for (int op = 0; op <= p.Ho; ++op) {                          // even input row 2 op closes output row op - 1
        mbar_wait(acc_done, n_even & 1u);
        tc_fence_after();
        ++n_even;
        const int sl = (op + 1) & 1;                                // slot of output row op - 1
        uint32_t v[32];
        tmem_ld32(t_lane + sl * 32, v);
        tmem_ld_wait();
        tmem_st32_zero(t_lane + sl * 32);
        tmem_st_wait();
        tc_fence_before();
        mbar_arrive(acc_free);
        if (op >= 1 && w < p.Wo) {
          __half* dst = p.out + (((size_t)img * p.Ho + (op - 1)) * p.Wo + w) * p.out_cstride;
          epilogue_chunk<32>(v, s_bias, dst, true, 1);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base, 64);
}

// 3x3 pooling on NHWC fp16.  mode 0: max, stride 2, valid.  mode 1: average, stride 1, 'same', divisor = number
// of in-bounds taps (TF AveragePooling2D semantics).  One thread owns (image, output row, 8 channels) and slides
// along W keeping the per-column partial results of the previous columns in registers, so every input element is
// loaded once per output row (3 loads per output for the stride-1 average, 6 for the stride-2 max) instead of 9.
__device__ __forceinline__ void load8(const __half* p, float (&v)[8]) {
  const uint4 raw = *reinterpret_cast<const uint4*>(p);
  const __half2* h2 = reinterpret_cast<const __half2*>(&raw);
#pragma unroll
  for (int j = 0; j < 4; ++j) { const float2 f = __half22float2(h2[j]); v[2 * j] = f.x; v[2 * j + 1] = f.y; }
}
__device__ __forceinline__ void store8(__half* p, const float (&v)[8]) {
  uint32_t pk[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) { __half2 hh = __floats2half2_rn(v[2 * j], v[2 * j + 1]); pk[j] = *reinterpret_cast<uint32_t*>(&hh); }
  *reinterpret_cast<uint4*>(p) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
}

// split mode: value = main + res * 2^-11 (see "precision = 1"); `off` is the element offset shared by both planes
__device__ __forceinline__ void load8s(const __half* main, const __half* res, size_t off, float (&v)[8]) {
  load8(main + off, v);
  if (res) {
    float r[8];
    load8(res + off, r);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] += r[j] * kSplitInv;
  }
}
__device__ __forceinline__ void store8s(__half* main, __half* res, size_t off, const float (&v)[8]) {
  if (!res) { store8(main + off, v); return; }
  uint32_t pm[4], pr[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) split_store2(v[2 * j], v[2 * j + 1], &pm[j], &pr[j]);
  *reinterpret_cast<uint4*>(main + off) = make_uint4(pm[0], pm[1], pm[2], pm[3]);
  *reinterpret_cast<uint4*>(res + off) = make_uint4(pr[0], pr[1], pr[2], pr[3]);
}

__global__ void pool3x3_kernel(const __half* __restrict__ in, __half* __restrict__ out, int n_images, int Hin, int Win, int C,
                               int Hout, int Wout, int out_cstride, int out_coff, int mode, const __half* __restrict__ in_res,
                               __half* __restrict__ out_res, const float* __restrict__ bias) {
  const int cvec = C / 8;
  const long long total = (long long)n_images * Hout * cvec;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int cv = (int)(i % cvec);
  long long t = i / cvec;
  const int oh = (int)(t % Hout);
  const int n = (int)(t / Hout);
  const size_t src = (size_t)n * Hin * Win * C + cv * 8;
  const size_t dst = ((size_t)n * Hout + oh) * Wout * out_cstride + out_coff + cv * 8;
  if (mode == 0) {
    // column maxima over rows 2oh..2oh+2; output ow uses columns 2ow, 2ow+1, 2ow+2
    const size_t r0 = src + (size_t)(2 * oh) * Win * C;
    float prev[8], a[8], b[8], c[8];
    auto colmax = [&](int iw, float (&m)[8]) {
      load8s(in, in_res, r0 + (size_t)iw * C, a); load8s(in, in_res, r0 + ((size_t)Win + iw) * C, b);
      load8s(in, in_res, r0 + ((size_t)2 * Win + iw) * C, c);
#pragma unroll
      for (int j = 0; j < 8; ++j) m[j] = fmaxf(a[j], fmaxf(b[j], c[j]));
    };
    colmax(0, prev);
    for (int ow = 0; ow < Wout; ++ow) {
      float m1[8], m2[8], o[8];
      colmax(2 * ow + 1, m1);
      colmax(2 * ow + 2, m2);
#pragma unroll
      for (int j = 0; j < 8; ++j) { o[j] = fmaxf(prev[j], fmaxf(m1[j], m2[j])); prev[j] = m2[j]; }
      store8s(out, out_res, dst + (size_t)ow * out_cstride, o);
    }
  } else {
    const int h_lo = oh > 0 ? oh - 1 : 0, h_hi = oh + 1 < Hin ? oh + 1 : Hin - 1;
    const int nrows = h_hi - h_lo + 1;
    float s0[8], s1[8], s2[8], v[8];
    auto colsum = [&](int iw, float (&m)[8]) {
#pragma unroll
      for (int j = 0; j < 8; ++j) m[j] = 0.f;
      if (iw < 0 || iw >= Win) return;
      for (int ih = h_lo; ih <= h_hi; ++ih) {
        load8s(in, in_res, src + ((size_t)ih * Win + iw) * C, v);
#pragma unroll
        for (int j = 0; j < 8; ++j) m[j] += v[j];
      }
    };
    colsum(-1, s0);
    colsum(0, s1);
    for (int ow = 0; ow < Wout; ++ow) {
      colsum(ow + 1, s2);
      const int ncols = (ow > 0 ? 1 : 0) + 1 + (ow + 1 < Win ? 1 : 0);
      const float inv = 1.f / (float)(nrows * ncols);
      float o[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) { o[j] = (s0[j] + s1[j] + s2[j]) * inv; s0[j] = s1[j]; s1[j] = s2[j]; }
      if (bias) {
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = fmaxf(o[j] + bias[cv * 8 + j], 0.f);
      }
      store8s(out, out_res, dst + (size_t)ow * out_cstride, o);
    }
  }
}

// 3x3 stride-2 'valid' max pool, precision 0: the maximum of fp16 values is exact in fp16, so the whole pool runs on packed
// half2 (__hmax2) without a single conversion - a third of the instructions and half the registers of the fp32 form above.
// One thread = (image, output row, segment of the row, 8 channels); segments shorten the serial sliding chain.
__global__ void __launch_bounds__(256) maxpool3x3s2_h2_kernel(const __half* __restrict__ in, __half* __restrict__ out, int n_images, int Hin, int Win,
                                                              int C, int Hout, int Wout, int out_cstride, int out_coff, int segs, int seg_len) {
  const int cvec = C / 8;
  const long long total = (long long)n_images * Hout * segs * cvec;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int cv = (int)(i % cvec);
  long long t = i / cvec;
  const int seg = (int)(t % segs); t /= segs;
  const int oh = (int)(t % Hout);
  const int n = (int)(t / Hout);
  const int ow0 = seg * seg_len, ow1 = min(Wout, ow0 + seg_len);
  if (ow0 >= ow1) return;
  const uint4* r0 = reinterpret_cast<const uint4*>(in + (((size_t)n * Hin + 2 * oh) * Win) * C + cv * 8);
  const size_t pitch = (size_t)C / 8;            // uint4 per pixel
  const size_t row = (size_t)Win * pitch;        // uint4 per input row
  auto colmax = [&](int iw) { return hmax2x4(r0[iw * pitch], hmax2x4(r0[row + iw * pitch], r0[2 * row + iw * pitch])); };
  __half* dst = out + (((size_t)n * Hout + oh) * Wout) * out_cstride + out_coff + cv * 8;
  uint4 prev = colmax(2 * ow0);
  for (int ow = ow0; ow < ow1; ++ow) {
    const uint4 m1 = colmax(2 * ow + 1), m2 = colmax(2 * ow + 2);
    *reinterpret_cast<uint4*>(dst + (size_t)ow * out_cstride) = hmax2x4(prev, hmax2x4(m1, m2));
    prev = m2;
  }
}

// 3x3 stride-1 'same' average pool (count excludes the padding) [+ bias + ReLU when it stands behind its 1x1 convolution], precision 0.
// One thread = one output pixel x 8 channels: its nine 16-byte loads are independent (the sliding form of pool3x3_kernel above chains
// Wout dependent load groups per thread: 1 TB/s on maps that should stream at 5), neighbours meet in L1.  The sums are taken in the
// order of pool3x3_kernel (per column top to bottom, then left + centre + right): results are bit-identical.
__global__ void __launch_bounds__(256) avgpool3x3s1_kernel(const __half* __restrict__ in, __half* __restrict__ out, int n_images, int H, int W, int C,
                                                           int out_cstride, int out_coff, const float* __restrict__ bias) {
  const int cvec = C / 8;
  const long long total = (long long)n_images * H * W * cvec;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const int cv = (int)(i % cvec);
  long long t = i / cvec;
  const int ow = (int)(t % W); t /= W;
  const int oh = (int)(t % H);
  const int n = (int)(t / H);
  const int h_lo = oh > 0 ? oh - 1 : 0, h_hi = oh + 1 < H ? oh + 1 : H - 1;
  const int w_lo = ow > 0 ? ow - 1 : 0, w_hi = ow + 1 < W ? ow + 1 : W - 1;
  const uint4* src = reinterpret_cast<const uint4*>(in + (size_t)n * H * W * C + cv * 8);
  const size_t pitch = (size_t)C / 8;
  uint4 v[3][3];
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int b = 0; b < 3; ++b) {
      const int ih = h_lo + a, iw = w_lo + b;
      v[a][b] = (ih <= h_hi && iw <= w_hi) ? src[((size_t)ih * W + iw) * pitch] : make_uint4(0, 0, 0, 0);
    }
  // columns left of / right of the map contribute an exact 0.f first or last, as colsum(-1) / colsum(W) do above
  float col[3][8];
#pragma unroll
  for (int b = 0; b < 3; ++b) {
#pragma unroll
    for (int j = 0; j < 8; ++j) col[b][j] = 0.f;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      if (h_lo + a > h_hi || w_lo + b > w_hi) continue;
      const __half2* h2 = reinterpret_cast<const __half2*>(&v[a][b]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = __half22float2(h2[j]);
        col[b][2 * j] += f.x; col[b][2 * j + 1] += f.y;
      }
    }
  }
  const int ncols = w_hi - w_lo + 1;
  const float inv = 1.f / (float)((h_hi - h_lo + 1) * ncols);
  float o[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    // pool3x3_kernel adds s0 + s1 + s2 = (column ow-1) + (column ow) + (column ow+1), absent columns as 0.f
    const float s0 = ow > 0 ? col[0][j] : 0.f;
    const float s1 = ow > 0 ? col[1][j] : col[0][j];
    const float s2 = ow > 0 ? (ncols == 3 ? col[2][j] : 0.f) : (ncols >= 2 ? col[1][j] : 0.f);
    o[j] = __fmul_rn(s0 + s1 + s2, inv);                                    // no FMA contraction with the bias: pool3x3_kernel rounds the mean first
    if (bias) o[j] = fmaxf(__fadd_rn(o[j], bias[cv * 8 + j]), 0.f);
  }
  uint32_t pk[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const __half2 h = __floats2half2_rn(o[2 * j], o[2 * j + 1]);
    pk[j] = *reinterpret_cast<const uint32_t*>(&h);
  }
  *reinterpret_cast<uint4*>(out + (((size_t)n * H + oh) * W + ow) * out_cstride + out_coff + cv * 8) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
}

// GlobalAveragePooling2D + Dense(3) + softmax, fp32.  One block per image.
__global__ void __launch_bounds__(256) tail_kernel(const __half* __restrict__ feat, int hw, int C, const float* __restrict__ dense_w,
                                                   const float* __restrict__ dense_b, float* __restrict__ probs, float* __restrict__ pooled_out,
                                                   const __half* __restrict__ feat_res) {
  const int n = blockIdx.x;
  const __half* f = feat + (size_t)n * hw * C;
  const __half* fr = feat_res ? feat_res + (size_t)n * hw * C : nullptr;
  float l0 = 0.f, l1 = 0.f, l2 = 0.f;
  const float inv = 1.f / (float)hw;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s = 0.f;
    for (int p = 0; p < hw; ++p) s += __half2float(f[(size_t)p * C + c]);
    if (fr) {
      float sr = 0.f;
      for (int p = 0; p < hw; ++p) sr += __half2float(fr[(size_t)p * C + c]);
      s += sr * kSplitInv;
    }
    s *= inv;
    if (pooled_out) pooled_out[(size_t)n * C + c] = s;
    l0 += s * dense_w[c * 3 + 0];
    l1 += s * dense_w[c * 3 + 1];
    l2 += s * dense_w[c * 3 + 2];
  }
  __shared__ float red[3][8];
  for (int o = 16; o > 0; o >>= 1) {
    l0 += __shfl_xor_sync(0xffffffffu, l0, o);
    l1 += __shfl_xor_sync(0xffffffffu, l1, o);
    l2 += __shfl_xor_sync(0xffffffffu, l2, o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { red[0][warp] = l0; red[1][warp] = l1; red[2][warp] = l2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    float z[3];
    for (int k = 0; k < 3; ++k) {
      float s = dense_b[k];
      for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[k][w];
      z[k] = s;
    }
    const float m = fmaxf(z[0], fmaxf(z[1], z[2]));
    const float e0 = expf(z[0] - m), e1 = expf(z[1] - m), e2 = expf(z[2] - m);
    const float d = e0 + e1 + e2;
    probs[n * 3 + 0] = e0 / d;
    probs[n * 3 + 1] = e1 / d;
    probs[n * 3 + 2] = e2 / d;
  }
}

__global__ void half_to_float_kernel(const __half* __restrict__ in, const __half* __restrict__ in_res, float* __restrict__ out, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __half2float(in[i]) + (in_res ? __half2float(in_res[i]) * kSplitInv : 0.f);
}

// ---------------------------------------------------------------------------------------------
// Host side: network plan
// ---------------------------------------------------------------------------------------------

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn GetEncodeTiled() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

struct TensorBuf {
  std::string name;
  int H = 0, W = 0, C = 0;   // C = stored channels (padded for the input)
  int Cl = 0;                // logical channels (<= C; the rest is zero padding)
  __half* ptr = nullptr;
  __half* ptr_res = nullptr;   // residual plane (precision 1), else null
};

struct OpDesc {
  int kind;  // 0 conv, 1 maxpool, 2 avgpool
  std::string src, dst;
  int off, cin, cout, kh, kw, stride, same;
  int no_act = 0;      // conv: raw accumulator out (no bias, no ReLU) - its bias + ReLU move behind the following pool
  int post_act = 0;    // pool: + bias of the preceding conv, ReLU
};

int PadCin(int cin) { return cin < 16 ? 16 : (cin + 7) / 8 * 8; }

// Restates deepvariant_b200/modeling.py inception_v3_graph() (tf_keras InceptionV3 topology).
void BuildGraph(int in_channels, std::vector<OpDesc>* ops, std::map<std::string, int>* ch) {
  (*ch)["input"] = in_channels;
  auto conv = [&](const std::string& s, const std::string& d, int cout, int kh, int kw, int stride = 1, int same = 1, int off = 0,
                  int total = 0) {
    if (!ch->count(d)) (*ch)[d] = total ? total : cout;
    ops->push_back({0, s, d, off, (*ch)[s], cout, kh, kw, stride, same});
  };
  auto pool = [&](int kind, const std::string& s, const std::string& d, int off = 0, int total = 0) {
    if (!ch->count(d)) (*ch)[d] = total ? total : (*ch)[s];
    ops->push_back({kind, s, d, off, (*ch)[s], (*ch)[s], 3, 3, kind == 1 ? 2 : 1, kind == 2});
  };
  conv("input", "s1", 32, 3, 3, 2, 0);
  conv("s1", "s2", 32, 3, 3, 1, 0);
  conv("s2", "s3", 64, 3, 3);
  pool(1, "s3", "p1");
  conv("p1", "s4", 80, 1, 1, 1, 0);
  conv("s4", "s5", 192, 3, 3, 1, 0);
  pool(1, "s5", "p2");
  std::string x = "p2";
  const int pool_ch[3] = {32, 64, 64};
  for (int i = 0; i < 3; ++i) {
    const std::string m = "mixed" + std::to_string(i);
    const int total = 64 + 64 + 96 + pool_ch[i];
    conv(x, m, 64, 1, 1, 1, 1, 0, total);
    conv(x, m + "_b5a", 48, 1, 1);
    conv(m + "_b5a", m, 64, 5, 5, 1, 1, 64);
    conv(x, m + "_d1", 64, 1, 1);
    conv(m + "_d1", m + "_d2", 96, 3, 3);
    conv(m + "_d2", m, 96, 3, 3, 1, 1, 128);
    pool(2, x, m + "_ap");
    conv(m + "_ap", m, pool_ch[i], 1, 1, 1, 1, 224);
    x = m;
  }
  {
    const int total = 384 + 96 + (*ch)[x];
    conv(x, "mixed3", 384, 3, 3, 2, 0, 0, total);
    conv(x, "mixed3_d1", 64, 1, 1);
    conv("mixed3_d1", "mixed3_d2", 96, 3, 3);
    conv("mixed3_d2", "mixed3", 96, 3, 3, 2, 0, 384);
    pool(1, x, "mixed3", 480);
    x = "mixed3";
  }
  const int c7s[4] = {128, 160, 160, 192};
  for (int i = 4; i <= 7; ++i) {
    const std::string m = "mixed" + std::to_string(i);
    const int c7 = c7s[i - 4];
    conv(x, m, 192, 1, 1, 1, 1, 0, 768);
    conv(x, m + "_s1", c7, 1, 1);
    conv(m + "_s1", m + "_s2", c7, 1, 7);
    conv(m + "_s2", m, 192, 7, 1, 1, 1, 192);
    conv(x, m + "_d1", c7, 1, 1);
    conv(m + "_d1", m + "_d2", c7, 7, 1);
    conv(m + "_d2", m + "_d3", c7, 1, 7);
    conv(m + "_d3", m + "_d4", c7, 7, 1);
    conv(m + "_d4", m, 192, 1, 7, 1, 1, 384);
    pool(2, x, m + "_ap");
    conv(m + "_ap", m, 192, 1, 1, 1, 1, 576);
    x = m;
  }
  {
    const int total = 320 + 192 + (*ch)[x];
    conv(x, "mixed8_a1", 192, 1, 1);
    conv("mixed8_a1", "mixed8", 320, 3, 3, 2, 0, 0, total);
    conv(x, "mixed8_b1", 192, 1, 1);
    conv("mixed8_b1", "mixed8_b2", 192, 1, 7);
    conv("mixed8_b2", "mixed8_b3", 192, 7, 1);
    conv("mixed8_b3", "mixed8", 192, 3, 3, 2, 0, 320);
    pool(1, x, "mixed8", 512);
    x = "mixed8";
  }
  for (int i = 9; i <= 10; ++i) {
    const std::string m = "mixed" + std::to_string(i);
    conv(x, m, 320, 1, 1, 1, 1, 0, 2048);
    conv(x, m + "_t1", 384, 1, 1);
    conv(m + "_t1", m, 384, 1, 3, 1, 1, 320);
    conv(m + "_t1", m, 384, 3, 1, 1, 1, 704);
    conv(x, m + "_d1", 448, 1, 1);
    conv(m + "_d1", m + "_d2", 384, 3, 3);
    conv(m + "_d2", m, 384, 1, 3, 1, 1, 1088);
    conv(m + "_d2", m, 384, 3, 1, 1, 1, 1472);
    pool(2, x, m + "_ap");
    conv(m + "_ap", m, 192, 1, 1, 1, 1, 1856);
    x = m;
  }
}

struct ConvLaunch {
  CUtensorMap map_a, map_b, map_a_res, map_b_res;
  ConvArgs args;
  dim3 grid;
  int smem;
  double macs_per_image;
  bool flat;
  int pixels_per_image;
  bool persist;          // conv_gemm_persistent_kernel
  bool pair;             // conv_gemm_pair_kernel (cta_group::2) instead of the persistent kernel
  CUtensorMap map_b_half;
  PairArgs pair_args;
  int pair_smem;
  int n_blocks, cout;
};
struct HaloLaunch {
  CUtensorMap map_a, map_b, map_a_res, map_b_res;
  HaloArgs args;
  int smem, ctas_per_nblock;
  double macs_per_image;
};
struct RowsLaunch {
  CUtensorMap map_a, map_b;
  RowsArgs args;
  int smem;
  double macs_per_image;
};
struct PoolLaunch {
  const __half* in; __half* out;
  int Hin, Win, C, Hout, Wout, out_cstride, out_coff, mode;
  const __half* in_res; __half* out_res;
  const float* bias;     // post_act pools: + bias[c], ReLU (else null)
};
// One launch of the forward.  The inception branches are independent chains: every step runs on one of kMaxLanes
// streams ("lanes"; lane 0 = the caller's stream) and waits on the events of the producers of its source tensor that
// ran on other lanes, so that the partial last wave of one branch's kernel is filled by another branch's CTAs.
constexpr int kMaxLanes = 4;
struct Step {
  int kind, index;          // 0 conv, 1 pool, 2 halo conv, 3 row-streaming conv (+ fused max pool)
  int lane = 0;
  bool record = false;      // some consumer on another lane waits on this step's event
  std::vector<int> deps;    // steps (other lanes) to wait on before launching
  cudaEvent_t event = nullptr;
};

}  // namespace

struct DvbCnn {
  int device = 0, H = 0, W = 0, C = 0, Cp = 16, max_batch = 0, precision = 0;
  int stem_Ho = 0, stem_Wo = 0, stem_Kp = 64, num_sms = 148;
  std::vector<TensorBuf> tensors;
  std::map<std::string, int> tensor_index;
  std::vector<ConvLaunch> convs;
  std::vector<HaloLaunch> halos;
  std::vector<RowsLaunch> rows;
  std::vector<PoolLaunch> pools;
  std::vector<Step> steps;
  std::vector<void*> allocs;
  float* d_dense_w = nullptr; float* d_dense_b = nullptr;
  float* d_pooled = nullptr;
  int feat_tensor = -1;
  double flops_per_image = 0;
  int64_t launches = 0;
  cudaStream_t stream = nullptr;
  bool stem_fused = false;
  StemArgs stem_args;
  bool stem_rows = false;          // stem_rows_kernel instead of stem_conv1_kernel
  Stem2Args stem2_args;
  int n_lanes = 1;
  cudaStream_t lane_streams[kMaxLanes] = {nullptr, nullptr, nullptr, nullptr};   // [0] unused (caller's stream)
  struct ChunkGraph { const uint8_t* images; float* probs; int n; cudaGraphExec_t exec; int64_t launches; };
  std::vector<ChunkGraph> graphs;      // DVB_CNN_GRAPH: captured chunk forwards, keyed by (images, probs, n)
  bool use_graphs = false;
  std::vector<int> tail_deps;
  dvb::DevBuf d_in, d_probs;
  dvb::PinBuf h_io;
};

namespace {

struct TileChoice { int Wt, Ht, Nt; };

int EnvInt(const char* name, int dflt) {
  const char* v = getenv(name);
  return v ? atoi(v) : dflt;
}


// The M tile is ANY box of Wt x Ht x Nt output pixels (row = (n * Ht + h) * Wt + w): batching images into the tile is
// not limited to whole feature maps, e.g. the 4x12 maps of mixed3..7 tile as 4 x 4 x 8 = 128 rows (100 % full; a
// whole-map tile would be 12 x 4 x 2 = 96 rows = 75 %).
TileChoice ChooseTile(int Hout, int Wout, int stride) {
  TileChoice best{1, 1, 1};
  double best_eff = -1;
  const int max_box = 256 / stride;  // boxDim <= 256 in input space
  const bool batch_any = EnvInt("DVB_CNN_TILE_ANY_N", 1) != 0;
  for (int Wt = 1; Wt <= std::min(std::min(Wout, 128), max_box); ++Wt) {
    for (int Ht = 1; Ht <= std::min(std::min(Hout, 128 / Wt), max_box); ++Ht) {
      const int nt_max = (batch_any || (Wt == Wout && Ht == Hout)) ? std::max(1, 128 / (Wt * Ht)) : 1;
      for (int Nt = 1; Nt <= nt_max; ++Nt) {
        const long tiles = (long)((Wout + Wt - 1) / Wt) * ((Hout + Ht - 1) / Ht);
        const double eff = (double)Wout * Hout * Nt / ((double)tiles * 128.0);
        // ties: wider rows first (longer contiguous TMA runs), then fewer images per tile
        if (eff > best_eff + 1e-9 || (std::fabs(eff - best_eff) <= 1e-9 && (Wt > best.Wt || (Wt == best.Wt && Nt < best.Nt)))) {
          best_eff = eff;
          best = {Wt, Ht, Nt};
        }
      }
    }
  }
  return best;
}

int ChooseBlockN(int cout) {
  if (cout <= 256) return cout;
  for (int d = 256; d >= 16; d -= 16)
    if (cout % d == 0) return d;
  return 16;
}

int TmemCols(int n) { int c = 32; while (c < n) c <<= 1; return c; }

int MakeMap(CUtensorMap* m, void* ptr, int rank, const cuuint64_t* dims, const cuuint64_t* strides_bytes, const cuuint32_t* box,
            const cuuint32_t* estr, int block_k) {
  EncodeTiledFn fn = GetEncodeTiled();
  if (!fn) return dvb::fail(DVB_ERR_CUDA, "cuTensorMapEncodeTiled entry point not found");
  CUtensorMapSwizzle sw = block_k == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : block_k == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, ptr, dims, strides_bytes, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return dvb::fail(DVB_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d (rank %d)", (int)r, rank);
  return DVB_OK;
}

int Plan(DvbCnn* net, const uint8_t* blob, int64_t blob_bytes) {
  std::vector<OpDesc> ops;
  std::map<std::string, int> ch;
  BuildGraph(net->C, &ops, &ch);
  // Average pool followed by a 1x1 convolution: both are linear and act on different axes (the pool per channel over
  // space, the convolution per pixel over channels; the 'same'-padding divisor depends on the pixel only), so
  //     relu(conv1x1(avgpool(x)) + b) == relu(avgpool(conv1x1(x)) + b).
  // Running the convolution first shrinks what the pool has to stream by Cin / Cout (768 -> 192, 2048 -> 192, ...).
  if (EnvInt("DVB_CNN_POOL_AFTER_CONV", 1)) {
    for (size_t i = 0; i + 1 < ops.size(); ++i) {
      OpDesc& pl = ops[i];
      OpDesc& cv = ops[i + 1];
      if (pl.kind == 2 && cv.kind == 0 && cv.kh == 1 && cv.kw == 1 && cv.stride == 1 && cv.src == pl.dst) {
        const std::string x = pl.src, mid = pl.dst, out = cv.dst;
        const int off = cv.off, cout = cv.cout;
        OpDesc conv = cv, pool = pl;
        conv.src = x; conv.dst = mid; conv.off = 0; conv.no_act = 1;
        pool.src = mid; pool.dst = out; pool.off = off; pool.cin = cout; pool.cout = cout; pool.post_act = 1;
        ch[mid] = cout;
        ops[i] = conv; ops[i + 1] = pool;
        ++i;
      }
    }
  }
  // --- header
  if (blob_bytes < 12) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "weights blob too small");
  const int32_t* hdr = reinterpret_cast<const int32_t*>(blob);
  if ((uint32_t)hdr[0] != kBlobMagic && (uint32_t)hdr[0] != kBlobMagic2) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "weights blob: bad magic");
  const bool blob_split = (uint32_t)hdr[0] == kBlobMagic2;
  const bool split = net->precision == 1;
  if (split && !blob_split)
    return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "precision 1 needs a weights blob with residual planes (modeling.pack_weights(w, precision=1))");
  if (hdr[1] != net->C) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "weights blob is for %d input channels, not %d", hdr[1], net->C);
  int n_conv = 0;
  for (auto& o : ops) n_conv += o.kind == 0;
  if (hdr[2] != n_conv) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "weights blob has %d convs, expected %d", hdr[2], n_conv);
  int64_t pos = 12;
  // blob offset of every convolution (network order), so that layers can be fetched out of order
  std::vector<int64_t> conv_pos;
  {
    int64_t q = 12;
    for (int ci = 0; ci < n_conv; ++ci) {
      if (q + 20 > blob_bytes) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "weights blob truncated");
      const int32_t* lh = reinterpret_cast<const int32_t*>(blob + q);
      if (lh[0] < 1 || lh[1] < 1 || lh[3] < 1 || lh[4] < 1) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "weights blob: bad conv header %d", ci);
      conv_pos.push_back(q);
      q += 20 + (int64_t)(blob_split ? 2 : 1) * lh[4] * lh[0] * lh[1] * lh[3] * (int64_t)sizeof(__half) + (int64_t)lh[4] * 4;
    }
    conv_pos.push_back(q);
    if (q > blob_bytes) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "weights blob truncated");
  }
  // 1x1 stride-1 convolutions that read the SAME tensor (the branch heads of an inception block, including the one the
  // average pool now follows) run as ONE GEMM over their concatenated filters: the input is fetched once instead of 2-4
  // times and the MMA's N grows from 32-192 to 208-256 (an M=128 SS-mode MMA streams 4 KB of A per instruction whatever
  // N is, so narrow N wastes the tensor pipe).  leader[i] = ops merged into op i (first of its group); merged_into[i] >= 0
  // for the others.
  std::vector<int> conv_index_of(ops.size(), -1);
  {
    int ci = 0;
    for (size_t i = 0; i < ops.size(); ++i)
      if (ops[i].kind == 0) conv_index_of[i] = ci++;
  }
  std::map<size_t, std::vector<size_t>> leader;
  std::vector<int> merged_into(ops.size(), -1);
  if (!split && EnvInt("DVB_CNN_MERGE_1X1", 1)) {
    std::map<std::string, std::vector<size_t>> by_src;
    for (size_t i = 1; i < ops.size(); ++i)
      if (ops[i].kind == 0 && ops[i].kh == 1 && ops[i].kw == 1 && ops[i].stride == 1) by_src[ops[i].src].push_back(i);
    for (auto& kv : by_src) {
      if (kv.second.size() < 2 || (int)kv.second.size() > kMaxSegs) continue;
      leader[kv.second[0]] = kv.second;
      for (size_t k = 1; k < kv.second.size(); ++k) merged_into[kv.second[k]] = (int)kv.second[0];
    }
  }
  std::map<std::string, const float*> pool_bias;   // '*_ap' tensor -> bias its pool adds (bias of the no_act convolution)
  // Storage channel counts: a tensor that feeds a k x k convolution and has a channel count that only 16 divides (s4: 80,
  // the 5x5 inputs: 48) is stored padded to a multiple of 32 (zeros, never written), so that its consumer runs 64-byte K
  // blocks of two MMAs instead of 32-byte blocks of one - half the barrier round trips per tile for 20-33 % more (cheap)
  // MMA work.  Measured per 16,384 images: 69.2 ms -> 67.4 (80 -> 96) -> 65.8 (48 -> 64 as well).
  std::map<std::string, int> store_ch;
  if (EnvInt("DVB_CNN_PAD_CIN32", 1)) {
    const int min_c = EnvInt("DVB_CNN_PAD_CIN32_MIN", 48);
    for (auto& o : ops) {
      if (o.kind != 0 || o.kh * o.kw == 1) continue;
      const int c = ch[o.src];
      if (c < min_c || c % 16 != 0) continue;
      const int pad64_min = EnvInt("DVB_CNN_PAD_CIN64_MIN", 0);   // > 0: tensors with at least this many channels are padded to multiples of 64 (128-byte TMA rows)
      const int target = (pad64_min > 0 && c >= pad64_min && c % 64) ? (c + 63) / 64 * 64
                                                                     : (c % 32 ? (c + 31) / 32 * 32 : c);   // (padding everything to 64 measured slower in round 1: 65.4 -> 66.0-66.4 ms)
      if (target != c) store_ch[o.src] = target;
    }
    // A pool copies its source's STORED channel count into its slice of the block tensor, so a padded source would spill into the
    // next pixel's first channels (seen with DVB_CNN_PAD_CIN64_MIN=160: mixed2, 288 -> 320, feeds conv27 AND the block's max pool;
    // the default rule only pads s4 and the 48-channel 5x5 inputs, which no pool reads).  Such tensors keep their own width.
    for (auto& o : ops)
      if (o.kind != 0) store_ch.erase(o.src);
  }
  auto stored = [&](const std::string& name) { return store_ch.count(name) ? store_ch[name] : ch[name]; };

  // --- tensors
  std::map<std::string, std::pair<int, int>> hw;
  hw["input"] = {net->H, net->W};
  auto add_tensor = [&](const std::string& name, int H, int W, int C) -> int {
    if (net->tensor_index.count(name)) return DVB_OK;
    TensorBuf t;
    t.name = name; t.H = H; t.W = W; t.C = C;
    t.Cl = store_ch.count(name) ? ch[name] : C;
    const size_t bytes = (size_t)net->max_batch * H * W * C * sizeof(__half);
    void* p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) return dvb::fail(DVB_ERR_CUDA, "cudaMalloc of %zu bytes for tensor %s failed", bytes, name.c_str());
    cudaMemset(p, 0, bytes);
    net->allocs.push_back(p);
    t.ptr = static_cast<__half*>(p);
    if (split) {
      void* q = nullptr;
      if (cudaMalloc(&q, bytes) != cudaSuccess) return dvb::fail(DVB_ERR_CUDA, "cudaMalloc of %zu bytes for tensor %s (residual plane) failed", bytes, name.c_str());
      cudaMemset(q, 0, bytes);
      net->allocs.push_back(q);
      t.ptr_res = static_cast<__half*>(q);
    }
    net->tensor_index[name] = (int)net->tensors.size();
    net->tensors.push_back(t);
    return DVB_OK;
  };
  // The first convolution (3x3 stride 2 valid) runs as a GEMM over pre-gathered patches (stem_patch_kernel):
  // tensor "input" holds [N][Ho][Wo][Kp] with k = (r*3 + s)*C + c.
  if (ops.empty() || ops[0].kind != 0 || ops[0].kh != 3 || ops[0].kw != 3 || ops[0].stride != 2 || ops[0].same)
    return dvb::fail(DVB_ERR_INTERNAL, "unexpected stem");
  if (net->H < 3 || net->W < 3) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "image %dx%d is too small for the network", net->H, net->W);
  net->stem_Ho = (net->H - 3) / 2 + 1;
  net->stem_Wo = (net->W - 3) / 2 + 1;
  net->stem_Kp = 9 * net->C <= 64 ? 64 : (9 * net->C + 31) / 32 * 32;
  hw["input"] = {net->stem_Ho, net->stem_Wo};
  int st = add_tensor("input", net->stem_Ho, net->stem_Wo, net->stem_Kp);
  if (st) return st;

  std::vector<std::pair<std::string, std::vector<std::string>>> step_io;   // (src, dst tensors) of every step
  std::vector<char> fused_pool(ops.size(), 0);
  std::map<std::string, int> n_consumers;
  for (auto& oo : ops) n_consumers[oo.src]++;
  const int force_bk = EnvInt("DVB_CNN_BLOCK_K", 0);       // 0 = per-layer choice
  double macs_total = 0;
  for (size_t op_index = 0; op_index < ops.size(); ++op_index) {
    OpDesc o = ops[op_index];
    const bool is_stem = op_index == 0;
    const OpDesc orig = o;
    if (is_stem) { o.kh = 1; o.kw = 1; o.stride = 1; o.same = 0; }   // GEMM over the patch tensor
    const auto [Hin, Win] = hw[o.src];
    int Hout, Wout;
    if (o.same) { Hout = Hin; Wout = Win; }
    else {   // a window larger than the map has no output (C++ division truncates toward zero: (2 - 3) / 2 + 1 would be 1)
      Hout = Hin < o.kh ? 0 : (Hin - o.kh) / o.stride + 1;
      Wout = Win < o.kw ? 0 : (Win - o.kw) / o.stride + 1;
    }
    if (Hout < 1 || Wout < 1) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "image %dx%d is too small for the network", net->H, net->W);
    hw[o.dst] = {Hout, Wout};
    if (merged_into[op_index] >= 0) continue;     // runs inside its group leader's GEMM
    if (fused_pool[op_index]) continue;           // this max pool runs in the epilogue of the convolution before it (conv_rows_kernel)
    std::vector<size_t> members = leader.count(op_index) ? leader[op_index] : std::vector<size_t>{op_index};
    // Row-streaming kernel (conv_rows_kernel): 3x3 stride-1 layers with <= 64 filters on maps up to 126 pixels wide - conv2 and
    // conv3 of the stem.  A 3x3 / stride-2 'valid' max pool that is the layer's only consumer runs in its epilogue.
    bool use_rows = false, rows_pool = false;
    if (o.kind == 0 && !split && !is_stem && members.size() == 1 && o.stride == 1 && o.kh == 3 && o.kw == 3 && !o.no_act &&
        (o.cout == 32 || o.cout == 64) && Wout <= 126 && EnvInt("DVB_CNN_ROWS", 1)) {
      const int cs = net->tensors[net->tensor_index[o.src]].C;
      use_rows = (cs == 32 || cs == 64) && o.off == 0 && stored(o.dst) == o.cout;
      if (use_rows && op_index + 1 < ops.size() && EnvInt("DVB_CNN_FUSE_POOL", 1)) {
        const OpDesc& nx = ops[op_index + 1];
        rows_pool = nx.kind == 1 && nx.src == o.dst && n_consumers[o.dst] == 1 && Hout >= 3 && Wout >= 3;
      }
    }
    std::vector<std::string> step_dsts;
    if (rows_pool) {
      const OpDesc& nx = ops[op_index + 1];
      fused_pool[op_index + 1] = 1;
      const int Hp = (Hout - 3) / 2 + 1, Wp = (Wout - 3) / 2 + 1;
      hw[nx.dst] = {Hp, Wp};
      st = add_tensor(nx.dst, Hp, Wp, stored(nx.dst));
      if (st) return st;
      step_dsts.push_back(nx.dst);
    } else {
      for (size_t m : members) {                    // all destination tensors exist before any reference is taken
        hw[ops[m].dst] = {Hout, Wout};
        st = add_tensor(ops[m].dst, Hout, Wout, stored(ops[m].dst));
        if (st) return st;
        step_dsts.push_back(ops[m].dst);
      }
    }
    const TensorBuf& src = net->tensors[net->tensor_index[o.src]];
    const TensorBuf& dst = net->tensors[net->tensor_index[rows_pool ? ops[op_index + 1].dst : o.dst]];
    if (o.kind != 0) {
      PoolLaunch pl{src.ptr, dst.ptr, Hin, Win, src.C, Hout, Wout, dst.C, o.off, o.kind == 1 ? 0 : 1, src.ptr_res, dst.ptr_res,
                    o.post_act ? pool_bias[o.src] : nullptr};
      if (o.post_act && !pl.bias) return dvb::fail(DVB_ERR_INTERNAL, "pool without the bias of its convolution");
      net->steps.push_back(Step{1, (int)net->pools.size()});
      step_io.push_back({o.src, step_dsts});
      net->pools.push_back(pl);
      continue;
    }
    // --- conv weights from the blob (one layer, or the members of a merged group stacked along Cout)
    const int cin_store = src.C;  // channels physically present in the source tensor
    const int blob_cin = PadCin(orig.cin);
    const size_t blob_planes = blob_split ? 2 : 1;
    int cout_total = 0;
    for (size_t m : members) cout_total += ops[m].cout;
    const bool merged = members.size() > 1;
    const size_t wbytes = (size_t)cout_total * o.kh * o.kw * cin_store * sizeof(__half);
    const size_t bbytes = (size_t)cout_total * sizeof(float);
    void* dw = nullptr; void* db = nullptr; void* dw_res = nullptr;
    if (cudaMalloc(&dw, wbytes) != cudaSuccess || cudaMalloc(&db, bbytes) != cudaSuccess) return dvb::fail(DVB_ERR_CUDA, "cudaMalloc (weights) failed");
    net->allocs.push_back(dw); net->allocs.push_back(db);
    if (split) {
      if (cudaMalloc(&dw_res, wbytes) != cudaSuccess) return dvb::fail(DVB_ERR_CUDA, "cudaMalloc (weights) failed");
      net->allocs.push_back(dw_res);
    }
    std::vector<float> bias_host((size_t)cout_total, 0.f);
    std::vector<OutSeg> segs;
    const uint8_t* blob_w_main = nullptr;
    size_t blob_wbytes = 0;
    {
      size_t row0 = 0;   // first output channel of this member inside the stacked filter matrix
      for (size_t m : members) {
        const OpDesc& mo = ops[m];
        pos = conv_pos[conv_index_of[m]];
        const int32_t* lh = reinterpret_cast<const int32_t*>(blob + pos);
        pos += 20;
        if (lh[0] != orig.kh || lh[1] != orig.kw || lh[2] != orig.cin || lh[3] != blob_cin || lh[4] != mo.cout || (!is_stem && blob_cin > cin_store))
          return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "weights blob: conv %d header mismatch (%d %d %d %d %d)", conv_index_of[m], lh[0], lh[1], lh[2],
                           lh[3], lh[4]);
        blob_wbytes = (size_t)mo.cout * orig.kh * orig.kw * blob_cin * sizeof(__half);
        const size_t m_wbytes = (size_t)mo.cout * o.kh * o.kw * cin_store * sizeof(__half);
        if (pos + (int64_t)(blob_planes * blob_wbytes + (size_t)mo.cout * 4) > blob_bytes) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "weights blob truncated");
        for (int plane = 0; plane < (split ? 2 : 1); ++plane) {
          const uint8_t* wsrc = blob + pos + (size_t)plane * blob_wbytes;
          uint8_t* wdst = static_cast<uint8_t*>(plane ? dw_res : dw) + row0 * o.kh * o.kw * cin_store * sizeof(__half);
          if (is_stem) {
            // [cout][3][3][blob_cin] -> [cout][Kp], k = (r*3 + s)*C + c (the patch order of stem_patch_kernel)
            std::vector<__half> w2((size_t)mo.cout * cin_store, __float2half(0.f));
            const __half* w = reinterpret_cast<const __half*>(wsrc);
            for (int co = 0; co < mo.cout; ++co)
              for (int t = 0; t < 9; ++t)
                for (int c = 0; c < net->C; ++c) w2[(size_t)co * cin_store + t * net->C + c] = w[((size_t)co * 9 + t) * blob_cin + c];
            cudaMemcpy(wdst, w2.data(), m_wbytes, cudaMemcpyHostToDevice);
          } else if (blob_cin != cin_store) {
            // the source tensor is stored with more (zero) channels than the blob's kernel has: pad Cin with zero weights
            std::vector<__half> w2((size_t)mo.cout * o.kh * o.kw * cin_store, __float2half(0.f));
            const __half* w = reinterpret_cast<const __half*>(wsrc);
            for (size_t rt = 0; rt < (size_t)mo.cout * o.kh * o.kw; ++rt)
              memcpy(&w2[rt * cin_store], &w[rt * blob_cin], (size_t)blob_cin * sizeof(__half));
            cudaMemcpy(wdst, w2.data(), m_wbytes, cudaMemcpyHostToDevice);
          } else {
            cudaMemcpy(wdst, wsrc, m_wbytes, cudaMemcpyHostToDevice);
          }
        }
        const float* b_blob = reinterpret_cast<const float*>(blob + pos + blob_planes * blob_wbytes);
        if (mo.no_act) {   // raw accumulator out; the pool behind it adds this bias and applies the ReLU
          void* pb = nullptr;
          if (cudaMalloc(&pb, (size_t)mo.cout * 4) != cudaSuccess) return dvb::fail(DVB_ERR_CUDA, "cudaMalloc (bias) failed");
          net->allocs.push_back(pb);
          cudaMemcpy(pb, b_blob, (size_t)mo.cout * 4, cudaMemcpyHostToDevice);
          pool_bias[mo.dst] = static_cast<const float*>(pb);
        } else {
          memcpy(&bias_host[row0], b_blob, (size_t)mo.cout * 4);
        }
        const TensorBuf& md = rows_pool ? dst : net->tensors[net->tensor_index[mo.dst]];
        segs.push_back(OutSeg{(int)row0, md.C, mo.off, mo.no_act ? 0 : 1, md.ptr});
        blob_w_main = blob + pos;
        row0 += (size_t)mo.cout;
      }
    }
    cudaMemcpy(db, bias_host.data(), bbytes, cudaMemcpyHostToDevice);
    const float* conv_bias = static_cast<const float*>(db);
    if (merged) { o.cout = cout_total; o.no_act = 0; }
    else if (o.no_act) o.no_act = 1;
    const int relu_single = segs[0].relu;

    // ---- conv1 fused with preprocess + im2col (stem_conv1_kernel): WGS geometry (7 channels), precision 0
    if (is_stem && !split && net->C == kStemC && o.cout <= 32 && o.cout % 16 == 0 && cin_store == 64 && EnvInt("DVB_CNN_STEM_FUSED", 1)) {
      StemArgs& a = net->stem_args;
      memset(&a, 0, sizeof(a));
      a.out = dst.ptr; a.bias = static_cast<const float*>(db); a.w = static_cast<const __half*>(dw);
      a.H = net->H; a.W = net->W; a.Ho = Hout; a.Wo = Wout; a.cout = o.cout; a.out_cstride = dst.C;
      a.tiles_w = (Wout + 127) / 128;
      a.idesc = (1u << 4) | ((uint32_t)(o.cout >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      a.h_pitch = 1808;   // (2 * 127 + 3) * 7 = 1799 bytes per row segment -> 450 words -> 1800 halves, rounded up to 8
      net->stem_fused = true;
      if (o.cout == 32 && Wout <= 128 && EnvInt("DVB_CNN_STEM_ROWS", 0)) {
        // filter tile of stem_rows_kernel: rows [W0 | W2 | W0 | W1] (kernel rows; 32 filters each) x K = 32 (k = s * 7 + c, zero from 21)
        std::vector<__half> wt((size_t)128 * 32, __float2half(0.f));
        const __half* w = reinterpret_cast<const __half*>(blob_w_main);
        const int blk_r[4] = {0, 2, 0, 1};
        for (int blk = 0; blk < 4; ++blk)
          for (int co = 0; co < 32; ++co)
            for (int sx = 0; sx < 3; ++sx)
              for (int c = 0; c < net->C; ++c)
                wt[((size_t)blk * 32 + co) * 32 + sx * net->C + c] = w[(((size_t)co * 3 + blk_r[blk]) * 3 + sx) * blob_cin + c];
        void* dwt = nullptr;
        if (cudaMalloc(&dwt, wt.size() * sizeof(__half)) != cudaSuccess) return dvb::fail(DVB_ERR_CUDA, "cudaMalloc (weights) failed");
        net->allocs.push_back(dwt);
        cudaMemcpy(dwt, wt.data(), wt.size() * sizeof(__half), cudaMemcpyHostToDevice);
        Stem2Args& b = net->stem2_args;
        memset(&b, 0, sizeof(b));
        b.out = dst.ptr; b.bias = static_cast<const float*>(db); b.w = static_cast<const __half*>(dwt);
        b.H = net->H; b.W = net->W; b.Ho = Hout; b.Wo = Wout; b.out_cstride = dst.C;
        net->stem_rows = true;
      }
      macs_total += (double)Hout * Wout * o.cout * orig.kh * orig.kw * orig.cin;
      continue;
    }
    // ---- conv2 / conv3 (+ max pool): row-streaming kernel with the kernel rows stacked along N (see conv_rows_kernel)
    if (use_rows) {
      RowsLaunch rl;
      memset(&rl, 0, sizeof(rl));
      RowsArgs& a = rl.args;
      a.cin = cin_store; a.cout = o.cout;
      a.pad = o.same ? 1 : 0;
      a.J = Hin + 2 * a.pad;
      a.Hout = Hout; a.Wout = Wout;
      a.pool = rows_pool ? 1 : 0;
      a.Hp = rows_pool ? dst.H : 0; a.Wp = rows_pool ? dst.W : 0;
      a.out = dst.ptr; a.out_cstride = dst.C; a.out_coff = rows_pool ? ops[op_index + 1].off : o.off;
      a.bias = conv_bias;
      a.row_bytes = (uint32_t)cin_store * 2u;
      a.layout_type = cin_store == 64 ? 2u : 4u;
      a.sbo_bytes = 8u * a.row_bytes;
      a.idesc = (1u << 4) | ((uint32_t)((3 * o.cout) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      a.b_blk_bytes = (uint32_t)o.cout * a.row_bytes;
      a.b_tap_bytes = 5u * a.b_blk_bytes;
      a.a_buf_bytes = 128u * a.row_bytes;
      rl.smem = 1024 + (int)(3 * a.b_tap_bytes + 2 * kRowsRing * a.a_buf_bytes + 2 * 128 * o.cout * 2) + (4 * kRowsRing + 6) * 8 + o.cout * 4 + 64;
      rl.macs_per_image = (double)Hout * Wout * o.cout * 9 * orig.cin;
      if (rl.smem <= 227 * 1024) {
        // filters [Cout][3][3][Cin] -> [kw tap s][block: kernel row 2, 1, 0, 2, 1][Cout][Cin]: three consecutive blocks starting at
        // block b are the kernel rows (2 - b, 1 - b, -b) mod 3 - the rotation the accumulator ring needs at step t = 2 - b (mod 3)
        std::vector<__half> w2((size_t)3 * 5 * o.cout * cin_store, __float2half(0.f));
        const __half* w = reinterpret_cast<const __half*>(blob_w_main);
        const int blk_r[5] = {2, 1, 0, 2, 1};
        for (int sx = 0; sx < 3; ++sx)
          for (int blk = 0; blk < 5; ++blk)
            for (int co = 0; co < o.cout; ++co)
              memcpy(&w2[(((size_t)sx * 5 + blk) * o.cout + co) * cin_store], &w[(((size_t)co * 3 + blk_r[blk]) * 3 + sx) * blob_cin],
                     (size_t)blob_cin * sizeof(__half));
        void* dw5 = nullptr;
        if (cudaMalloc(&dw5, w2.size() * sizeof(__half)) != cudaSuccess) return dvb::fail(DVB_ERR_CUDA, "cudaMalloc (weights) failed");
        net->allocs.push_back(dw5);
        cudaMemcpy(dw5, w2.data(), w2.size() * sizeof(__half), cudaMemcpyHostToDevice);
        {
          const cuuint64_t dims[4] = {(cuuint64_t)src.C, (cuuint64_t)Win, (cuuint64_t)Hin, (cuuint64_t)net->max_batch};
          const cuuint64_t strides[3] = {(cuuint64_t)src.C * 2, (cuuint64_t)Win * src.C * 2, (cuuint64_t)Hin * Win * src.C * 2};
          const cuuint32_t box[4] = {(cuuint32_t)cin_store, 128, 1, 1};
          const cuuint32_t estr[4] = {1, 1, 1, 1};
          st = MakeMap(&rl.map_a, src.ptr, 4, dims, strides, box, estr, cin_store);
          if (st) return st;
        }
        {
          const cuuint64_t dims[3] = {(cuuint64_t)cin_store, (cuuint64_t)(5 * o.cout), 3};
          const cuuint64_t strides[2] = {(cuuint64_t)cin_store * 2, (cuuint64_t)5 * o.cout * cin_store * 2};
          const cuuint32_t box[3] = {(cuuint32_t)cin_store, (cuuint32_t)o.cout, 1};
          const cuuint32_t estr[3] = {1, 1, 1};
          st = MakeMap(&rl.map_b, dw5, 3, dims, strides, box, estr, cin_store);
          if (st) return st;
        }
        macs_total += rl.macs_per_image;
        net->steps.push_back(Step{3, (int)net->rows.size()});
        step_io.push_back({o.src, step_dsts});
        net->rows.push_back(rl);
        continue;
      }
      if (rows_pool) return dvb::fail(DVB_ERR_INTERNAL, "conv_rows_kernel: %d bytes of shared memory", rl.smem);
    }
    // ---- large stride-1 k x k layers: persistent halo-reusing kernel (see conv_halo_kernel)
    const bool halo_split = split && EnvInt("DVB_HALO_RULE", 1) == 2 && EnvInt("DVB_HALO_SPLIT", 0);   // precision 1 runs the halo kernel only under rule 2
    if ((!split || halo_split) && !is_stem && o.stride == 1 && o.kh * o.kw > 1 && Hout * Wout >= EnvInt("DVB_HALO_MIN_PIXELS", 250) && EnvInt("DVB_CNN_HALO", 1)) {
      HaloLaunch hl;
      memset(&hl, 0, sizeof(hl));
      HaloArgs& a = hl.args;
      const int taps = o.kh * o.kw;
      const int halo_rule = EnvInt("DVB_HALO_RULE", 1);
      int bk = cin_store % 64 == 0 ? 64 : cin_store % 32 == 0 ? 32 : 16;
      int k_channels = cin_store;
      if (halo_rule == 2) {
        // K block: the fewest 16-wide K steps over the layer's REAL input channels - a tensor stored wider than the layer's Cin carries
        // zero channels (48 stored as 64, 80 as 96) that the tap-by-tap kernels multiply along; narrow blocks also shrink the resident weights
        int best_units = 1 << 30;
        for (int cand = 64; cand >= 16; cand >>= 1) {
          if (cin_store % cand) continue;
          const int units = ((blob_cin + cand - 1) / cand) * (cand / 16);
          if (units < best_units) { best_units = units; bk = cand; }
        }
        const int force_halo_bk = EnvInt("DVB_HALO_FORCE_BK", 0);     // experiment switch
        if (force_halo_bk && cin_store % force_halo_bk == 0) bk = force_halo_bk;
        k_channels = blob_cin;
      }
      const int row_bytes = bk * 2;
      a.kh = o.kh; a.kw = o.kw;
      a.pad_h = o.same ? (o.kh - 1) / 2 : 0;
      a.pad_w = o.same ? (o.kw - 1) / 2 : 0;
      a.block_k = bk;
      a.cin_blocks = (k_channels + bk - 1) / bk;
      // slots per tile row: vertical tap offsets (r * P rows) must stay 1024-byte aligned
      // slots per tile row: the row pitch P * row_bytes keeps vertical taps 1024-byte aligned; P - kw + 1 slots are valid
      int bestP = 0; double best_eff = -1;
      for (int P = 1024 / row_bytes; P <= 128; P *= 2) {
        const int Ht = 128 / P;
        const int Wv = P - o.kw + 1;
        if (Wv < 1) continue;
        const double eff = (double)Hout * Wout / ((double)((Wout + Wv - 1) / Wv) * ((Hout + Ht - 1) / Ht) * 128.0);
        if (eff > best_eff + 0.04) { best_eff = eff; bestP = P; }   // small P = small halo: a wider row must pay > 4 % in fill
      }
      {
        const int force_p = EnvInt("DVB_HALO_FORCE_P", 0);            // experiment switch: slots per tile row (power of two)
        if (force_p >= 1024 / row_bytes && force_p <= 128 && (force_p & (force_p - 1)) == 0 && force_p - o.kw + 1 >= 1 && Hout * Wout > 1000) bestP = force_p;
      }
      a.P = bestP; a.Ht = 128 / bestP;
      a.Wv = a.P - o.kw + 1;
      a.tiles_w = (Wout + a.Wv - 1) / a.Wv;
      a.tiles_h = (Hout + a.Ht - 1) / a.Ht;
      a.Hout = Hout; a.Wout = Wout;
      const int Hh = a.Ht + o.kh;   // Ht + kh - 1 rows are needed; one spare row absorbs the kw-1 pixel overrun of the last tap
      const int planes = split ? 2 : 1;
      a.a_copy_bytes = (uint32_t)Hh * a.P * row_bytes;
      a.a_res_off = (a.a_copy_bytes + 1023u) & ~1023u;
      a.a_stage = (uint32_t)planes * a.a_res_off;
      // N block: the resident weight slice must leave room for the halo ring
      int bn = ChooseBlockN(o.cout);
      if (split && bn > 128) {   // [D0 | D1] in one instruction: N = 2 block_n <= 256
        for (int d = 128; d >= 16; d -= 16)
          if (o.cout % d == 0) { bn = d; break; }
      }
      auto b_total = [&](int n) { return (size_t)planes * a.cin_blocks * taps * (((size_t)n * row_bytes + 1023) & ~(size_t)1023); };
      while ((halo_rule == 2 ? b_total(bn) + 2 * a.a_stage > 216 * 1024 : b_total(bn) + 4 * a.a_stage > 200 * 1024) && bn > 16) {
        int next = 0;
        for (int d = bn - 16; d >= 16; d -= 16)
          if (o.cout % d == 0) { next = d; break; }
        if (!next) break;
        bn = next;
      }
      a.block_n = bn; a.n_blocks = o.cout / bn;
      a.b_tile = (uint32_t)((bn * row_bytes + 1023) & ~1023);
      a.b_total_bytes = (uint32_t)a.cin_blocks * taps * bn * row_bytes;   // bytes the TMA delivers (per plane)
      const size_t b_smem = (size_t)planes * a.cin_blocks * taps * a.b_tile;
      const int acc_cols = planes * bn;                                   // TMEM columns of one tile
      // T tiles in flight = T independent accumulation chains (measured issue interval per MMA, N <= 64: 222 cycles
      // with 1 chain, 80 with 4, 46 with 8).  Two TMEM buffers of T accumulators when 2*T*bn <= 512 columns, else one.
      // Rule 2 (round 2, after the issue path was fixed - one accumulation chain now runs at the tensor pipe's own interval, see
      // DESIGN.md 4.0): what bounds the tap-by-tap kernels on these layers is the SM's ingest from L2 (about 36-40 B per clock:
      // 9 taps x (A tile + weight tile) per 128 pixels), so the halo kernel pays whenever its weights fit, with T = 1 or 2 tiles in
      // flight (2 when TMEM holds two double-buffered accumulators and the halo ring has 4 slots) - any N block count.
      const int avail_stages = (int)((216 * 1024 - (long)b_smem) / (long)a.a_stage);
      int T;
      if (halo_rule == 2) {
        T = (4 * acc_cols <= 512 && avail_stages >= 4) ? 2 : 1;
        T = std::max(1, std::min(T, EnvInt("DVB_HALO_T", 8)));
        a.T = T;
        a.nbuf = 2 * a.T * acc_cols <= 512 ? 2 : 1;
        a.stages = std::max(1, std::min(std::min(2 * kMaxStages, std::max(4, 2 * a.T)), avail_stages));
      } else {
      T = std::min(kMaxGroup, 512 / bn);
      T = T >= 8 ? 8 : T >= 4 ? 4 : T;
      T = std::min(T, EnvInt("DVB_HALO_T", 8));
      while (T > 1 && b_smem + (size_t)(T + 2) * a.a_stage > 216 * 1024) T = T > 4 ? 4 : T - 1;
      a.T = std::max(1, T);
      if (2 * a.T * bn > 512 && a.T == 8 && EnvInt("DVB_HALO_PREFER_DB", 1)) a.T = 4;   // measured: T=4 double-buffered beats T=8 single
      a.nbuf = (2 * a.T * bn <= 512 && EnvInt("DVB_HALO_NBUF", 2) == 2) ? 2 : 1;
      a.stages = std::min(2 * kMaxStages, std::max(a.T, std::min(2 * a.T, (int)((216 * 1024 - (long)b_smem) / (long)a.a_stage))));
      }
      // epilogue work units: T tiles x n_split column ranges over the 4 warp groups of a TMEM lane quarter
      a.n_split = 1;
      for (int ns = std::max(1, 4 / a.T); ns >= 1; --ns)
        if (bn % ns == 0 && (bn / ns) % 16 == 0) { a.n_split = ns; break; }
      a.tmem_cols = TmemCols(a.nbuf * a.T * acc_cols);
      a.out = dst.ptr; a.out_res = dst.ptr_res; a.out_cstride = dst.C; a.out_coff = o.off; a.relu = relu_single;
      a.bias = conv_bias;
      a.idesc = (1u << 4) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      a.idesc_cat = (1u << 4) | ((uint32_t)((2 * bn) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
      a.layout_type = bk == 64 ? 2u : bk == 32 ? 4u : 6u;
      a.sbo_bytes = 8u * (uint32_t)row_bytes;
      hl.smem = (int)(b_smem + (size_t)a.stages * a.a_stage) + 1024 + 512 + bn * 4;
      hl.macs_per_image = (double)Hout * Wout * o.cout * o.kh * o.kw * o.cin;
      // Only worth it when >= 4 double-buffered accumulation chains fit in TMEM (N block <= 64); wider layers (conv5,
      // N = 192) measured slower here than with the tap-by-tap kernel and stay there.
      const bool halo_ok = halo_rule == 2 ? (a.stages >= std::max(2, a.T) && a.nbuf == 2 && (bn >= 64 || bn == o.cout || split) && bn >= 32 &&
                                             a.b_tile == (uint32_t)(bn * row_bytes) && (!split || 2 * bn <= 256))
                                           : (a.stages >= a.T && a.T >= 4 && a.nbuf == 2 && a.n_blocks == 1);
      if (a.tmem_cols <= 512 && hl.smem <= 227 * 1024 && halo_ok) {
        // weights [Cout][taps][Cin] -> [taps][Cout][Cin] so that one (tap, N block, Cin block) is a canonical K-major tile
        std::vector<__half> w2((size_t)taps * o.cout * cin_store, __float2half(0.f));
        const __half* w = reinterpret_cast<const __half*>(blob_w_main);
        for (int co = 0; co < o.cout; ++co)
          for (int t = 0; t < taps; ++t)
            memcpy(&w2[((size_t)t * o.cout + co) * cin_store], &w[((size_t)co * taps + t) * blob_cin], (size_t)blob_cin * sizeof(__half));
        cudaMemcpy(dw, w2.data(), wbytes, cudaMemcpyHostToDevice);
        if (split) {   // the residual plane of the filters, same re-layout
          const __half* wr = reinterpret_cast<const __half*>(blob_w_main + blob_wbytes);
          for (int co = 0; co < o.cout; ++co)
            for (int t = 0; t < taps; ++t)
              memcpy(&w2[((size_t)t * o.cout + co) * cin_store], &wr[((size_t)co * taps + t) * blob_cin], (size_t)blob_cin * sizeof(__half));
          cudaMemcpy(dw_res, w2.data(), wbytes, cudaMemcpyHostToDevice);
        }
        {
          const cuuint64_t dims[4] = {(cuuint64_t)src.C, (cuuint64_t)Win, (cuuint64_t)Hin, (cuuint64_t)net->max_batch};
          const cuuint64_t strides[3] = {(cuuint64_t)src.C * 2, (cuuint64_t)Win * src.C * 2, (cuuint64_t)Hin * Win * src.C * 2};
          const cuuint32_t box[4] = {(cuuint32_t)bk, (cuuint32_t)a.P, (cuuint32_t)Hh, 1};
          const cuuint32_t estr[4] = {1, 1, 1, 1};
          st = MakeMap(&hl.map_a, src.ptr, 4, dims, strides, box, estr, bk);
          if (st) return st;
          hl.map_a_res = hl.map_a;
          if (split) {
            st = MakeMap(&hl.map_a_res, src.ptr_res, 4, dims, strides, box, estr, bk);
            if (st) return st;
          }
        }
        {
          const cuuint64_t dims[3] = {(cuuint64_t)cin_store, (cuuint64_t)o.cout, (cuuint64_t)taps};
          const cuuint64_t strides[2] = {(cuuint64_t)cin_store * 2, (cuuint64_t)o.cout * cin_store * 2};
          const cuuint32_t box[3] = {(cuuint32_t)bk, (cuuint32_t)bn, 1};
          const cuuint32_t estr[3] = {1, 1, 1};
          st = MakeMap(&hl.map_b, dw, 3, dims, strides, box, estr, bk);
          if (st) return st;
          hl.map_b_res = hl.map_b;
          if (split) {
            st = MakeMap(&hl.map_b_res, dw_res, 3, dims, strides, box, estr, bk);
            if (st) return st;
          }
        }
        macs_total += hl.macs_per_image;
        net->steps.push_back(Step{2, (int)net->halos.size()});
        step_io.push_back({o.src, step_dsts});
        net->halos.push_back(hl);
        continue;
      }
    }

    ConvLaunch cl;
    memset(&cl, 0, sizeof(cl));
    ConvArgs& a = cl.args;
    a.kh = o.kh; a.kw = o.kw; a.stride = o.stride;
    a.pad_h = o.same ? (o.kh - 1) / 2 : 0;
    a.pad_w = o.same ? (o.kw - 1) / 2 : 0;
    int bk = force_bk ? force_bk : (cin_store % 64 == 0 ? 64 : cin_store % 32 == 0 ? 32 : 16);
    if (cin_store < bk) bk = cin_store >= 32 ? 32 : 16;
    a.block_k = bk;
    a.cin_blocks = (cin_store + bk - 1) / bk;
    // 1x1 stride-1 convolutions have no halo: all N*H*W pixels are flattened into one dimension and every
    // M tile is a full 128 rows.
    const bool flat = o.kh == 1 && o.kw == 1 && o.stride == 1;
    cl.flat = flat;
    cl.pixels_per_image = Hout * Wout;
    const TileChoice tc = flat ? TileChoice{128, 1, 1} : ChooseTile(Hout, Wout, o.stride);
    a.Wt = tc.Wt; a.Ht = tc.Ht; a.Nt = tc.Nt;
    a.tiles_w = (Wout + tc.Wt - 1) / tc.Wt;
    a.tiles_h = (Hout + tc.Ht - 1) / tc.Ht;
    a.Hout = Hout; a.Wout = Wout;
    // BLOCK_N: the whole Cout when it fits one instruction (<= 256), except that layers with few M tiles are
    // split further so that the grid still covers >= 2 CTAs on each of the 148 SMs.
    {
      const long m_tiles = flat ? ((long)net->max_batch * Hout * Wout + 127) / 128
                                : (long)a.tiles_w * a.tiles_h * ((net->max_batch + tc.Nt - 1) / tc.Nt);
      int bn = ChooseBlockN(o.cout);
      if (split && bn > 128) {   // two accumulators + {main, res} operand tiles per stage: keep N <= 128
        int best = 16;
        for (int d = 128; d >= 16; d -= 16)
          if (o.cout % d == 0) { best = d; break; }
        bn = best;
      }
      // Persistent kernel where it measured faster (B200, 2048 images): 64-wide K blocks, N block >= 160 and at least four
      // tiles per SM (1x1 768->192/160: 56 -> 42 us, 1x7/7x1 192->192: 66 -> 61 us).  Narrow N blocks or 16/32-wide K blocks
      // leave its single accumulation chain per SM latency-bound (96->96 3x3: 141 -> 234 us), and on the 1x5 maps of
      // mixed8-10 a few hundred tiles quantise badly over 148 CTAs; those stay on the one-tile-per-CTA kernel, where
      // 3-4 co-resident CTAs give 3-4 independent chains.
      {
        const int mode = EnvInt("DVB_CNN_PERSIST", 1);   // 0 never, 1 by rule, 2 always
        const long tiles = m_tiles * (o.cout / bn);
        cl.persist = !split && (mode == 2 || (mode == 1 && bk == 64 && bn >= EnvInt("DVB_PERSIST_MIN_N", 160) && tiles >= (long)EnvInt("DVB_PERSIST_MIN_TILES_PER_SM", 4) * net->num_sms));
      }
      const long want_ctas = cl.persist ? 0L : 4L * net->num_sms;   // the persistent kernel keeps the widest N block
      while (m_tiles * (o.cout / bn) < want_ctas && bn > 64) {
        int next = 0;
        for (int d = bn - 16; d >= 32; d -= 16)
          if (o.cout % d == 0) { next = d; break; }
        if (!next) break;
        bn = next;
      }
      a.block_n = bn;
    }
    a.tmem_cols = TmemCols(split || cl.persist ? 2 * a.block_n : a.block_n);
    cl.n_blocks = o.cout / a.block_n; cl.cout = o.cout;
    a.out = dst.ptr; a.out_cstride = dst.C; a.out_coff = o.off; a.relu = relu_single;
    a.out_res = dst.ptr_res;
    if (merged) {
      a.n_segs = (int)segs.size();
      for (size_t k = 0; k < segs.size(); ++k) a.segs[k] = segs[k];
    }
    a.skip_a_res = is_stem ? 1 : 0;   // the preprocessed input is exact in fp16: its residual plane is zero
    a.dbg = EnvInt("DVB_CNN_DBG", 0);
    a.bias = conv_bias;
    // instruction descriptor (cute/arch/mma_sm100_desc.hpp InstrDescriptor): D=F32, A=B=F16, K-major, M=128
    a.idesc = (1u << 4) | ((uint32_t)(a.block_n >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    a.layout_type = bk == 64 ? 2u : bk == 32 ? 4u : 6u;
    a.sbo_bytes = 8u * (uint32_t)bk * 2u;
    const int rows = tc.Wt * tc.Ht * tc.Nt;
    a.a_bytes = (uint32_t)rows * bk * 2;
    a.b_bytes = (uint32_t)a.block_n * bk * 2;
    a.a_stage = 128u * bk * 2;
    a.b_stage = ((uint32_t)a.block_n * bk * 2 + 1023u) & ~1023u;
    if (split) {
      a.idesc_cat = (a.b_bytes == a.b_stage && 2 * a.block_n <= 256 && EnvInt("DVB_CNN_SPLIT_CAT", 1))
                        ? ((1u << 4) | ((uint32_t)((2 * a.block_n) >> 3) << 17) | ((uint32_t)(128 >> 4) << 24)) : 0u;
      a.a_res_off = a.a_stage; a.b_res_off = a.b_stage; a.a_stage *= 2; a.b_stage *= 2;
    }
    // Pipeline depth: as deep as fits in ~108 KB so that two CTAs (one in its epilogue, one issuing MMAs) share an SM.
    {
      const int stage_bytes = (int)(a.a_stage + a.b_stage);
      const int num_kb = o.kh * o.kw * a.cin_blocks;
      // Occupancy beats pipeline depth here (measured): aim for ~4 co-resident CTAs of 2-4 stages each.
      const int target_kb = split ? 200 : EnvInt("DVB_CNN_SMEM_KB", 72);
      const int max_stages = std::min(EnvInt("DVB_CNN_MAX_STAGES", 3), kMaxStages);
      int stages = (target_kb * 1024 - 1280) / stage_bytes;
      stages = std::max(2, std::min(stages, max_stages));
      stages = std::max(1, std::min(stages, num_kb));
      a.stages = EnvInt("DVB_CNN_STAGES", 0) > 0 ? std::min(EnvInt("DVB_CNN_STAGES", 0), kMaxStages) : stages;
      cl.smem = a.stages * stage_bytes + 1024 + 256 + a.block_n * 4;
      if (cl.persist) {   // one CTA per SM: the ring takes what the SM has
        a.stages = std::max(2, std::min(kMaxStages, (EnvInt("DVB_PERSIST_SMEM_KB", 200) * 1024) / stage_bytes));
        cl.smem = a.stages * stage_bytes + 1024 + 256 + o.cout * 4;
        if (cl.smem > 227 * 1024) return dvb::fail(DVB_ERR_INTERNAL, "conv %zu: %d bytes of shared memory", net->convs.size(), cl.smem);
      }
    }
    cl.macs_per_image = (double)Hout * Wout * o.cout * orig.kh * orig.kw * orig.cin;
    macs_total += cl.macs_per_image;
    // --- tensor maps
    {
      cuuint64_t dims[4] = {(cuuint64_t)src.C, (cuuint64_t)Win, (cuuint64_t)Hin, (cuuint64_t)net->max_batch};
      cuuint64_t strides[3] = {(cuuint64_t)src.C * 2, (cuuint64_t)Win * src.C * 2, (cuuint64_t)Hin * Win * src.C * 2};
      if (flat) {
        dims[1] = (cuuint64_t)Win * Hin * net->max_batch; dims[2] = 1; dims[3] = 1;
        strides[1] = dims[1] * src.C * 2; strides[2] = strides[1];
      }
      // With elementStrides = s the box is stated in UN-strided input elements and the TMA delivers
      // ceil(box / s) of them (measured on B200: box = Wt loads too few bytes and the mbarrier never
      // completes; box = Wt * s delivers exactly Wt).
      const cuuint32_t bw = tc.Wt * o.stride, bh = tc.Ht * o.stride;
      const cuuint32_t box[4] = {(cuuint32_t)bk, bw, bh, (cuuint32_t)tc.Nt};
      const cuuint32_t estr[4] = {1, (cuuint32_t)o.stride, (cuuint32_t)o.stride, 1};
      st = MakeMap(&cl.map_a, src.ptr, 4, dims, strides, box, estr, bk);
      if (st) return st;
      cl.map_a_res = cl.map_a;
      if (split) {
        st = MakeMap(&cl.map_a_res, src.ptr_res, 4, dims, strides, box, estr, bk);
        if (st) return st;
      }
    }
    {
      const cuuint64_t dims[3] = {(cuuint64_t)cin_store, (cuuint64_t)(o.kh * o.kw), (cuuint64_t)o.cout};
      const cuuint64_t strides[2] = {(cuuint64_t)cin_store * 2, (cuuint64_t)o.kh * o.kw * cin_store * 2};
      const cuuint32_t box[3] = {(cuuint32_t)bk, 1, (cuuint32_t)a.block_n};
      const cuuint32_t estr[3] = {1, 1, 1};
      st = MakeMap(&cl.map_b, dw, 3, dims, strides, box, estr, bk);
      if (st) return st;
      cl.map_b_res = cl.map_b;
      if (split) {
        st = MakeMap(&cl.map_b_res, dw_res, 3, dims, strides, box, estr, bk);
        if (st) return st;
      }
    }
    // CTA-pair variant (cta_group::2): same layers as the persistent kernel, when asked for
    // CTA pairs (cta_group::2, M = 256): DVB_CNN_PAIR = 0 never, 1 every persistent layer, 2 (default) by the measured rule - the
    // single-destination k x k layers with a 192-wide N block (1x7 / 7x1 192->192: 93 -> 84 us per 4096 images; the merged 1x1 GEMMs with
    // their multi-destination epilogue measured 8 % slower as pairs, 128->192 the same).
    {
      const int pair_mode = EnvInt("DVB_CNN_PAIR", 2);
      cl.pair = cl.persist && a.block_n % 16 == 0 &&
                (pair_mode == 1 || (pair_mode == 2 && !merged && a.block_n == 192 && o.kh * o.kw > 1 && a.cin_blocks >= 3) ||
                 (pair_mode == 3 && !merged && a.block_n >= 128 && o.kh * o.kw > 1 && a.cin_blocks >= 2));
    }
    if (cl.pair) {
      PairArgs& q2 = cl.pair_args;
      q2.idesc = (1u << 4) | ((uint32_t)(a.block_n >> 3) << 17) | ((uint32_t)(256 >> 4) << 24);
      q2.b_half_bytes = (uint32_t)(a.block_n / 2) * bk * 2;
      q2.b_half_stage = (q2.b_half_bytes + 1023u) & ~1023u;
      const int stage_bytes = (int)(a.a_stage + q2.b_half_stage);
      q2.stages = std::max(2, std::min(kMaxStages, (EnvInt("DVB_PERSIST_SMEM_KB", 200) * 1024) / stage_bytes));
      cl.pair_smem = q2.stages * stage_bytes + 1024 + 256 + o.cout * 4;
      const cuuint64_t dims[3] = {(cuuint64_t)cin_store, (cuuint64_t)(o.kh * o.kw), (cuuint64_t)o.cout};
      const cuuint64_t strides[2] = {(cuuint64_t)cin_store * 2, (cuuint64_t)o.kh * o.kw * cin_store * 2};
      const cuuint32_t box[3] = {(cuuint32_t)bk, 1, (cuuint32_t)(a.block_n / 2)};
      const cuuint32_t estr[3] = {1, 1, 1};
      st = MakeMap(&cl.map_b_half, dw, 3, dims, strides, box, estr, bk);
      if (st) return st;
    }
    cl.grid = dim3(1, (unsigned)(o.cout / a.block_n), 1);
    net->steps.push_back(Step{0, (int)net->convs.size()});
    step_io.push_back({o.src, step_dsts});
    net->convs.push_back(cl);
  }
  pos = conv_pos[n_conv];
  // --- lanes: chains of single-producer/single-consumer steps stay on one stream, every other consumer starts a new one
  {
    net->n_lanes = std::max(1, std::min(kMaxLanes, EnvInt("DVB_CNN_LANES", kMaxLanes)));
    std::map<std::string, std::vector<int>> writers;   // tensor -> steps writing (a slice of) it; -1 = stem_patch_kernel
    writers["input"].push_back(-1);
    if (net->stem_fused) writers["s1"].push_back(-1);
    std::map<int, bool> continued;
    int rr = 1;
    auto lane_of = [&](int st_i) { return st_i < 0 ? 0 : net->steps[st_i].lane; };
    for (size_t i = 0; i < net->steps.size(); ++i) {
      Step& stp = net->steps[i];
      const std::vector<int>& w = writers[step_io[i].first];
      if (w.size() == 1 && !continued[w[0]]) { stp.lane = lane_of(w[0]); continued[w[0]] = true; }
      else { stp.lane = rr % net->n_lanes; ++rr; }
      for (int d : w)
        if (d >= 0 && lane_of(d) != stp.lane) { stp.deps.push_back(d); net->steps[d].record = true; }
      for (const std::string& d : step_io[i].second) writers[d].push_back((int)i);
    }
    for (int d : writers["mixed10"])
      if (lane_of(d) != 0) { net->tail_deps.push_back(d); net->steps[d].record = true; }
    for (Step& stp : net->steps)
      if (stp.record && cudaEventCreateWithFlags(&stp.event, cudaEventDisableTiming) != cudaSuccess)
        return dvb::fail(DVB_ERR_CUDA, "cudaEventCreate failed");
    for (int l = 1; l < net->n_lanes; ++l)
      if (cudaStreamCreateWithFlags(&net->lane_streams[l], cudaStreamNonBlocking) != cudaSuccess)
        return dvb::fail(DVB_ERR_CUDA, "cudaStreamCreate failed");
  }
  // --- head
  const size_t dwb = 2048 * 3 * sizeof(float), dbb = 3 * sizeof(float);
  if (pos + (int64_t)(dwb + dbb) != blob_bytes) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "weights blob size mismatch (%lld of %lld bytes consumed before the head)", (long long)pos, (long long)blob_bytes);
  if (ch["mixed10"] != 2048) return dvb::fail(DVB_ERR_INTERNAL, "backbone does not end in 2048 channels");
  cudaMalloc(&net->d_dense_w, dwb); cudaMalloc(&net->d_dense_b, dbb);
  cudaMemcpy(net->d_dense_w, blob + pos, dwb, cudaMemcpyHostToDevice);
  cudaMemcpy(net->d_dense_b, blob + pos + dwb, dbb, cudaMemcpyHostToDevice);
  cudaMalloc(&net->d_pooled, (size_t)net->max_batch * 2048 * sizeof(float));
  net->feat_tensor = net->tensor_index["mixed10"];
  net->flops_per_image = 2.0 * macs_total;
  int max_smem = 0;
  for (auto& c : net->convs) max_smem = std::max(max_smem, c.smem);
  int max_pair = 0;
  for (const ConvLaunch& c : net->convs)
    if (c.pair) max_pair = std::max(max_pair, c.pair_smem);
  if (max_pair && cudaFuncSetAttribute(conv_gemm_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_pair) != cudaSuccess)
    return dvb::fail(DVB_ERR_CUDA, "cannot reserve %d bytes of shared memory (pair kernel)", max_pair);
  int max_persist = 0;
  for (auto& c : net->convs)
    if (c.persist) max_persist = std::max(max_persist, c.smem);
  if (max_persist && cudaFuncSetAttribute(conv_gemm_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, max_persist) != cudaSuccess)
    return dvb::fail(DVB_ERR_CUDA, "cannot reserve %d bytes of shared memory (persistent kernel)", max_persist);
  if ((split ? cudaFuncSetAttribute(conv_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem)
             : cudaFuncSetAttribute(conv_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem)) != cudaSuccess)
    return dvb::fail(DVB_ERR_CUDA, "cannot reserve %d bytes of shared memory", max_smem);
  // several CTAs per SM are the point of these two kernels: ask for the largest shared-memory carveout (the default heuristic may
  // settle for one that fits fewer blocks)
  cudaFuncSetAttribute(conv_gemm_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  cudaFuncSetAttribute(conv_gemm_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  cudaFuncSetAttribute(stem_conv1_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  cudaFuncSetAttribute(stem_conv1_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
  if (net->stem_rows && cudaFuncSetAttribute(stem_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                             1024 + kS1ARing * 8192 + 8192 + kS1RawSlots * kS1RawPitch + (2 * kS1ARing + 4) * 8 + 32 * 4 + 64) != cudaSuccess)
    return dvb::fail(DVB_ERR_CUDA, "cannot reserve shared memory (stem rows kernel)");
  int max_rows = 0;
  for (auto& r : net->rows) max_rows = std::max(max_rows, r.smem);
  if (max_rows && (cudaFuncSetAttribute(conv_rows_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_rows) != cudaSuccess ||
                   cudaFuncSetAttribute(conv_rows_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_rows) != cudaSuccess))
    return dvb::fail(DVB_ERR_CUDA, "cannot reserve %d bytes of shared memory (rows kernel)", max_rows);
  int max_halo = 0;
  for (auto& h : net->halos) max_halo = std::max(max_halo, h.smem);
  if (max_halo && (cudaFuncSetAttribute(conv_halo_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_halo) != cudaSuccess ||
                   cudaFuncSetAttribute(conv_halo_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_halo) != cudaSuccess))
    return dvb::fail(DVB_ERR_CUDA, "cannot reserve %d bytes of shared memory (halo kernel)", max_halo);
  for (auto& h : net->halos) {
    int occ = 1;
    if (net->precision == 1) cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, conv_halo_kernel<true>, kHaloThreads, h.smem);
    else cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, conv_halo_kernel<false>, kHaloThreads, h.smem);
    occ = std::max(1, std::min(occ, 512 / h.args.tmem_cols));
    h.ctas_per_nblock = std::max(1, net->num_sms * occ / h.args.n_blocks);
  }
  // Plan listing: which kernel runs each layer (dst = first tensor the step writes).  A [conv] line also gives the M tile box
  // (Wt x Ht x Nt output pixels, flat = all pixels of the chunk in one row) and the M tile count at max_batch images.
  if (EnvInt("DVB_CNN_LIST", 0)) {
    fprintf(stderr, "[stem] %s\n", net->stem_rows ? "rows" : net->stem_fused ? "fused" : "patch");
    for (size_t si = 0; si < net->steps.size(); ++si) {
      const Step& stp = net->steps[si];
      const char* dst = step_io[si].second[0].c_str();
      if (stp.kind == 0) {
        const ConvLaunch& c = net->convs[stp.index];
        const ConvArgs& a = c.args;
        const long m_tiles = c.flat ? ((long)net->max_batch * c.pixels_per_image + 127) / 128
                                    : (long)a.tiles_w * a.tiles_h * ((net->max_batch + a.Nt - 1) / a.Nt);
        fprintf(stderr, "[conv %d] %dx%d cin_blocks=%d bk=%d N=%d n_blocks=%d persist=%d pair=%d stages=%d dst=%s out=%dx%d box=%dx%dx%d flat=%d m_tiles=%ld\n",
                stp.index, a.kh, a.kw, a.cin_blocks, a.block_k, a.block_n, c.n_blocks, (int)c.persist, (int)c.pair, a.stages, dst, a.Hout, a.Wout, a.Wt, a.Ht,
                a.Nt, (int)c.flat, m_tiles);
      } else if (stp.kind == 2) {
        const HaloArgs& h = net->halos[stp.index].args;
        fprintf(stderr, "[halo %d] %dx%d %dx%d cin_blocks=%d bk=%d N=%d n_blocks=%d P=%d Ht=%d T=%d nbuf=%d stages=%d n_split=%d smem=%d dst=%s\n", stp.index, h.kh,
                h.kw, h.Hout, h.Wout, h.cin_blocks, h.block_k, h.block_n, h.n_blocks, h.P, h.Ht, h.T, h.nbuf, h.stages, h.n_split, net->halos[stp.index].smem, dst);
      } else if (stp.kind == 3) {
        const RowsArgs& r = net->rows[stp.index].args;
        fprintf(stderr, "[rows %d] 3x3 %dx%d cout=%d pool=%d dst=%s\n", stp.index, r.Hout, r.Wout, r.cout, r.pool, dst);
      } else {   // the kernel ForwardChunkLaunches picks for this pool (same switches, read again there)
        const PoolLaunch& p = net->pools[stp.index];
        const char* kernel = p.mode == 0 ? (!p.in_res && EnvInt("DVB_CNN_MAXPOOL_H2", 1) ? "maxpool3x3s2_h2" : "pool3x3")
                                         : (!p.in_res && p.Hout == p.Hin && p.Wout == p.Win && EnvInt("DVB_CNN_AVGPOOL_FLAT", 1) ? "avgpool3x3s1" : "pool3x3");
        fprintf(stderr, "[pool %d] %s %dx%d -> %dx%d bias=%d kernel=%s dst=%s\n", stp.index, p.mode ? "avg" : "max", p.Hin, p.Win, p.Hout, p.Wout,
                (int)(p.bias != nullptr), kernel, dst);
      }
    }
  }
  if (cudaDeviceSynchronize() != cudaSuccess) return dvb::fail(DVB_ERR_CUDA, "weight upload failed: %s", cudaGetErrorString(cudaGetLastError()));
  return DVB_OK;
}

int ForwardChunkLaunches(DvbCnn* net, const uint8_t* images, int n, float* probs, cudaStream_t s0);

// One chunk's forward = ~80 dependent launches on four lanes.  DVB_CNN_GRAPH=1: the launch sequence of a (images, probs, n) triple is
// captured once into a CUDA graph (the lanes fork from and join the caller's stream through the steps' events) and replayed, so that the
// inter-kernel launch gaps and the host's launch work disappear from the loop; callers that reuse their buffers (the bench loop, the fused
// caller's batch buffer) hit the cache every time.  Anything that cannot be captured falls back to direct launches for good.
int ForwardChunk(DvbCnn* net, const uint8_t* images, int n, float* probs, cudaStream_t s0) {
  if (!net->use_graphs || s0 == nullptr) return ForwardChunkLaunches(net, images, n, probs, s0);   // (the legacy default stream cannot be captured)
  for (DvbCnn::ChunkGraph& g : net->graphs)
    if (g.images == images && g.probs == probs && g.n == n) {
      DVB_CUDA(cudaGraphLaunch(g.exec, s0));
      net->launches += g.launches;
      return DVB_OK;
    }
  const int64_t before = net->launches;
  if (cudaStreamBeginCapture(s0, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
    cudaGetLastError();
    net->use_graphs = false;
    return ForwardChunkLaunches(net, images, n, probs, s0);
  }
  const int st = ForwardChunkLaunches(net, images, n, probs, s0);
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  const cudaError_t e1 = cudaStreamEndCapture(s0, &graph);
  const cudaError_t e2 = (e1 == cudaSuccess && st == DVB_OK) ? cudaGraphInstantiate(&exec, graph, 0) : cudaErrorUnknown;
  if (graph) cudaGraphDestroy(graph);
  if (e2 != cudaSuccess) {
    cudaGetLastError();
    net->use_graphs = false;
    net->launches = before;
    return ForwardChunkLaunches(net, images, n, probs, s0);
  }
  if (net->graphs.size() >= 16) { cudaGraphExecDestroy(net->graphs.front().exec); net->graphs.erase(net->graphs.begin()); }
  net->graphs.push_back({images, probs, n, exec, net->launches - before});
  DVB_CUDA(cudaGraphLaunch(exec, s0));
  return DVB_OK;
}

int ForwardChunkLaunches(DvbCnn* net, const uint8_t* images, int n, float* probs, cudaStream_t s0) {
  const TensorBuf& in = net->tensors[0];
  cudaStream_t s = s0;
  if (net->stem_rows) {
    Stem2Args a = net->stem2_args;
    a.in = images; a.n_images = n;
    a.total_bytes = (long long)n * net->H * net->W * net->C;
    const int smem = 1024 + kS1ARing * 8192 + 8192 + kS1RawSlots * kS1RawPitch + (2 * kS1ARing + 4) * 8 + 32 * 4 + 64;
    stem_rows_kernel<<<(unsigned)std::min(net->num_sms, n), kS1Threads, smem, s>>>(a);
  } else if (net->stem_fused) {
    StemArgs a = net->stem_args;
    a.in = images; a.n_images = n;
    a.total_bytes = (long long)n * net->H * net->W * net->C;
    const long long tiles = (long long)n * a.Ho * a.tiles_w;
    const int smem = 1024 + 16384 + 4096 + 3 * a.h_pitch * 2 + 2 * 3 * kStemRawPitch + 48 + a.cout * 4;
    const int occ = EnvInt("DVB_STEM_CTAS_PER_SM", 4);   // 64 registers x 256 threads -> 4 resident CTAs per SM
    const unsigned grid = (unsigned)std::min<long long>(tiles, (long long)net->num_sms * occ);
    if (EnvInt("DVB_STEM_PIPE", 0)) stem_conv1_kernel<true><<<grid, kStemThreads, smem, s>>>(a);
    else stem_conv1_kernel<false><<<grid, kStemThreads, smem, s>>>(a);
  } else {
    const int groups = (net->stem_Ho + kPatchRows - 1) / kPatchRows;
    const int row_pitch = (net->W * net->C + 3 + 15) & ~15;
    const int smem = (2 * kPatchRows + 1) * row_pitch + 2 * net->stem_Kp;
    stem_patch_kernel<<<(unsigned)((long long)n * groups), 256, smem, s>>>(images, in.ptr, n, net->H, net->W, net->C, net->stem_Ho,
                                                                          net->stem_Wo, net->stem_Kp);
  }
  net->launches++;
  for (const Step& stp : net->steps) {
    cudaStream_t s = stp.lane == 0 ? s0 : net->lane_streams[stp.lane];
    for (int d : stp.deps) cudaStreamWaitEvent(s, net->steps[d].event, 0);
    if (stp.kind == 3) {
      RowsLaunch& rl = net->rows[stp.index];
      RowsArgs a = rl.args;
      a.n_images = n;
      static long long* d_rtrace = nullptr;
      const bool tracing = EnvInt("DVB_CNN_TRACE", 0) != 0;
      if (tracing && !d_rtrace) cudaMalloc(&d_rtrace, 48 * 8 * sizeof(long long));
      if (tracing) { cudaMemsetAsync(d_rtrace, 0, 48 * 8 * sizeof(long long), s); a.trace = d_rtrace; }
      if (a.pool) conv_rows_kernel<true><<<(unsigned)std::min(net->num_sms, n), kRowsThreads, rl.smem, s>>>(rl.map_a, rl.map_b, a);
      else conv_rows_kernel<false><<<(unsigned)std::min(net->num_sms, n), kRowsThreads, rl.smem, s>>>(rl.map_a, rl.map_b, a);
      if (tracing) {
        std::vector<long long> h(48 * 8);
        cudaStreamSynchronize(s);
        cudaMemcpy(h.data(), d_rtrace, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
        fprintf(stderr, "[rows trace] layer %d cout=%d pool=%d: step: mma_ready mma_committed acc_done_seen drained stored (cycles rel. to step 0)\n", stp.index, a.cout, a.pool);
        for (int i = 0; i < 40; ++i) {
          fprintf(stderr, "  step %2d:", i);
          for (int e = 0; e < 7; ++e) fprintf(stderr, " %8lld", h[i * 8 + e] ? h[i * 8 + e] - h[0] : -1);
          fprintf(stderr, "\n");
        }
      }
    } else if (stp.kind == 2) {
      HaloLaunch& hl = net->halos[stp.index];
      HaloArgs a = hl.args;
      a.n_images = n;
      const int total_tiles = n * a.tiles_w * a.tiles_h;
      const int G = std::min(hl.ctas_per_nblock, (total_tiles + a.T - 1) / a.T);
      static long long* d_trace = nullptr;
      const bool tracing = EnvInt("DVB_CNN_TRACE", 0) != 0;
      if (tracing && !d_trace) { cudaMalloc(&d_trace, 64 * 8 * sizeof(long long)); }
      if (tracing) { cudaMemsetAsync(d_trace, 0, 64 * 8 * sizeof(long long), s); a.trace = d_trace; }
      if (net->precision == 1)
        conv_halo_kernel<true><<<(unsigned)(G * a.n_blocks), kHaloThreads, hl.smem, s>>>(hl.map_a, hl.map_b, hl.map_a_res, hl.map_b_res, a);
      else
        conv_halo_kernel<false><<<(unsigned)(G * a.n_blocks), kHaloThreads, hl.smem, s>>>(hl.map_a, hl.map_b, hl.map_a_res, hl.map_b_res, a);
      if (tracing) {
        std::vector<long long> h(64 * 8);
        cudaStreamSynchronize(s);
        cudaMemcpy(h.data(), d_trace, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
        fprintf(stderr, "[halo trace] layer %d P=%d Ht=%d bn=%d stages=%d T=%d kw=%d cinb=%d (cycles rel. to first event)\n", stp.index, a.P, a.Ht,
                a.block_n, a.stages, a.T * 10 + a.nbuf, a.kw, a.cin_blocks);
        const long long t0 = h[1];
        for (int i = 0; i < 12; ++i) {
          fprintf(stderr, "  group %2d:", i);
          for (int e = 1; e < 7; ++e) fprintf(stderr, " %8lld", h[i * 8 + e] ? h[i * 8 + e] - t0 : -1);
          fprintf(stderr, "\n");
        }
      }
    } else if (stp.kind == 0) {
      ConvLaunch& c = net->convs[stp.index];
      ConvArgs a = c.args;
      a.n_images = n;
      a.tiles_n = (n + a.Nt - 1) / a.Nt;
      if (c.flat) {  // one long row of n * H * W pixels
        a.Wout = n * c.pixels_per_image; a.Hout = 1; a.n_images = 1;
        a.tiles_w = (a.Wout + 127) / 128; a.tiles_h = 1; a.tiles_n = 1;
      }
      dim3 grid((unsigned)(a.tiles_w * a.tiles_h * a.tiles_n), c.grid.y, 1);
      if (c.pair) {
        const long pairs = (((long)grid.x + 1) / 2) * c.n_blocks;
        const unsigned ctas = 2u * (unsigned)std::min<long>(pairs, net->num_sms / 2);
        conv_gemm_pair_kernel<<<ctas, kPersistThreads, c.pair_smem, s>>>(c.map_a, c.map_b_half, a, c.pair_args, c.n_blocks, c.cout);
      } else if (c.persist) {
        const long total = (long)grid.x * c.n_blocks;
        static long long* d_gtrace = nullptr;
        const bool tracing = EnvInt("DVB_CNN_TRACE", 0) == 2 && stp.index == EnvInt("DVB_CNN_TRACE_LAYER", -1);
        if (tracing && !d_gtrace) cudaMalloc(&d_gtrace, 96 * 4 * sizeof(long long));
        if (tracing) { cudaMemsetAsync(d_gtrace, 0, 96 * 4 * sizeof(long long), s); a.trace = d_gtrace; }
        conv_gemm_persistent_kernel<<<(unsigned)std::min<long>(total, net->num_sms), kPersistThreads, c.smem, s>>>(c.map_a, c.map_b, a, c.n_blocks,
                                                                                                                   c.cout);
        if (tracing) {
          std::vector<long long> h(96 * 4);
          cudaStreamSynchronize(s);
          cudaMemcpy(h.data(), d_gtrace, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
          fprintf(stderr, "[gemm trace] conv %d: kh=%d kw=%d cin_blocks=%d block_k=%d block_n=%d stages=%d: k block: full_seen mmas_issued commit_issued (cycles)\n", stp.index, a.kh,
                  a.kw, a.cin_blocks, a.block_k, a.block_n, a.stages);
          for (int i = 0; i < 90; ++i) fprintf(stderr, "  kb %2d: %8lld %8lld %8lld\n", i, h[i * 4] - h[0], h[i * 4 + 1] - h[0], h[i * 4 + 2] - h[0]);
        }
      } else if (net->precision == 1)
        conv_gemm_kernel<true><<<grid, kConvThreads, c.smem, s>>>(c.map_a, c.map_b, c.map_a_res, c.map_b_res, a);
      else
        conv_gemm_kernel<false><<<grid, kConvThreads, c.smem, s>>>(c.map_a, c.map_b, c.map_a_res, c.map_b_res, a);
    } else {
      const PoolLaunch& p = net->pools[stp.index];
      if (p.mode == 0 && !p.in_res && EnvInt("DVB_CNN_MAXPOOL_H2", 1)) {
        // segments so that ~2M threads exist even for the widest maps
        int segs = 1;
        while (segs < 8 && (long long)n * p.Hout * (p.C / 8) * segs < (2LL << 20) && p.Wout / (segs * 2) >= 4) segs *= 2;
        const int seg_len = (p.Wout + segs - 1) / segs;
        const long long total = (long long)n * p.Hout * segs * (p.C / 8);
        maxpool3x3s2_h2_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(p.in, p.out, n, p.Hin, p.Win, p.C, p.Hout, p.Wout, p.out_cstride,
                                                                               p.out_coff, segs, seg_len);
        net->launches++;
        if (stp.record) cudaEventRecord(stp.event, s);
        continue;
      }
      if (p.mode == 1 && !p.in_res && p.Hout == p.Hin && p.Wout == p.Win && EnvInt("DVB_CNN_AVGPOOL_FLAT", 1)) {
        const long long total = (long long)n * p.Hout * p.Wout * (p.C / 8);
        avgpool3x3s1_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(p.in, p.out, n, p.Hin, p.Win, p.C, p.out_cstride, p.out_coff, p.bias);
        net->launches++;
        if (stp.record) cudaEventRecord(stp.event, s);
        continue;
      }
      const long long total = (long long)n * p.Hout * (p.C / 8);
      pool3x3_kernel<<<(unsigned)((total + 127) / 128), 128, 0, s>>>(p.in, p.out, n, p.Hin, p.Win, p.C, p.Hout, p.Wout, p.out_cstride,
                                                                      p.out_coff, p.mode, p.in_res, p.out_res, p.bias);
    }
    net->launches++;
    if (stp.record) cudaEventRecord(stp.event, s);
  }
  for (int d : net->tail_deps) cudaStreamWaitEvent(s0, net->steps[d].event, 0);
  s = s0;
  const TensorBuf& f = net->tensors[net->feat_tensor];
  tail_kernel<<<n, 256, 0, s>>>(f.ptr, f.H * f.W, f.C, net->d_dense_w, net->d_dense_b, probs, net->d_pooled, f.ptr_res);
  net->launches++;
  DVB_CUDA(cudaGetLastError());
  return DVB_OK;
}

}  // namespace

extern "C" {

int dvb_cnn_create(const void* weights, int64_t weights_bytes, int32_t height, int32_t width, int32_t channels, int32_t max_batch,
                   int32_t precision, int device, DvbCnn** out) {
  if (!weights || !out || height < 1 || width < 1 || channels < 1 || channels > 16 || max_batch < 1)
    return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "dvb_cnn_create: bad arguments");
  *out = nullptr;
  if (precision != 0 && precision != 1)
    return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "precision %d is unknown (0 = fp16 operands / fp32 accumulate, 1 = split-fp16 x3)", precision);
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return dvb::fail(DVB_ERR_NO_DEVICE, "no CUDA device (this library has no CPU path)");
  if (device < 0 || device >= ndev) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "device %d out of range", device);
  DVB_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  DVB_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return dvb::fail(DVB_ERR_NO_DEVICE, "the CNN kernels are tcgen05 (sm_100a) only; device is sm_%d%d", prop.major, prop.minor);
  DvbCnn* net = new DvbCnn();
  net->num_sms = prop.multiProcessorCount;
  net->device = device; net->H = height; net->W = width; net->C = channels; net->Cp = PadCin(channels);
  net->max_batch = max_batch; net->precision = precision;
  int st = Plan(net, static_cast<const uint8_t*>(weights), weights_bytes);
  if (st) { dvb_cnn_destroy(net); return st; }
  DVB_CUDA(cudaStreamCreateWithFlags(&net->stream, cudaStreamNonBlocking));
  net->use_graphs = EnvInt("DVB_CNN_GRAPH", 0) != 0 && EnvInt("DVB_CNN_TRACE", 0) == 0;
  *out = net;
  return DVB_OK;
}

void dvb_cnn_destroy(DvbCnn* net) {
  if (!net) return;
  cudaSetDevice(net->device);
  for (DvbCnn::ChunkGraph& g : net->graphs) cudaGraphExecDestroy(g.exec);
  for (void* p : net->allocs) cudaFree(p);
  if (net->d_dense_w) cudaFree(net->d_dense_w);
  if (net->d_dense_b) cudaFree(net->d_dense_b);
  if (net->d_pooled) cudaFree(net->d_pooled);
  net->d_in.release(); net->d_probs.release(); net->h_io.release();
  if (net->stream) cudaStreamDestroy(net->stream);
  for (int l = 1; l < kMaxLanes; ++l)
    if (net->lane_streams[l]) cudaStreamDestroy(net->lane_streams[l]);
  for (Step& stp : net->steps)
    if (stp.event) cudaEventDestroy(stp.event);
  delete net;
}

int dvb_cnn_forward_device(DvbCnn* net, const uint8_t* images, int32_t n, float* probs, void* stream) {
  if (!net || (n > 0 && (!images || !probs)) || n < 0) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "dvb_cnn_forward_device: bad arguments");
  DVB_CUDA(cudaSetDevice(net->device));
  const size_t image_bytes = (size_t)net->H * net->W * net->C;
  for (int i = 0; i < n; i += net->max_batch) {
    const int m = std::min(net->max_batch, n - i);
    int st = ForwardChunk(net, images + (size_t)i * image_bytes, m, probs + (size_t)i * 3, static_cast<cudaStream_t>(stream));
    if (st) return st;
  }
  return DVB_OK;
}

int dvb_cnn_forward_host(DvbCnn* net, const uint8_t* images_host, int32_t n, float* probs_host) {
  if (!net || (n > 0 && (!images_host || !probs_host)) || n < 0) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "dvb_cnn_forward_host: bad arguments");
  if (n == 0) return DVB_OK;
  DVB_CUDA(cudaSetDevice(net->device));
  const size_t image_bytes = (size_t)net->H * net->W * net->C;
  DVB_CUDA(net->d_in.reserve((size_t)n * image_bytes));
  DVB_CUDA(net->d_probs.reserve((size_t)n * 3 * sizeof(float)));
  DVB_CUDA(cudaMemcpyAsync(net->d_in.p, images_host, (size_t)n * image_bytes, cudaMemcpyHostToDevice, net->stream));
  int st = dvb_cnn_forward_device(net, static_cast<const uint8_t*>(net->d_in.p), n, static_cast<float*>(net->d_probs.p), net->stream);
  if (st) return st;
  DVB_CUDA(cudaMemcpyAsync(probs_host, net->d_probs.p, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToHost, net->stream));
  DVB_CUDA(cudaStreamSynchronize(net->stream));
  return DVB_OK;
}

int64_t dvb_cnn_launch_count(const DvbCnn* net) { return net ? net->launches : 0; }
double dvb_cnn_flops_per_image(const DvbCnn* net) { return net ? net->flops_per_image : 0.0; }
int32_t dvb_cnn_max_batch(const DvbCnn* net) { return net ? net->max_batch : 0; }

// Debug / test access to an intermediate activation of the LAST forward (first `n` images):
// out_host = float[n][H][W][C] (NHWC).  name: "input", "s1".."s5", "p1", "p2", "mixed0".."mixed10", branch tensors.
// name "pooled" returns float[n][2048].  *h/*w/*c receive the shape.
int dvb_cnn_debug_tensor(DvbCnn* net, const char* name, int32_t n, float* out_host, int32_t* h, int32_t* w, int32_t* c) {
  if (!net || !name) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "null argument");
  DVB_CUDA(cudaSetDevice(net->device));
  DVB_CUDA(cudaDeviceSynchronize());
  if (std::string(name) == "pooled") {
    if (h) *h = 1; if (w) *w = 1; if (c) *c = 2048;
    if (out_host) DVB_CUDA(cudaMemcpy(out_host, net->d_pooled, (size_t)n * 2048 * sizeof(float), cudaMemcpyDeviceToHost));
    return DVB_OK;
  }
  auto it = net->tensor_index.find(name);
  if (it == net->tensor_index.end()) return dvb::fail(DVB_ERR_INVALID_ARGUMENT, "no tensor named %s", name);
  const TensorBuf& t = net->tensors[it->second];
  if (h) *h = t.H; if (w) *w = t.W; if (c) *c = t.Cl;
  if (!out_host) return DVB_OK;
  const long long cnt = (long long)n * t.H * t.W * t.C;
  float* tmp = nullptr;
  DVB_CUDA(cudaMalloc(&tmp, cnt * sizeof(float)));
  half_to_float_kernel<<<(unsigned)((cnt + 255) / 256), 256>>>(t.ptr, t.ptr_res, tmp, cnt);
  cudaError_t e;
  if (t.Cl == t.C) {
    e = cudaMemcpy(out_host, tmp, cnt * sizeof(float), cudaMemcpyDeviceToHost);
  } else {   // drop the zero padding channels
    e = cudaMemcpy2D(out_host, (size_t)t.Cl * sizeof(float), tmp, (size_t)t.C * sizeof(float), (size_t)t.Cl * sizeof(float),
                     (size_t)n * t.H * t.W, cudaMemcpyDeviceToHost);
  }
  cudaFree(tmp);
  if (e != cudaSuccess) return dvb::fail(DVB_ERR_CUDA, "debug copy failed: %s", cudaGetErrorString(e));
  return DVB_OK;
}

}  // extern "C"
