// sm_100a tensor-core building blocks written as inline PTX: mbarrier, bulk async copies (TMA
// engine, 1-D), tcgen05 alloc / mma / commit / ld, UMMA shared-memory + instruction descriptors,
// and the split-bf16 ("bf16x3") operand images.
//
// Operand images (bf16):
//  * SW128 K-major tile of R rows x 64 elements: row pitch 128 B, 8-row groups 1024 B apart (SBO),
//    16-byte chunk c of row r stored at chunk position c ^ (r & 7) (the 128B swizzle).  The same bytes
//    read as an MN-major operand (MN = the 64 contiguous elements, K = rows) are the canonical
//    MN-major SW128 layout, so one activation image serves  X.W (K = features)  and  X^T.Y (K = rows).
//  * INTERLEAVE (no swizzle) K-major tile of R rows x 16 elements: 8x16B core matrices, the two K halves
//    128 B apart (LBO), 8-row groups 256 B apart (SBO).
// fp32 accuracy comes from 3 bf16 products per contraction: a.b ~= a_hi.b_hi + a_lo.b_hi + a_hi.b_lo with
// x_hi = bf16(x), x_lo = bf16(x - x_hi); the dropped terms are O(2^-16) relative (SURVEY.md 7.3).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace mpg {
namespace tc {

// hidden width of the tensor-core path: the weight ring, the TMEM column map, the epilogue warp <-> 64-column quarter
// map and the image sizes are all laid out for 256 (the handle offers this backend at hidden = 256 only)
constexpr int H = 256;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier --------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity), "r"(0x989680) : "memory");
  return ok != 0;
}
// Watchdog of the mbarrier waits: a protocol error must not hang the GPU.  g_wait_dbg points to pinned, mapped host
// memory (set once per process by the library); a wait that does not complete within MPG_WAIT_LIMIT_CYCLES records
// {site (source line), block, thread, parity} there and traps, so that the launch fails with an error the host can report.
// Every translation unit has its own copy of the record pointer and of mbar_timeout: the library attaches each unit's
// copy with wait_dbg_attach (api.cu: wait_dbg_init, MlpKernels::attach_watchdog).
static __device__ unsigned long long* g_wait_dbg = nullptr;
#ifndef MPG_WAIT_LIMIT_CYCLES
#define MPG_WAIT_LIMIT_CYCLES 4000000000ll    /* ~2 s at 1.965 GHz; the longest legitimate wait is a few hundred microseconds */
#endif
static inline bool wait_dbg_attach(unsigned long long* dev_ptr) {
  return cudaMemcpyToSymbol(g_wait_dbg, &dev_ptr, sizeof(dev_ptr)) == cudaSuccess;
}
static __device__ __noinline__ void mbar_timeout(int site, uint32_t parity) {
  if (g_wait_dbg) {
    // records {site, block, thread, parity} at g_wait_dbg[4 + 4 k], k = warpgroup of the thread (0..3 epilogue, 4 row warps,
    // 5/6 producer / mma warp), g_wait_dbg[0] = flag.  The first thread to give up lingers a little before it traps, so that
    // the other stuck roles of the CTA get to record as well.
    const int w = (int)(threadIdx.x >> 5);
    const int k = w >= 20 ? 5 + (w & 1) : w / 4;
    volatile unsigned long long* r = g_wait_dbg + 4 + 4 * k;
    r[0] = (unsigned long long)site;
    r[1] = (unsigned long long)blockIdx.x;
    r[2] = (unsigned long long)threadIdx.x;
    r[3] = (unsigned long long)parity + 1ull;
    g_wait_dbg[0] = 1ull;
    __threadfence_system();
  }
}
// try_wait suspends the thread in hardware (up to the time hint) and wakes it on phase completion, so
// waiting warps do not burn issue slots of the warps doing the per-row math on the same sub-partition
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int site = 0) {
  if (mbar_try(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try(bar, parity)) {
    if (clock64() - t0 > MPG_WAIT_LIMIT_CYCLES) {
      mbar_timeout(site, parity);
      const long long t1 = clock64();
      while (clock64() - t1 < 400000000ll) {}     // a little later, so that the other stuck roles record too
      __trap();
    }
  }
}
#define MBAR_WAIT(bar, parity) mbar_wait((bar), (parity), __LINE__)
// 2^x, flush-to-zero approximate (one MUFU, no denormal fix-up code)
__device__ __forceinline__ float ex2_ftz(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float exp_fast(float x) { return ex2_ftz(x * 1.4426950408889634f); }
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// make generic-proxy shared-memory writes visible to the async proxy (tcgen05.mma / bulk copies)
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- bulk async copies (1-D, no tensor map) -----------------------------------------------------
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)),
               "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// wait until at most `pending` of the most recent bulk groups of this thread still read their shared-memory source
__device__ __forceinline__ void bulk_wait_read_pending(int pending) {
  switch (pending) {
    case 3: asm volatile("cp.async.bulk.wait_group.read 3;" ::: "memory"); break;
    case 2: asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory"); break;
    case 1: asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); break;
    default: asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); break;
  }
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- tcgen05 -------------------------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_result, uint32_t ncols) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_result)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {       // same warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] . B[smem]^T, bf16 inputs, fp32 accumulate; issued by ONE thread
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc),
      "r"(accumulate) : "memory");
}
// arrive on an mbarrier when all previously issued tcgen05.mma of this thread have completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 32 consecutive fp32 columns of this thread's TMEM lane (lane = 32 * (warp % 4) + laneid)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// split-phase variant: issue the load, keep working, then make the registers valid with tmem_ld_wait (which takes them as
// in/out operands so that no use can be scheduled above it)
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_ld_wait(uint32_t (&r)[16]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
               :: "memory");
}

// One thread of a fully converged warp.  Roles that issue tcgen05.mma / tcgen05.commit / bulk copies from a single thread must
// be entered through this and not through `lane == 0`: both pick lane 0, but only after elect.sync does the compiler
// know that exactly one thread is active and emit the uniform-datapath instructions (UTCHMMA, UTCBAR, UBLKCP) straight;
// behind a thread-index test it wraps EVERY one of them in an ELECT / BRA.U.ANY loop (6 instructions and a branch per UMMA,
// ~100 cycles each from a lone thread -- the "small UMMAs cost 100 cycles whatever their N" of the first round-2 kernels).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.b32 %0, 1, 0, P;\n}\n" : "=r"(pred));
  return pred != 0;
}

// ---- descriptors ---------------------------------------------------------------------------------
// UMMA shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [49,52) base_offset=0 | [61,64) layout
enum : uint64_t { LAYOUT_NONE = 0, LAYOUT_SW128 = 2, LAYOUT_SW64 = 4, LAYOUT_SW32 = 6 };
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint64_t layout) {
  return (uint64_t)((smem_addr & 0x3FFFF) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(sbo_bytes >> 4) << 32)
         | (1ull << 46) | (layout << 61);
}
// UMMA instruction descriptor, kind::f16, bf16 x bf16 -> fp32 (cute::UMMA::InstrDescriptor bit layout):
//   [4,6) c_format=1 (F32) | [7,10) a_format=1 (BF16) | [10,13) b_format=1 | [15] a_major | [16] b_major
//   | [17,23) N>>3 | [24,29) M>>4          major: 0 = K-major, 1 = MN-major
// a_fmt / b_fmt: operand element formats of kind::f16, 0 = F16, 1 = BF16; the two operands may differ
enum : int { FMT_F16 = 0, FMT_BF16 = 1 };
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, int a_mn_major, int b_mn_major, int a_fmt = FMT_BF16,
                                                   int b_fmt = FMT_BF16) {
  return (1u << 4) | ((uint32_t)a_fmt << 7) | ((uint32_t)b_fmt << 10) | ((uint32_t)a_mn_major << 15)
         | ((uint32_t)b_mn_major << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---- split-bf16 helpers ----------------------------------------------------------------------------
// two floats -> packed bf16x2 hi and lo words (element 0 in the low half-word)
__device__ __forceinline__ void split2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  __nv_bfloat162 h = __floats2bfloat162_rn(x0, x1);
  hi = *reinterpret_cast<uint32_t*>(&h);
  const float h0 = __uint_as_float(hi << 16), h1 = __uint_as_float(hi & 0xFFFF0000u);
  __nv_bfloat162 l = __floats2bfloat162_rn(x0 - h0, x1 - h1);
  lo = *reinterpret_cast<uint32_t*>(&l);
}

// Forward-side operands ([p|a|1], h1 and the weight images they meet: W1aug, W2^T) use the same three-product scheme on
// FP16 pairs: 11 + 11 significant bits instead of 8 + 8, i.e. ~2^-22 per product against ~2^-16.  With bf16 pairs the
// closed-loop actions / rewards sit at 1-2e-5 of the fp64 oracle -- over the 1e-5 bar on some seeds; with fp16 pairs at
// 1-2e-6 (tests/test_gpu_parity.py::test_tc_closed_loop_margin_over_seeds).  Everything on the backward side (deltas
// scaled by 1/(M B) and gamma^t, their weight images, the h2 store) keeps bf16 pairs for the exponent range; kind::f16
// takes the A and B formats independently, so delta (bf16) x p / h1 (fp16) contractions need no conversion.
// Values beyond the fp16 range saturate (satfinite) instead of becoming inf.
__device__ __forceinline__ void split2h(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));
  const __half2 h = *reinterpret_cast<const __half2*>(&hi);
  const float2 hf = __half22float2(h);
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(x1 - hf.y), "f"(x0 - hf.x));
}
template <bool F16>
__device__ __forceinline__ void split2x(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  if (F16) split2h(x0, x1, hi, lo); else split2(x0, x1, hi, lo);
}

constexpr int ACT_ROWS = 128;                 // rows per CTA tile (= UMMA M)
constexpr int ACT_BLOCK = ACT_ROWS * 128;     // one 64-feature block: 128 rows x 128 B = 16 KB
constexpr int ACT_SPLIT = 4 * ACT_BLOCK;      // 256 features: 64 KB per split (hi | lo)

// byte offset of the 16-byte chunk holding features [8*cc, 8*cc+8) of row r inside one split of an
// activation image (cc in [0,32))
__device__ __forceinline__ uint32_t act_chunk_off(int r, int cc) {
  return (uint32_t)((cc >> 3) * ACT_BLOCK + (r >> 3) * 1024 + (r & 7) * 128 + (((cc & 7) ^ (r & 7)) << 4));
}
// store 8 consecutive features (fp32) of row r as hi / lo bf16 chunks; when `gimg` is given the same two
// chunks also go to the global copy of the image (dW operand store, identical layout)
template <bool F16 = false>
__device__ __forceinline__ void act_store8(uint8_t* act_hi, uint8_t* act_lo, int r, int cc, const float* x,
                                           uint8_t* gimg = nullptr) {
  uint4 h, l;
  split2x<F16>(x[0], x[1], h.x, l.x);
  split2x<F16>(x[2], x[3], h.y, l.y);
  split2x<F16>(x[4], x[5], h.z, l.z);
  split2x<F16>(x[6], x[7], h.w, l.w);
  const uint32_t off = act_chunk_off(r, cc);
  *reinterpret_cast<uint4*>(act_hi + off) = h;
  *reinterpret_cast<uint4*>(act_lo + off) = l;
  if (gimg) {
    *reinterpret_cast<uint4*>(gimg + off) = h;
    *reinterpret_cast<uint4*>(gimg + ACT_SPLIT + off) = l;
  }
}
// INTERLEAVE K-major image of R rows x 16 elements: byte offset of the 16-byte chunk (k half kh) of row r
__device__ __forceinline__ uint32_t il_chunk_off(int r, int kh) { return (uint32_t)((r >> 3) * 256 + kh * 128 + (r & 7) * 16); }
// [p|a|1] image: R rows x (16 hi | 16 lo) elements, the four 16-byte chunks (hi0, hi1, lo0, lo1) of an 8-row group next to
// each other (512 B per group).  Read K-major it is two R x 16 INTERLEAVE operands (hi at +0, lo at +256; LBO 128, SBO 512);
// read MN-major (K = rows) it is ONE operand with N = 32 = [p_hi | p_lo] (SBO 128, LBO 512), so that delta1^T [p_hi | p_lo]
// needs two UMMAs per row step (delta1_hi, delta1_lo) instead of three products.
constexpr int P_GROUP = 512, P_LO = 256;
__device__ __forceinline__ uint32_t p_chunk_off(int r, int c) { return (uint32_t)((r >> 3) * P_GROUP + c * 128 + (r & 7) * 16); }

}  // namespace tc
}  // namespace mpg
