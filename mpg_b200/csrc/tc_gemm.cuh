// Warp-specialised GEMM machinery shared by the tensor-core rollout kernels.
//
// Roles inside one CTA (576 threads):
//   warps 0-15 "epilogue": thread = (TMEM lane = row, 64-column quarter); they build the A-operand images in
//              shared memory, read accumulators back with tcgen05.ld and run all per-row math;
//   warp 16    "producer": one elected lane streams weight images from global/L2 into a 4-slot ring with
//              1-D bulk async copies (TMA engine) completing on mbarriers;
//   warp 17    "mma": one elected lane issues tcgen05.mma and commits to mbarriers.
// The three roles execute the SAME schedule (same function, same CTA-uniform control flow) and meet only
// through mbarriers:  a_full / a_blk[] (epilogue -> mma: operand image / 64-feature block written), d_full
// (mma -> epilogue: accumulator complete), z_full[] / z_empty[] (first-layer chunk stream), kb_done[] (K-block of
// a big GEMM complete: its image block may leave for the record store), acc_done (in-kernel dW1 UMMAs done),
// ring full[]/empty[] (producer <-> mma).
#pragma once
#include "tc_common.cuh"

namespace mpg {
namespace tc {

#ifndef MPG_EPI_WARPS
#define MPG_EPI_WARPS 16
#endif
constexpr int EPI_WARPS = MPG_EPI_WARPS;                 // 4 per TMEM lane quadrant: each owns 64 accumulator columns
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int CTA_THREADS = EPI_THREADS + 64;  // + producer warp + mma warp
constexpr int COLS_PER_WARP = 256 / (EPI_WARPS / 4);
constexpr int STAGE_BYTES = 16384;            // ring slot: one split (hi or lo) of all 256 output features x 32 contraction elements
constexpr int NSLOT = 4;                      // 3 loads in flight while one slot is consumed
constexpr int BIG_STAGES = 16;                // (k-block, split, k-half)
constexpr int BIG_IMAGE_BYTES = BIG_STAGES * STAGE_BYTES;
constexpr int TMEM_COLS = 512;
// TMEM column regions: two 64-column first-layer chunk buffers (z1 is streamed, never resident), the 256-column
// working accumulator (z2 / g_h1), the 16-column input gradient, and the persistent weight-gradient accumulators
// D1 = delta1^T [p|1] and D3 = h2^T [delta3|0] (two 128-feature halves x 16 columns each)
// Small-N UMMAs that accumulate into the same tile form a dependent chain and pay the tensor pipe's latency (~150 cycles)
// each instead of its throughput, so g_p and D3 (both on the critical path of a BPTT step) are split over TWO accumulator
// sets (32 columns apart) that the reader adds up.
// The small contractions put the hi and lo halves of their B operand side by side in N, so that one UMMA per A split does
// the work of the three split products (and keeps the lo.lo term):
//   g_p [128 x 32]     = delta1 . [W1_hi ; W1_lo]^T      -> g_p = columns [0,16) + [16,32)
//   D1  [2 x 128 x 32] = delta1^T . [p_hi | p_lo]         -> dW1 = columns [0,16) + [16,32)
//   D3  [2 x 128 x 16] = h2^T . [d3_hi | d3_lo | 0]       -> dW3[:, j] = column j + column 2 + j
constexpr int TM_Z1C = 0, TM_WORK = 128, TM_GP = 384, TM_D1 = 416, TM_D3 = 480;

// shared memory map (bytes, 1024-aligned base)
struct SmemMap {
  static constexpr int ACT = 0;                               // activation image hi|lo: 128 KB
  static constexpr int RING = ACT + 2 * ACT_SPLIT;            // 4 x 16 KB
  static constexpr int PIMG = RING + NSLOT * STAGE_BYTES;     // [p|a|1] image hi|lo: 2 x 4 KB (ring = 4 x 16 KB)
  static constexpr int MISC = PIMG + 8192;                    // fp32 scratch, see MiscF
  static constexpr int MISC_BYTES = 12288;
  static constexpr int BARS = MISC + MISC_BYTES;              // mbarriers + tmem pointer
  static constexpr int TOTAL = BARS + 512;
};

struct Bars {
  uint64_t full[NSLOT];
  uint64_t empty[NSLOT];
  uint64_t a_full;       // [p|a|1] image written (first-layer GEMMs)
  uint64_t a_blk[4];     // 64-feature block kb of the activation image written (K-block pipelining)
  uint64_t d_full;
  uint64_t d_half;       // second publish of an accumulator that is handed over in two parts (forward GEMM halves, D3 halves): a
                         // waiter that lags TWO phases behind a parity barrier never wakes up, so each part has its own barrier
  uint64_t z_full[2];    // first-layer chunk buffer j holds a fresh 64-column chunk (mma -> epilogue)
  uint64_t z_empty[2];   // chunk buffer j has been read out (epilogue -> mma)
  uint64_t acc_done;     // the D1 accumulation UMMAs have read the delta1 / [p|1] images
  uint64_t kb_done[4];   // big GEMM: the UMMAs of K-block kb are complete (block kb of the A image is no longer read)
  uint64_t p_full;       // BPTT: the [p|1] image of this step is written (row threads -> mma, first-layer recompute)
  uint64_t img_empty[2]; // BPTT: nothing reads 128-feature half h of the activation image any more (mma commit + elected
                         // epilogue thread): the h2 image of the next step may land there
  uint64_t img_full[2];  // BPTT: half h of the h2 image of this step has landed (TMA complete_tx)
  uint64_t gp_full;      // the input gradient g_p is complete (mma -> row warps; the epilogue warps use d_full)
  uint32_t tmem_base;
};
static_assert(sizeof(Bars) <= 512, "BARS region too small");

// per-role running counters (phase tracking)
struct Sync {
  uint32_t stage = 0;    // ring stages produced / consumed so far
  uint32_t a_cnt = 0;    // a_full phases seen
  uint32_t g_cnt = 0;    // a_blk[] phases seen (GEMMs whose A operand is the activation image)
  uint32_t d_cnt = 0;    // d_full phases seen
  uint32_t h_cnt = 0;    // d_half phases seen
  uint32_t acc_cnt = 0;  // acc_done phases seen (epilogue side)
  uint32_t k_cnt = 0;    // big GEMMs issued so far (kb_done[] phases, epilogue side)
  uint32_t p_cnt = 0;    // p_full phases seen
  uint32_t i_cnt = 0;    // img_empty / img_full phases seen (h2 image loads)
  uint32_t gp_cnt = 0;   // gp_full phases seen (row warps)
};

enum Role { ROLE_EPI = 0, ROLE_PRODUCER = 1, ROLE_MMA = 2, ROLE_ROW = 3 };

// ---- producer: stream `nstages` stages of `bytes` each ------------------------------------------------
__device__ __forceinline__ void produce(Bars* b, uint8_t* ring, Sync& s, const uint8_t* gsrc, int nstages, uint32_t bytes) {
  for (int i = 0; i < nstages; ++i, ++s.stage) {
    const uint32_t slot = s.stage & (NSLOT - 1), par = (s.stage / NSLOT) & 1;
    mbar_wait(&b->empty[slot], par ^ 1, 10000 + __LINE__);
    mbar_expect_tx(&b->full[slot], bytes);
    bulk_g2s(ring + slot * STAGE_BYTES, gsrc + (size_t)i * bytes, bytes, &b->full[slot]);
  }
}

// The 16 KB images of the small GEMMs (first layer, input gradient) are ONE stage, followed by an empty one, so that every
// GEMM consumes an even number of stages (the big GEMM's k-halves start on an even slot).
__device__ __forceinline__ uint32_t wait_single(Bars* b, const Sync& s) {
  const uint32_t slot = s.stage & (NSLOT - 1), par = (s.stage / NSLOT) & 1;
  mbar_wait(&b->full[slot], par, 10000 + __LINE__);
  tc_fence_after();
  return slot;
}
__device__ __forceinline__ void consume_pad(Bars* b, Sync& s) {   // the empty stage behind a single-stage image
  const uint32_t pad = s.stage & (NSLOT - 1), par = (s.stage / NSLOT) & 1;
  mbar_wait(&b->full[pad], par, 10000 + __LINE__);
  umma_commit(&b->empty[pad]);
  ++s.stage;
}
__device__ __forceinline__ void release_single(Bars* b, Sync& s, uint32_t slot) {
  umma_commit(&b->empty[slot]);
  ++s.stage;
  consume_pad(b, s);
}
// producer side of a 16 KB single-stage image + its empty stage
__device__ __forceinline__ void produce_single(Bars* b, uint8_t* ring, Sync& s, const uint8_t* gsrc) {
  produce(b, ring, s, gsrc, 1, STAGE_BYTES);
  const uint32_t slot = s.stage & (NSLOT - 1), par = (s.stage / NSLOT) & 1;
  mbar_wait(&b->empty[slot], par ^ 1, 10000 + __LINE__);
  mbar_arrive(&b->full[slot]);
  ++s.stage;
}

// ---- mma role ----------------------------------------------------------------------------------------
// big GEMM: D[128 x 256] = ACT[128 x 256] . Wt^T.  The Wt image is streamed as 16 stages of 16 KB ordered
// (k-block kb, split, k-half kh); a stage holds ALL 256 output features of 32 contraction elements (64-byte rows,
// SW64 K-major), so every ring slot is an independent B operand: it feeds two K = 16 steps of N = 256 UMMAs and goes
// back to the producer as soon as those have completed -- three 16 KB loads stay in flight.
//   Measured (tools/gemm_probe.py, one CTA per SM): 6.7 K cycles per GEMM = the rate with resident operands (6.6 K);
//   832 KB of shared-memory traffic per GEMM (576 KB operand reads + 256 KB ring writes) = 125 of the 128 B/clk.
//   (kb, split, n-half) stages of 128 features x 64 elements consumed and released in PAIRS (round 2's first layout):
//   8.8 K -- only two 32 KB granules in flight, every refill exposed the L2 latency.  32 stages of 8 KB (one K = 16 step
//   each, 8 slots; SW32 or no-swizzle): 9.8 K -- ~190 cycles of fixed cost per stage (wait + commit + bulk copy) x 32.
// K-block kb is issued as soon as the epilogue has published that 64-feature block of the activation image, so the
// UMMAs overlap the epilogue that produces A.
// FMT: element format of BOTH operands (forward GEMMs: fp16 pairs, dX GEMMs: bf16 pairs)
struct NoHook { __device__ __forceinline__ void operator()() const {} };
// after_first: issued right behind the first two stages (split 0 of K-block 0); the forward pass puts its last first-layer chunk
// there -- not later: the first-layer image still holds one of the four ring slots, and the third stage needs it back
template <int FMT = FMT_BF16, typename Hook = NoHook>
__device__ __forceinline__ void mma_big(Bars* b, uint32_t act_addr, uint32_t ring_addr, Sync& s, uint32_t d_tmem,
                                        bool wait_a = true, long long* prof = nullptr, Hook after_first = Hook()) {
  constexpr uint32_t idesc = make_idesc(128, 256, 0, 0, FMT, FMT);
  for (int kb = 0; kb < 4; ++kb) {
    if (wait_a) mbar_wait(&b->a_blk[kb], s.g_cnt & 1, 10000 + __LINE__);
    if (prof) prof[kb * 5] = clock64();          // timeline probe (debug library): A block kb seen
    tc_fence_after();
    const uint64_t dah = make_desc(act_addr + kb * ACT_BLOCK, 16, 1024, LAYOUT_SW128);
    const uint64_t dal = make_desc(act_addr + ACT_SPLIT + kb * ACT_BLOCK, 16, 1024, LAYOUT_SW128);
#pragma unroll
    for (int sp = 0; sp < 2; ++sp) {
#pragma unroll
      for (int kh = 0; kh < 2; ++kh) {
        const uint32_t slot = s.stage & (NSLOT - 1), par = (s.stage / NSLOT) & 1;
        mbar_wait(&b->full[slot], par, 10000 + __LINE__);
        if (prof) prof[kb * 5 + 1 + sp * 2 + kh] = clock64();   // stage (kb, sp, kh) seen in its slot
        tc_fence_after();
        const uint64_t db = make_desc(ring_addr + slot * STAGE_BYTES, 16, 512, LAYOUT_SW64);
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const uint64_t ka = (uint64_t)((kh * 2 + j) * 2);   // +32 bytes along K inside the 128-byte swizzle atom of A
          const uint64_t kw = (uint64_t)(j * 2);              // +32 bytes inside the 64-byte swizzle atom of the weights
          if (sp == 0) {
            umma_bf16(d_tmem, dah + ka, db + kw, idesc, (kb | kh | j) ? 1u : 0u);   // a_hi . b_hi
            umma_bf16(d_tmem, dal + ka, db + kw, idesc, 1u);                        // a_lo . b_hi
          } else {
            umma_bf16(d_tmem, dah + ka, db + kw, idesc, 1u);                        // a_hi . b_lo
          }
        }
        umma_commit(&b->empty[slot]);
        ++s.stage;
      }
      if (kb == 0 && sp == 0) after_first();
    }
    umma_commit(&b->kb_done[kb]);
  }
  ++s.g_cnt;
}
// 64-column chunk c of the first-layer GEMM into chunk buffer c & 1.  Every streamed first-layer GEMM issues
// exactly chunks 0..3, so buffer j is used twice per GEMM and the mbarrier parities depend on c only.
template <int FMT>
__device__ __forceinline__ void mma_l1_chunk(Bars* b, uint32_t p_addr, uint32_t bbase, int c, uint32_t tm_z1c) {
  constexpr uint32_t idesc = make_idesc(128, 64, 0, 0, FMT, FMT);
  mbar_wait(&b->z_empty[c & 1], ((c >> 1) & 1) ^ 1, 10000 + __LINE__);
  tc_fence_after();
  const uint64_t dah = make_desc(p_addr, 128, P_GROUP, LAYOUT_NONE), dal = make_desc(p_addr + P_LO, 128, P_GROUP, LAYOUT_NONE);
  const uint64_t dbh = make_desc(bbase + c * 2048, 128, 256, LAYOUT_NONE), dbl = make_desc(bbase + 8192 + c * 2048, 128, 256, LAYOUT_NONE);
  const uint32_t d = tm_z1c + (c & 1) * 64;
  umma_bf16(d, dah, dbh, idesc, 0u);
  umma_bf16(d, dal, dbh, idesc, 1u);
  umma_bf16(d, dah, dbl, idesc, 1u);
  umma_commit(&b->z_full[c & 1]);
}
// epilogue side of the chunk stream
__device__ __forceinline__ void epi_wait_chunk(Bars* b, int c) {
  mbar_wait(&b->z_full[c & 1], (c >> 1) & 1, 10000 + __LINE__);
  tc_fence_after();
}
__device__ __forceinline__ void epi_release_chunk(Bars* b, int c) {
  tc_fence_before();
  mbar_arrive(&b->z_empty[c & 1]);
}
// Weight-gradient accumulation with the operands where they already are: D[half][128 features x N] +=
// IMG[:, half]^T . R, IMG = activation image read MN-major (K = rows), R = an image with hi and lo side by side in N
// read MN-major: the [p|a|1] image (N = 32, D1) or the delta3 image (N = 16, D3).  16 UMMAs per half (8 row steps x the
// two splits of IMG); a half needs only its two 64-feature blocks of the image, so it can be issued as soon as those are
// written and lets the image be overwritten half by half.
// lin: the image is in the row-interleaved no-swizzle layout [chunk][row][16 B] (h2 images loaded from the h2 store):
// MN-major INTERLEAVE, 8-row groups 128 B apart (LBO), 8-feature chunks 2048 B apart (SBO), 16 rows = 256 B per k-step.
template <int N, int B_FMT = FMT_BF16>
__device__ __forceinline__ void mma_acc_half(uint32_t act_addr, uint32_t r_addr, uint32_t r_group, uint32_t d_tmem, int half,
                                             bool started, bool lin = false, bool img_hi_only = false) {
  constexpr uint32_t idesc = make_idesc(128, N, 1, 1, FMT_BF16, B_FMT);
  const uint32_t d = d_tmem + half * N;
#pragma unroll
  for (int ks = 0; ks < ACT_ROWS / 16; ++ks) {
    const uint32_t a = act_addr + half * 2 * ACT_BLOCK + (lin ? ks * 256 : ks * 2048);
    const uint64_t dah = lin ? make_desc(a, 128, 2048, LAYOUT_NONE) : make_desc(a, ACT_BLOCK, 1024, LAYOUT_SW128);
    const uint64_t dal = lin ? make_desc(a + ACT_SPLIT, 128, 2048, LAYOUT_NONE) : make_desc(a + ACT_SPLIT, ACT_BLOCK, 1024, LAYOUT_SW128);
    const uint64_t db = make_desc(r_addr + ks * 2 * r_group, r_group, 128, LAYOUT_NONE);   // 8-row groups r_group apart (LBO)
    umma_bf16(d, dah, db, idesc, (started || ks) ? 1u : 0u);
    if (!img_hi_only) umma_bf16(d, dal, db, idesc, 1u);
  }
}
// first-layer GEMM: D[128 x 256] = P[128 x 16] . W1aug^T ; P is the INTERLEAVE image in shared memory,
// W1aug image streamed as ONE stage = [hi: 256 rows x 32 B][lo: 256 rows x 32 B] = 16 KB
__device__ __forceinline__ void mma_l1(Bars* b, uint32_t p_addr, uint32_t ring_addr, Sync& s, uint32_t d_tmem) {
  constexpr uint32_t idesc = make_idesc(128, 256, 0, 0, FMT_F16, FMT_F16);
  mbar_wait(&b->a_full, s.a_cnt & 1, 10000 + __LINE__);
  ++s.a_cnt;
  const uint32_t slot = wait_single(b, s);
  const uint32_t bbase = ring_addr + slot * STAGE_BYTES;
  const uint64_t dah = make_desc(p_addr, 128, P_GROUP, LAYOUT_NONE), dal = make_desc(p_addr + P_LO, 128, P_GROUP, LAYOUT_NONE);
  const uint64_t dbh = make_desc(bbase, 128, 256, LAYOUT_NONE), dbl = make_desc(bbase + 8192, 128, 256, LAYOUT_NONE);
  umma_bf16(d_tmem, dah, dbh, idesc, 0u);
  umma_bf16(d_tmem, dal, dbh, idesc, 1u);
  umma_bf16(d_tmem, dah, dbl, idesc, 1u);
  release_single(b, s, slot);
}
// input-gradient GEMM: D[128 x 32] = ACT[128 x 256] . [W1nat_hi ; W1nat_lo]^T (W1nat: 16 rows x 256); the image is
// streamed as ONE stage = 4 k-blocks x (32 rows x 128 B) = 16 KB; g = D[:, 0:16] + D[:, 16:32]
__device__ __forceinline__ void mma_in_block(uint32_t act_addr, uint32_t ibase, int kb, uint32_t d_tmem) {
  constexpr uint32_t idesc = make_idesc(128, 32, 0, 0);
#pragma unroll
  for (int ks = 0; ks < 4; ++ks) {
    const uint32_t a_hi = act_addr + kb * ACT_BLOCK + ks * 32, a_lo = a_hi + ACT_SPLIT;
    const uint64_t dah = make_desc(a_hi, 16, 1024, LAYOUT_SW128), dal = make_desc(a_lo, 16, 1024, LAYOUT_SW128);
    const uint64_t db = make_desc(ibase + kb * 4096 + ks * 32, 16, 1024, LAYOUT_SW128);
    umma_bf16(d_tmem, dah, db, idesc, (kb | ks) ? 1u : 0u);
    umma_bf16(d_tmem, dal, db, idesc, 1u);
  }
}
__device__ __forceinline__ void mma_in(Bars* b, uint32_t act_addr, uint32_t ring_addr, Sync& s, uint32_t d_tmem) {
  uint32_t slot = 0;
  for (int kb = 0; kb < 4; ++kb) {
    mbar_wait(&b->a_blk[kb], s.g_cnt & 1, 10000 + __LINE__);
    if (kb == 0) slot = wait_single(b, s);
    tc_fence_after();
    mma_in_block(act_addr, ring_addr + slot * STAGE_BYTES, kb, d_tmem);
  }
  release_single(b, s, slot);
  ++s.g_cnt;
}

// ---- handshakes ----------------------------------------------------------------------------------------
// epilogue side: [p|a|1] image (and any TMEM reads) done -> let the first-layer GEMM go
__device__ __forceinline__ void epi_publish_a(Bars* b) {
  tc_fence_before();
  fence_proxy_async();
  mbar_arrive(&b->a_full);
}
// epilogue side: 64-feature block kb of the activation image written by this thread
__device__ __forceinline__ void epi_block_done(Bars* b, int kb) {
  tc_fence_before();
  fence_proxy_async();
  mbar_arrive(&b->a_blk[kb]);
}
__device__ __forceinline__ void mma_publish_d(Bars* b) { umma_commit(&b->d_full); }
__device__ __forceinline__ void epi_wait_half(Bars* b, Sync& s) {
  mbar_wait(&b->d_half, s.h_cnt & 1, 10000 + __LINE__);
  ++s.h_cnt;
  tc_fence_after();
}
__device__ __forceinline__ void epi_wait_d(Bars* b, Sync& s) {
  mbar_wait(&b->d_full, s.d_cnt & 1, 10000 + __LINE__);
  ++s.d_cnt;
  tc_fence_after();
}

// Issue side of one GEMM. kind: 0 big, 1 first layer, 2 input gradient.  Producer: stream the weight image.
// MMA: wait for the operands (per K-block), issue, commit d_full.  Epilogue: kind 1 publishes the [p|a|1]
// image here; kinds 0/2 publish their A blocks from inside the epilogue loops (epi_block_done).  The
// epilogue picks the result up later with epi_wait_d.
template <int ROLE>
__device__ __forceinline__ void gemm_issue(int kind, Bars* b, uint8_t* smem, Sync& s, const uint8_t* gimg, uint32_t d_tmem) {
  if (ROLE == ROLE_PRODUCER) {
    if (kind == 0) produce(b, smem + SmemMap::RING, s, gimg, BIG_STAGES, STAGE_BYTES);
    else produce_single(b, smem + SmemMap::RING, s, gimg);
  } else if (ROLE == ROLE_MMA) {
    const uint32_t base = smem_u32(smem);
    if (kind == 0) mma_big(b, base + SmemMap::ACT, base + SmemMap::RING, s, d_tmem);
    else if (kind == 1) mma_l1(b, base + SmemMap::PIMG, base + SmemMap::RING, s, d_tmem);
    else mma_in(b, base + SmemMap::ACT, base + SmemMap::RING, s, d_tmem);
    mma_publish_d(b);
  } else {
    if (kind == 1) epi_publish_a(b);     // epilogue warps: TMEM reads done; row warps: [p|a|1] image written
    if (kind == 0) ++s.k_cnt;
  }
}
// Streamed first layer + layer 2 (or the Q net's): the first-layer result never sits in TMEM as a whole; its four
// 64-column chunks go through two buffers, chunk c+2 is issued when the epilogue has read chunk c, and the K-blocks
// of the big GEMM follow the h1 blocks the epilogue publishes.  Result: z2 in tm_work (d_full).
template <int ROLE>
__device__ __forceinline__ void fwd_pair_issue(Bars* b, uint8_t* smem, Sync& s, const uint8_t* l1_img, const uint8_t* big_img,
                                               uint32_t tm_z1c, uint32_t tm_work, long long* prof = nullptr) {
  if (ROLE == ROLE_PRODUCER) {
    produce_single(b, smem + SmemMap::RING, s, l1_img);
    produce(b, smem + SmemMap::RING, s, big_img, BIG_STAGES, STAGE_BYTES);
  } else if (ROLE == ROLE_MMA) {
    const uint32_t base = smem_u32(smem), p_addr = base + SmemMap::PIMG, ring = base + SmemMap::RING;
    mbar_wait(&b->a_full, s.a_cnt & 1, 10000 + __LINE__);
    ++s.a_cnt;
    if (prof) prof[21] = clock64();           // [p|a|1] image published
    const uint32_t slot = wait_single(b, s);
    const uint32_t bbase = ring + slot * STAGE_BYTES;
    if (prof) prof[22] = clock64();           // first-layer weight image in its slot
    mma_l1_chunk<FMT_F16>(b, p_addr, bbase, 0, tm_z1c);
    mma_l1_chunk<FMT_F16>(b, p_addr, bbase, 1, tm_z1c);
    if (prof) prof[23] = clock64();
    mma_l1_chunk<FMT_F16>(b, p_addr, bbase, 2, tm_z1c);
    if (prof) prof[24] = clock64();
    ++s.stage;
    consume_pad(b, s);                        // hands the empty slot to the big GEMM's first stages right away
    if (prof) prof[25] = clock64();
    // the last chunk waits for the epilogue to have read chunk 1, which happens about when h1 block 0 is published:
    // issuing it BEFORE the first big UMMAs keeps it from queueing behind them in the tensor pipe and frees the ring slot of
    // the first-layer image (behind the first two stages of K-block 0 it made the third stage wait 1.8 K cycles for that slot)
    mma_l1_chunk<FMT_F16>(b, p_addr, bbase, 3, tm_z1c);
    umma_commit(&b->empty[slot]);
    if (prof) prof[20] = clock64();              // first-layer chunk 3 issued, layer-2 GEMM starts
    mma_big<FMT_F16>(b, base + SmemMap::ACT, ring, s, tm_work, true, prof);
    mma_publish_d(b);
  } else {
    epi_publish_a(b);
    ++s.k_cnt;
  }
}
// Tail of a backward step: the first-layer pre-activations are recomputed chunk by chunk for act'(z1) (the [p|a|1]
// image of this step is still in place), then the input-gradient GEMM (do_gp) follows the delta1 blocks, then the
// delta1 / [p|1] images are contracted over the rows into the persistent D1 accumulator (do_d1).
template <int ROLE>
__device__ __forceinline__ void bwd_tail_issue(Bars* b, uint8_t* smem, Sync& s, const uint8_t* l1_img, const uint8_t* in_img,
                                               bool do_gp, bool do_d1, bool& d1_started, uint32_t tm_z1c, uint32_t tm_gp,
                                               uint32_t tm_d1, bool wait_p = false, bool release_img = false) {
  if (ROLE == ROLE_PRODUCER) {
    produce_single(b, smem + SmemMap::RING, s, l1_img);
    if (do_gp) produce_single(b, smem + SmemMap::RING, s, in_img);
  } else if (ROLE == ROLE_MMA) {
    const uint32_t base = smem_u32(smem), p_addr = base + SmemMap::PIMG, ring = base + SmemMap::RING;
    if (wait_p) {                                 // the [p|1] image of this step was written at the start of the step
      mbar_wait(&b->p_full, s.p_cnt & 1, 10000 + __LINE__);
      ++s.p_cnt;
    }
    const uint32_t slot = wait_single(b, s);
    const uint32_t bbase = ring + slot * STAGE_BYTES;
    for (int c = 0; c < 4; ++c) mma_l1_chunk<FMT_BF16>(b, p_addr, bbase, c, tm_z1c);   // backward side: bf16 [p|1] image + bf16 W1aug
    release_single(b, s, slot);
    // g_p K-block kb follows delta1 block kb.  D1 += delta1^T [p|1] is issued per 128-feature half: half 0 as soon as
    // delta1 blocks 0, 1 exist (it runs under the second half of the delta1 epilogue, when the tensor pipe has nothing
    // else to do), half 1 after g_p has been committed, so that it runs under the epilogue's lambda update and the start
    // of the next step (acc_done gates the next image writes)
    const uint32_t act_addr = base + SmemMap::ACT;
    const uint32_t islot = s.stage & (NSLOT - 1), ipar = (s.stage / NSLOT) & 1;
    const uint32_t ibase = ring + islot * STAGE_BYTES;
    for (int kb = 0; kb < 4; ++kb) {
      mbar_wait(&b->a_blk[kb], s.g_cnt & 1, 10000 + __LINE__);
      if (do_gp) {
        if (kb == 0) mbar_wait(&b->full[islot], ipar, 10000 + __LINE__);
        tc_fence_after();
        mma_in_block(act_addr, ibase, kb, tm_gp);
      } else {
        tc_fence_after();
      }
      if (kb == 1) {
        if (do_d1) mma_acc_half<32>(act_addr, p_addr, P_GROUP, tm_d1, 0, d1_started);
        if (release_img) umma_commit(&b->img_empty[0]);   // blocks 0, 1 of the image have been read for the last time
      }
    }
    ++s.g_cnt;
    if (do_gp) {
      release_single(b, s, islot);
      mma_publish_d(b);
      umma_commit(&b->gp_full);
    }
    if (do_d1) {
      mma_acc_half<32>(act_addr, p_addr, P_GROUP, tm_d1, 1, d1_started);
      d1_started = true;
      umma_commit(&b->acc_done);
    }
    if (release_img) umma_commit(&b->img_empty[1]);
  }
}
// D3 += h2^T [delta3|0]: the epilogue publishes (h2 image + delta3 image written); the UMMAs complete on d_full
// twice, once per 128-feature half, so that the delta2 epilogue can start on the first half of the image
template <int ROLE>
// h2_hi_only: large policy-gradient contractions (the hi-only dW2 record regime, api.cu: rec_hi_only) also take only the hi
// plane of h2 into dW3 -- the same 1/sqrt(K) averaging, emulated 1.1e-5 at 16,384 rows x 26 steps, and half the UMMAs
// between delta3 and the delta2 epilogue
__device__ __forceinline__ void d3_issue(Bars* b, uint8_t* smem, Sync& s, uint32_t d3_off, bool& d3_started, uint32_t tm_d3,
                                         bool lin = false, bool h2_hi_only = false) {
  if (ROLE == ROLE_MMA) {
    const uint32_t base = smem_u32(smem);
    mbar_wait(&b->a_full, s.a_cnt & 1, 10000 + __LINE__);
    ++s.a_cnt;
    tc_fence_after();
    mma_acc_half<16>(base + SmemMap::ACT, base + d3_off, 256, tm_d3, 0, d3_started, lin, h2_hi_only);
    mma_publish_d(b);                      // blocks 0, 1 of the h2 image may be overwritten
    if (lin) {                             // BPTT: the second half of the h2 image arrives separately
      mbar_wait(&b->img_full[1], (s.i_cnt - 1) & 1, 10000 + __LINE__);
      tc_fence_after();
    }
    mma_acc_half<16>(base + SmemMap::ACT, base + d3_off, 256, tm_d3, 1, d3_started, lin, h2_hi_only);
    umma_commit(&b->d_half);               // blocks 2, 3
    d3_started = true;
  } else if (ROLE == ROLE_EPI || ROLE == ROLE_ROW) {
    epi_publish_a(b);                      // epilogue warps: h2 image in place; row warps: delta3 image written
  }
}
// compatibility wrapper: issue + wait, A image published as a whole (self test)
template <int ROLE>
__device__ __forceinline__ void gemm(int kind, Bars* b, uint8_t* smem, Sync& s, const uint8_t* gimg, uint32_t d_tmem) {
  if (ROLE == ROLE_EPI && kind != 1)
    for (int kb = 0; kb < 4; ++kb) epi_block_done(b, kb);
  gemm_issue<ROLE>(kind, b, smem, s, gimg, d_tmem);
  if (ROLE == ROLE_EPI) epi_wait_d(b, s);
}

// ---- CTA prologue / epilogue -----------------------------------------------------------------------------
__device__ __forceinline__ Bars* cta_setup(uint8_t* smem, int a_full_count = EPI_THREADS, int mma_warp = EPI_WARPS + 1) {
  Bars* b = reinterpret_cast<Bars*>(smem + SmemMap::BARS);
  const int warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    for (int i = 0; i < NSLOT; ++i) { mbar_init(&b->full[i], 1); mbar_init(&b->empty[i], 1); }
    mbar_init(&b->a_full, a_full_count);
    for (int i = 0; i < 4; ++i) mbar_init(&b->a_blk[i], EPI_THREADS);
    mbar_init(&b->d_full, 1);
    mbar_init(&b->d_half, 1);
    for (int i = 0; i < 2; ++i) { mbar_init(&b->z_full[i], 1); mbar_init(&b->z_empty[i], EPI_THREADS); }
    mbar_init(&b->acc_done, 1);
    for (int i = 0; i < 4; ++i) mbar_init(&b->kb_done[i], 1);
    mbar_init(&b->p_full, ACT_ROWS);
    for (int i = 0; i < 2; ++i) { mbar_init(&b->img_empty[i], 2); mbar_init(&b->img_full[i], 1); }
    mbar_init(&b->gp_full, 1);
    fence_barrier_init();
  }
  if (warp == mma_warp) tmem_alloc(&b->tmem_base, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  return b;
}
__device__ __forceinline__ void cta_teardown(Bars* b, int mma_warp = EPI_WARPS + 1) {
  tc_fence_before();
  __syncthreads();
  if ((threadIdx.x >> 5) == mma_warp) tmem_dealloc(b->tmem_base, TMEM_COLS);
}

// ---- global weight-image packing (run once per set_weights) ------------------------------------------------
// big image: value(row, k) = src[row * rs + k * cs], 256 rows x 256 k -> 16 stages (kb, split, kh) of 256 rows x 64 B,
// SW64 K-major (8-row groups of 512 B, 16-byte chunk index ^ ((row >> 1) & 3))
template <bool F16>
__global__ void pack_big_image(const float* __restrict__ src, int rs, int cs, uint8_t* __restrict__ img) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // one thread per (row, 8-element chunk): 256 x 32
  if (idx >= 256 * 32) return;
  const int row = idx >> 5, cc = idx & 31;
  float x[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) x[e] = src[(size_t)row * rs + (size_t)(cc * 8 + e) * cs];
  uint4 h, l;
  split2x<F16>(x[0], x[1], h.x, l.x); split2x<F16>(x[2], x[3], h.y, l.y); split2x<F16>(x[4], x[5], h.z, l.z); split2x<F16>(x[6], x[7], h.w, l.w);
  const int kb = cc >> 3, kh = (cc >> 2) & 1, c = cc & 3;
  const size_t stage = (size_t)(kb * 4 + kh) * STAGE_BYTES;   // streamed in (k-block, split, k-half) order
  const uint32_t off = (row >> 3) * 512 + (row & 7) * 64 + ((c ^ ((row >> 1) & 3)) << 4);
  *reinterpret_cast<uint4*>(img + stage + off) = h;
  *reinterpret_cast<uint4*>(img + stage + 2 * STAGE_BYTES + off) = l;
}
// first-layer image: value(n, k) = scale * (k < in_dim ? W1[k][n] : (k == bias_k ? b1[n] : 0)); 256 rows x 16 k,
// (scale = log2(e) for the bf16 image of the BPTT recompute, whose z1 only feeds act'(z1), e.g. elu'(z1) = 2^(min(z1, 0) log2 e))
// INTERLEAVE K-major: [hi 8 KB | lo 8 KB]
template <bool F16>
__global__ void pack_l1_image(const float* __restrict__ W1, const float* __restrict__ b1, int in_dim, int bias_k,
                              uint8_t* __restrict__ img, float scale = 1.f) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // (n, k-half): 256 x 2
  if (idx >= 512) return;
  const int n = idx >> 1, kh = idx & 1;
  float x[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int k = kh * 8 + e;
    x[e] = scale * (k < in_dim ? W1[(size_t)k * H + n] : (k == bias_k ? b1[n] : 0.f));
  }
  uint4 h, l;
  split2x<F16>(x[0], x[1], h.x, l.x); split2x<F16>(x[2], x[3], h.y, l.y); split2x<F16>(x[4], x[5], h.z, l.z); split2x<F16>(x[6], x[7], h.w, l.w);
  const uint32_t off = il_chunk_off(n, kh);
  *reinterpret_cast<uint4*>(img + off) = h;
  *reinterpret_cast<uint4*>(img + 8192 + off) = l;
}
#ifndef MPG_ACT_UNIT   // non-template kernels are defined in api.cu's unit only (act_instances.cuh)
// input-gradient image: value(i, n) = i < in_dim ? W1[i][n] : 0; per 64-k block 32 rows (hi of rows 0..15, then lo of rows
// 0..15) x 128 B, SW128 K-major: 4 x 4 KB
__global__ void pack_in_image(const float* __restrict__ W1, int in_dim, uint8_t* __restrict__ img) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;   // (i, chunk): 16 x 32
  if (idx >= 512) return;
  const int i = idx >> 5, cc = idx & 31;
  float x[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) x[e] = i < in_dim ? W1[(size_t)i * H + cc * 8 + e] : 0.f;
  uint4 h, l;
  split2(x[0], x[1], h.x, l.x); split2(x[2], x[3], h.y, l.y); split2(x[4], x[5], h.z, l.z); split2(x[6], x[7], h.w, l.w);
  const int kb = cc >> 3, c = cc & 7;
  auto off = [&](int row) { return (uint32_t)(kb * 4096 + (row >> 3) * 1024 + (row & 7) * 128 + ((c ^ (row & 7)) << 4)); };
  *reinterpret_cast<uint4*>(img + off(i)) = h;
  *reinterpret_cast<uint4*>(img + off(16 + i)) = l;
}
#endif

#if defined(MPG_DEBUG_PROBES) && !defined(MPG_ACT_UNIT)
// ---- self test: the three GEMM kinds against caller-provided fp32 data ---------------------------------------
//   kind 0: Z[128 x 256] = X[128 x 256] . (image of Wt[256 x 256])^T
//   kind 1: Z[128 x 256] = X16[128 x 16] . (first-layer image)^T
//   kind 2: Z[128 x 16]  = X[128 x 256] . (input-gradient image)^T
__global__ void __launch_bounds__(CTA_THREADS, 1) selftest_kernel(int kind, const float* __restrict__ X,
                                                                 const uint8_t* __restrict__ img, float* __restrict__ Z,
                                                                 int repeats) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // SW128 needs 1024-byte alignment
  Bars* b = cta_setup(smem);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t tmem = b->tmem_base;
  Sync s;
  if (warp < EPI_WARPS) {
    const int row = (warp & 3) * 32 + lane, hc = warp >> 2;
    constexpr int CW = COLS_PER_WARP;
    for (int rep = 0; rep < repeats; ++rep) {
      if (kind >= 3) {          // timing probes: back-to-back big GEMMs on whatever the images hold, one wait at the end
        if (rep == repeats - 1) epi_wait_d(b, s);
        continue;
      }
      if (kind == 1) {
        if (hc == 0) {
          for (int kh = 0; kh < 2; ++kh) {
            float x[8];
            for (int e = 0; e < 8; ++e) x[e] = X[row * 16 + kh * 8 + e];
            uint4 h, l;
            split2h(x[0], x[1], h.x, l.x); split2h(x[2], x[3], h.y, l.y); split2h(x[4], x[5], h.z, l.z); split2h(x[6], x[7], h.w, l.w);
            *reinterpret_cast<uint4*>(smem + SmemMap::PIMG + p_chunk_off(row, kh)) = h;
            *reinterpret_cast<uint4*>(smem + SmemMap::PIMG + p_chunk_off(row, 2 + kh)) = l;
          }
        }
      } else {
        for (int cc = hc * (CW / 8); cc < (hc + 1) * (CW / 8); ++cc) {
          float x[8];
          for (int e = 0; e < 8; ++e) x[e] = X[row * 256 + cc * 8 + e];
          act_store8(smem + SmemMap::ACT, smem + SmemMap::ACT + ACT_SPLIT, row, cc, x);
        }
      }
      gemm<ROLE_EPI>(kind, b, smem, s, img, tmem + TM_WORK);
      const uint32_t lane_base = tmem + TM_WORK + ((uint32_t)((warp & 3) * 32) << 16);
      if (kind == 2) {
        if (hc == 0) {
          float v[16], v2[16];
          tmem_ld16(lane_base, v);
          tmem_ld16(lane_base + 16, v2);
          for (int j = 0; j < 16; ++j) Z[row * 16 + j] = v[j] + v2[j];
        }
      } else {
        for (int c0 = hc * CW; c0 < (hc + 1) * CW; c0 += 32) {
          float v[32];
          tmem_ld32(lane_base + c0, v);
          for (int j = 0; j < 32; ++j) Z[row * 256 + c0 + j] = v[j];
        }
      }
    }
    tc_fence_before();
  } else if (warp == EPI_WARPS) {
    if (lane == 0)
      for (int rep = 0; rep < repeats; ++rep)
        if (kind != 4) gemm<ROLE_PRODUCER>(kind == 3 ? 0 : kind, b, smem, s, img, 0);
  } else {
    if (lane == 0)
      for (int rep = 0; rep < repeats; ++rep) {
        if (kind == 3) {          // weights streamed through the ring, no epilogue in the loop
          mma_big<FMT_BF16>(b, smem_u32(smem) + SmemMap::ACT, smem_u32(smem) + SmemMap::RING, s, tmem + TM_WORK, false);
          if (rep == repeats - 1) mma_publish_d(b);
        } else if (kind == 4) {   // operands resident, no streaming: the tensor pipe's own rate for this shape
          constexpr uint32_t idesc = make_idesc(128, 256, 0, 0);
          const uint32_t act = smem_u32(smem) + SmemMap::ACT, ring = smem_u32(smem) + SmemMap::RING;
          for (int k = 0; k < 16; ++k) {
            const uint64_t ko = (uint64_t)((k & 3) * 2);
            const uint64_t dah = make_desc(act + (k >> 2) * ACT_BLOCK, 16, 1024, LAYOUT_SW128) + ko;
            const uint64_t dal = make_desc(act + ACT_SPLIT + (k >> 2) * ACT_BLOCK, 16, 1024, LAYOUT_SW128) + ko;
            const uint64_t dbh = make_desc(ring, 16, 1024, LAYOUT_SW128) + ko;
            const uint64_t dbl = make_desc(ring + 32768, 16, 1024, LAYOUT_SW128) + ko;
            umma_bf16(tmem + TM_WORK, dah, dbh, idesc, 1u);
            umma_bf16(tmem + TM_WORK, dal, dbh, idesc, 1u);
            umma_bf16(tmem + TM_WORK, dah, dbl, idesc, 1u);
          }
          if (rep == repeats - 1) mma_publish_d(b);
        } else {
          gemm<ROLE_MMA>(kind, b, smem, s, img, tmem + TM_WORK);
        }
      }
  }
  cta_teardown(b);
}
#endif

}  // namespace tc
}  // namespace mpg
