// Implicit-GEMM convolution for sm_100a: TMA -> shared memory -> tcgen05.mma -> TMEM -> fused epilogue.
//
// Replaces every nn.Conv2d (+ folded eval BatchNorm / bias / residual add / ReLU / GroupNorm statistics)
// on the SipMask inference path (reference: SipMask-mmdetection/mmdet/models/backbones/resnet.py:203-239,
// models/necks/fpn.py:138-178, ops/conv_module.py:124-132, models/anchor_heads/sipmask_head.py:241-287;
// the reference runs them through cuDNN + separate ATen kernels).
//
//   D[pixel, co] = sum_{tap, ci} A[pixel (+) tap, ci] * Wt[co, tap*Cin + ci]
//
//  * A (activations) is NHWC fp16.  One M-tile is a BH x BW patch of output pixels (BH*BW = 128); for every
//    filter tap the producer issues ONE 4-D TMA box {64 ch, BW, BH, 1} at the tap-shifted coordinate, so
//    im2col never exists in memory and zero padding is TMA out-of-bounds fill.  Stride-2 convolutions use
//    parity-split tensor maps (doubled global strides), the 7x7/2 stem an 8-pixel sliding-window map.
//  * W is [Cout, taps*Cin] fp16, K-major, loaded as {64, N_TILE} boxes.  Both operands use the 128-byte
//    swizzle, the canonical K-major UMMA layout (8-row groups 1024 B apart).
//  * One elected thread issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=N_TILE<=256, K=16), fp32
//    accumulators live in TMEM (double-buffered when 2*N_TILE <= 512 columns), tcgen05.commit releases
//    shared-memory stages and publishes finished accumulators through mbarriers.
//  * Persistent CTAs (one per SM), warp-specialised: warp 0 = TMA producer, warp 1 = MMA issuer,
//    warps 2..5 = epilogue (tcgen05.ld -> scale/bias/residual/ReLU/GN statistics -> global NHWC store).
#include <cuda.h>
#include <stdlib.h>

#include "common.cuh"

namespace smb {

constexpr int kMaxTaps = 9;
constexpr int kMaxMaps = 8;
constexpr int kMaxLevels = 5;
constexpr int kThreads = 352;          // warp 0 = TMA, warp 1 = MMA, warps 2..9 = epilogue (2 per TMEM lane quadrant),
                                       // warp 10 = staging ring: TMA stores of finished chunks + residual prefetch
constexpr int kStoreWarp = 10;
constexpr int kEpiThreads = 256;
constexpr int kABytes = 128 * 64 * 2;   // one A stage: 128 pixels x 64 channels fp16

// One pyramid level (or the only tensor) of a launch.  Convolutions whose weights are shared by several feature-pyramid
// levels (the FCOS towers and heads, sipmask_head.py:250-257) run as ONE launch over the union of the levels' tiles.
struct LevelDesc {
  int H_out, W_out, BH, BW, tiles_x, tiles_y;
  int tile_start;                 // first M-tile of this level in the launch-wide tile order
  int map0;                       // index of this level's first A tensor map
  void* out;
  const __half* residual;
  long long* gn_stats;            // fixed-point per-(image,group) {sum * 2^20, sumsq * 2^16}
  int res_h, res_w;
  int pad_;
};

struct ConvParams {
  CUtensorMap amap[kMaxMaps];
  CUtensorMap bmap;
  CUtensorMap rmap[kMaxLevels];   // per-level residual maps (res_tma): residual tiles are TMA-prefetched into smem
  CUtensorMap omap[kMaxLevels];   // per-level output maps for the TMA-store epilogue (fp16 outputs, n_tile % 64 == 0)
  LevelDesc lv[kMaxLevels];
  int num_levels;
  int tap_map[kMaxTaps], tap_dx[kMaxTaps], tap_dy[kMaxTaps];
  int num_taps, kb_per_tap;       // k-blocks (64 channels) per tap
  int n_img, tiles_m;
  int Cout, n_tile, n_tiles_n, stages, tmem_cols, num_acc;
  int cluster;                    // CTAs per cluster sharing (multicasting) the weight tile: 1, 2 or 4
  long long* dbg_ts;              // profiling only: clock64 stamps of CTA 0 (SMB_CONV_TS buffer), else null
  int epi_split;                  // 1: the two epilogue warp groups work on different 64-channel chunks (epilogue_split)
  int debug_mode;                 // profiling only (SMB_CONV_DEBUG): 1 = no MMAs (TMA pipeline only), 2 = no TMA (MMA only)
  int pair;                       // 1: tcgen05 cta_group::2 - two CTAs (SMs) compute one 256 x N tile, each holding half of B
  int out_pitch; int out_f32; int out_tma; int res_tma;
  int store_lag;                  // TMA stores kept in flight before a slot is recycled (1..4, < stage_slots)
  int stage_slots;                // staging ring: n_tile/64 (one tile) or 2*n_tile/64 (two tiles) chunk buffers of 128 px x 64 ch
  const float* bias; float alpha;
  int res_pitch; int res_mode;
  int gn_group;                   // channels per GroupNorm group (8 or 16), 0 = no statistics
  int relu;
};

// ------------------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// One elected lane of a fully converged warp.  Keeping the surrounding control flow warp-uniform (instead of an
// `if (lane == 0)` region) lets the compiler keep TMA / UMMA operands in uniform registers; a divergent region makes
// it wrap every UTMALDG / UTCHMMA in a per-lane "waterfall" loop (~200 cycles per instruction).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE;\n"
      "bra WAIT_LOOP;\n"
      "WAIT_DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_mc(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}
__device__ __forceinline__ uint32_t mapa_u32(uint32_t saddr, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(cta));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// cta_group::2 TMA loads: data lands in the issuing CTA's shared memory, completion is signalled on the LEADER CTA's barrier
__device__ __forceinline__ void tma_load_4d_2sm(void* dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(leader_bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_2sm(void* dst, const CUtensorMap* map, uint32_t leader_bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(leader_bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_commit2_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}
__device__ __forceinline__ void umma2_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, const void* src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(map),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// Explicit shared-window accesses.  In a cluster launch every generic->shared conversion costs an S2R SR_CgaCtaId (the
// compiler re-derives the CTA's window each time); the epilogue keeps 32-bit shared addresses instead.
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, const uint4& v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void mbar_arrive_a(uint32_t addr) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_a(uint32_t addr, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_LOOP_A:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra WAIT_DONE_A;\n"
      "bra WAIT_LOOP_A;\n"
      "WAIT_DONE_A:\n"
      "}\n" ::"r"(addr),
      "r"(parity)
      : "memory");
}
// value the compiler must keep in a register (kernel parameters are otherwise re-read from the constant bank inside loops)
__device__ __forceinline__ int opaque(int x) {
  asm volatile("" : "+r"(x));
  return x;
}
// wait that carries a data dependency on the 16 destination registers of an earlier (prefetched) tcgen05.ld, so that no
// consumer of v[] can be scheduled above it
__device__ __forceinline__ void tmem_ld_wait16(uint32_t* v) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3]), "+r"(v[4]), "+r"(v[5]), "+r"(v[6]), "+r"(v[7]), "+r"(v[8]),
                 "+r"(v[9]), "+r"(v[10]), "+r"(v[11]), "+r"(v[12]), "+r"(v[13]), "+r"(v[14]), "+r"(v[15])
               :
               : "memory");
}

// Packed fp32 pair add (FADD2 on sm_100: two independent IEEE adds per instruction) and fp32x2 -> fp16x2 pack with the ReLU
// folded into the conversion (F2FP.RELU).  The epilogue is issue-bound (DESIGN.md 6): ~12 instructions per output element.
__device__ __forceinline__ void fadd2(float& a0, float& a1, float b0, float b1) {
  unsigned long long ua, ub;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ua) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(ub) : "f"(b0), "f"(b1));
  asm("add.rn.f32x2 %0, %0, %1;" : "+l"(ua) : "l"(ub));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(ua));
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}
__device__ __forceinline__ uint32_t pack_f16x2_relu(float lo, float hi) {      // max(round(x), 0) == round(max(x, 0))
  uint32_t r;
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

// K-major, 128-byte swizzle shared-memory matrix descriptor (cute::UMMA::SmemDescriptor, sm_100):
//   [0,14) start>>4 | [16,30) LBO>>4 (unused for swizzled K-major, 1) | [32,46) SBO>>4 = 1024>>4 |
//   [46,48) version = 1 | [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_sdesc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::f16 instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 (1) @4, a/b format F16 (0),
// a/b K-major (0), n_dim = N>>3 @17, m_dim = M>>4 @24.
__device__ __forceinline__ uint32_t make_idesc(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ------------------------------------------------------------------------------------------------ kernel
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* v) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}

__device__ __forceinline__ void tmem_ld_wait32x2(uint32_t* a, uint32_t* b) {
  // one tcgen05.wait::ld for two prefetched 32-column loads; the "+r" operands pin every consumer of a[] / b[] below it
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(a[4]), "+r"(a[5]), "+r"(a[6]), "+r"(a[7]), "+r"(a[8]),
                 "+r"(a[9]), "+r"(a[10]), "+r"(a[11]), "+r"(a[12]), "+r"(a[13]), "+r"(a[14]), "+r"(a[15]), "+r"(a[16]),
                 "+r"(a[17]), "+r"(a[18]), "+r"(a[19]), "+r"(a[20]), "+r"(a[21]), "+r"(a[22]), "+r"(a[23]), "+r"(a[24]),
                 "+r"(a[25]), "+r"(a[26]), "+r"(a[27]), "+r"(a[28]), "+r"(a[29]), "+r"(a[30]), "+r"(a[31])
               :
               : "memory");
  asm volatile(""
               : "+r"(b[0]), "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(b[4]), "+r"(b[5]), "+r"(b[6]), "+r"(b[7]), "+r"(b[8]),
                 "+r"(b[9]), "+r"(b[10]), "+r"(b[11]), "+r"(b[12]), "+r"(b[13]), "+r"(b[14]), "+r"(b[15]), "+r"(b[16]),
                 "+r"(b[17]), "+r"(b[18]), "+r"(b[19]), "+r"(b[20]), "+r"(b[21]), "+r"(b[22]), "+r"(b[23]), "+r"(b[24]),
                 "+r"(b[25]), "+r"(b[26]), "+r"(b[27]), "+r"(b[28]), "+r"(b[29]), "+r"(b[30]), "+r"(b[31])
               :
               : "memory");
}


// work unit -> tile.  A unit is a group of `cluster` consecutive M-tiles that share one N-tile (their CTAs multicast the
// weight tile to each other); units of the same M-group with different N-tiles are adjacent so concurrently running
// clusters share the activation patches in L2.  A CTA whose M-tile index runs past the end gets a clamped tile and
// active == false (it still takes part in the multicast / barrier protocol but stores nothing).
struct TileCoord {
  int lvl, img, x0, y0, n0;
  bool active;
};

__device__ __forceinline__ int cdiv_dev(int a, int b) { return (a + b - 1) / b; }

// n / d and n % d for small non-negative n (< 2^22) without the ~30-instruction integer division: float reciprocal estimate
// plus one correction step (exact: the estimate is off by at most one).  The tile decode runs once per tile in every
// epilogue thread, on the critical path of the short-K (epilogue-bound) plans.
__device__ __forceinline__ int fast_divmod(int n, int d, int& rem) {
  int q = __float2int_rz(__int2float_rn(n) * __frcp_rn(__int2float_rn(d)));
  int r = n - q * d;
  if (r >= d) { ++q; r -= d; }
  if (r < 0) { --q; r += d; }
  rem = r;
  return q;
}

__device__ __forceinline__ TileCoord decode_tile(const ConvParams& p, int unit, int rank) {
  TileCoord t;
  int nt = 0, um = unit;
  if (p.n_tiles_n > 1) um = fast_divmod(unit, p.n_tiles_n, nt);
  int mt = um * p.cluster + rank;
  t.active = mt < p.tiles_m;
  if (!t.active) mt = p.tiles_m - 1;
  int l = 0;
#pragma unroll
  for (int i = 1; i < kMaxLevels; ++i)
    if (i < p.num_levels && mt >= p.lv[i].tile_start) l = i;
  mt -= p.lv[l].tile_start;
  int tx, ty;
  mt = fast_divmod(mt, p.lv[l].tiles_x, tx);
  t.img = fast_divmod(mt, p.lv[l].tiles_y, ty);
  t.lvl = l;
  t.x0 = tx * p.lv[l].BW;
  t.y0 = ty * p.lv[l].BH;
  t.n0 = nt * p.n_tile;
  return t;
}

#ifdef SMB_TRACE   // per-role, per-tile clock64 trace of CTA 0 (tools/conv_trace.py; tools/build_trace_lib.sh builds with -DSMB_TRACE)
#define TR(role, t, e) do { if (p.dbg_ts && blockIdx.x == 0 && (threadIdx.x & 31) == 0 && (t) < 16) \
    p.dbg_ts[64 + (role) * 64 + (int)(t) * 4 + (e)] = clock64(); } while (0)
#else
#define TR(role, t, e) do { } while (0)
#endif

// ---------------------------------------------------------------------------------------------------------------------------
// Split-group epilogue (TMA-store plans with bias, no GroupNorm, alpha == 1; residual none or TMA-staged).
//
// Measured (profiles/r02_conv_trace_*.txt, tools/conv_trace.py): on the short-K plans the tile period IS the epilogue - the
// TMA/MMA main loop alone runs at 0.7 us per 128 x 256 tile, the lockstep epilogue at 3.0-3.7 us - and a 64-channel chunk
// costs ~1300 cycles of which ~470 are the bare slot-wait / arrive skeleton: a serial chain of latencies (wait -> LDS ->
// tcgen05.wait::ld -> adds -> STS -> MEMBAR -> arrive) that the eight warps execute simultaneously, so nothing overlaps.
// Here the two warp groups (warps 2-5, 6-9: each covers the four TMEM lane quadrants) take ALTERNATE chunks: a warp drains
// all 64 channels of its 32 rows, and the chains of chunk g and chunk g+1 run concurrently.  The staging-ring protocol with
// the store warp is unchanged except that a slot is complete after 4 warp arrivals.
template <bool kPair, bool kRes, bool kRelu>
__device__ __forceinline__ void epilogue_split(const ConvParams& p, int cluster_id, int num_clusters, int total_units, int crank,
                                               uint32_t tmem_base, uint64_t* tfull_bar, uint64_t* tempty_bar, uint32_t stage_a,
                                               uint32_t rfull_a, uint32_t sfull_a, uint32_t sfree_a, int warp, int lane) {
  const int lane_grp = warp & 3, grp = (warp - 2) >> 2;
  const int row = lane_grp * 32 + lane;
  const int nch = p.n_tile >> 6, nslots = p.stage_slots, n_tile = p.n_tile, n_tiles_n = p.n_tiles_n;
  const float* __restrict__ bias = p.bias;
  uint32_t soff[8];                                  // this thread's row, 16-byte pieces in swizzled order
#pragma unroll
  for (int q = 0; q < 8; ++q) soff[q] = (uint32_t)row * 128u + (uint32_t)((q ^ (row & 7)) * 16);
  int acc = 0;
  uint32_t acc_ph = 0;
  int g0 = 0;                                        // chunk counter of this CTA at the start of the tile,
  int slot0 = 0;                                     // its ring slot and the slot's use parity
  uint32_t ph0 = 0;
  for (int unit = cluster_id; unit < total_units; unit += num_clusters, g0 += nch) {
    int nt = 0;
    if (n_tiles_n > 1) { int um = fast_divmod(unit, n_tiles_n, nt); (void)um; }
    const float* btile = bias + nt * n_tile;
    if (warp == 2) TR(2, g0 / nch, 0);
    mbar_wait(&tfull_bar[acc], acc_ph);
    if (warp == 2) TR(2, g0 / nch, 1);
    tc_fence_after();
    const uint32_t t_base = tmem_base + ((uint32_t)(lane_grp * 32) << 16) + (uint32_t)(acc * n_tile);
#pragma unroll 1
    for (int c64 = (g0 + grp) & 1 ? 1 : 0; c64 < nch; c64 += 2) {
      // chunks alternate between the groups over the CTA's whole chunk sequence: with an odd nch (1) the tiles alternate
      int slot = slot0 + c64;                          // nch <= nslots: at most one wrap
      uint32_t slot_ph = ph0;
      if (slot >= nslots) { slot -= nslots; slot_ph ^= 1u; }
      const uint32_t sbase = stage_a + (uint32_t)slot * 16384u;
      uint32_t va[32], vb[32];
      tmem_ld32(t_base + (uint32_t)(c64 * 64), va);
      tmem_ld32(t_base + (uint32_t)(c64 * 64 + 32), vb);
      const float4* b4 = reinterpret_cast<const float4*>(btile + c64 * 64);
      float4 bq[8];
#pragma unroll
      for (int q = 0; q < 8; ++q) bq[q] = __ldg(b4 + q);
      uint4 r[8];
      if (kRes) {
        mbar_wait_a(rfull_a + (uint32_t)slot * 8u, slot_ph);           // residual landed (and the slot's last store read out)
#pragma unroll
        for (int q = 0; q < 8; ++q) r[q] = lds128(sbase + soff[q]);
      } else {
        mbar_wait_a(sfree_a + (uint32_t)slot * 8u, slot_ph ^ 1u);      // the slot's previous TMA store has been read out
      }
      tmem_ld_wait32x2(va, vb);
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        uint32_t* v = h ? vb : va;
        float f[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
        if (h == 1) {
#pragma unroll
          for (int q = 0; q < 8; ++q) bq[q] = __ldg(b4 + 8 + q);
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          fadd2(f[4 * q], f[4 * q + 1], bq[q].x, bq[q].y);
          fadd2(f[4 * q + 2], f[4 * q + 3], bq[q].z, bq[q].w);
        }
        if (kRes) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const __half2* hh = reinterpret_cast<const __half2*>(&r[h * 4 + q]);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float2 a = __half22float2(hh[e]);
              fadd2(f[q * 8 + 2 * e], f[q * 8 + 2 * e + 1], a.x, a.y);
            }
          }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint4 o;
          uint32_t* ho = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
          for (int e = 0; e < 4; ++e)
            ho[e] = kRelu ? pack_f16x2_relu(f[q * 8 + 2 * e], f[q * 8 + 2 * e + 1]) : pack_f16x2(f[q * 8 + 2 * e], f[q * 8 + 2 * e + 1]);
          sts128(sbase + soff[h * 4 + q], o);
        }
      }
      fence_async_smem();                              // generic-proxy writes -> visible to the TMA store
      __syncwarp();
      if (lane == 0) mbar_arrive_a(sfull_a + (uint32_t)slot * 8u);       // 4 warps -> the store warp ships the slot
    }
    tc_fence_before();
    __syncwarp();
    if (lane == 0) {
      if (kPair && crank != 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty_bar[acc]), 0));
      else mbar_arrive(&tempty_bar[acc]);
    }
    if (warp == 2) TR(2, g0 / nch, 2);
    if (++acc == p.num_acc) { acc = 0; acc_ph ^= 1; }
    slot0 += nch;
    if (slot0 >= nslots) { slot0 -= nslots; ph0 ^= 1u; }
  }
}

// kPair = true: tcgen05 cta_group::2 instantiation (must be launched with 2-CTA clusters); false: single-CTA MMA.
template <bool kPair>
__global__ void __launch_bounds__(kThreads, 1) conv_gemm_kernel(const __grid_constant__ ConvParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  // the 128-byte swizzle atoms (8 rows x 128 B) must start on 1024-byte boundaries
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#define TS(slot) do { if (p.dbg_ts && blockIdx.x == 0 && (threadIdx.x & 31) == 0) p.dbg_ts[slot] = clock64(); } while (0)
  if (threadIdx.x == 0) TS(0);
  const int b_bytes = (kPair ? p.n_tile / 2 : p.n_tile) * 128;      // per-CTA bytes of one B stage
  uint8_t* sA = smem;
  uint8_t* sB = smem + (size_t)p.stages * kABytes;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sB + (size_t)p.stages * b_bytes);
  uint64_t* empty_bar = full_bar + p.stages;
  uint64_t* tfull_bar = empty_bar + p.stages;
  uint64_t* tempty_bar = tfull_bar + 2;
  // staging ring (TMA-store epilogue): slot = chunk counter % stage_slots
  uint64_t* rfull_bar = tempty_bar + 2;                               // [8] residual chunk landed in the slot (res_tma)
  uint64_t* sfull_bar = rfull_bar + 8;                                // [8] the 8 epilogue warps have written the slot
  uint64_t* sfree_bar = sfull_bar + 8;                                // [8] the slot's TMA store has been read out (no residual)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(sfree_bar + 8);
  float* s_bias = reinterpret_cast<float*>(tmem_slot + 4);          // [2][256] double-buffered per tile
  // Ring of staging chunks, each 128 px x 64 ch fp16 (128-byte swizzle).  The residual chunk is TMA-loaded INTO a slot, each
  // epilogue thread overwrites exactly the 64 bytes it read with its result, the store warp TMA-stores the slot and, once the
  // store has been read out, requests the residual of the chunk that will use the slot next.
  uint8_t* s_stage = smem + (size_t)p.stages * (kABytes + b_bytes) + 4096;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < kMaxMaps; ++i) tma_prefetch_desc(&p.amap[i]);
    tma_prefetch_desc(&p.bmap);
    if (kPair) {
      // full: leader's expect_tx arrive + peer's remote arrive; empty / tfull: one multicast tcgen05.commit;
      // tempty (used in the leader): 8 local + 8 remote epilogue warps
      for (int i = 0; i < p.stages; ++i) { mbar_init(&full_bar[i], 2); mbar_init(&empty_bar[i], 1); }
      for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 16); }
    } else {
      for (int i = 0; i < p.stages; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], (uint32_t)p.cluster); }
      for (int i = 0; i < 2; ++i) { mbar_init(&tfull_bar[i], 1); mbar_init(&tempty_bar[i], 8); }
    }
    for (int i = 0; i < 8; ++i) { mbar_init(&rfull_bar[i], 1); mbar_init(&sfull_bar[i], p.epi_split ? 4 : 8); mbar_init(&sfree_bar[i], 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if constexpr (kPair) tmem_alloc2(tmem_slot, (uint32_t)p.tmem_cols);
    else tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  }
  tc_fence_before();
  if (p.cluster > 1) cluster_sync_all();             // peers must see initialised barriers before any remote arrive
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  if (threadIdx.x == 0) TS(1);
  // Programmatic dependent launch: everything above (barrier init, TMEM allocation, descriptor prefetch) may overlap the
  // tail of the previous kernel in the stream; from here on we touch global memory, so wait for it to complete, and let
  // the next kernel begin its own prologue as SMs free up.
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  const int crank = (p.cluster > 1) ? (int)cluster_ctarank() : 0;
  const int cluster_id = blockIdx.x / p.cluster, num_clusters = gridDim.x / p.cluster;
  const uint16_t cmask = (uint16_t)((1u << p.cluster) - 1u);
  const int total_units = cdiv_dev(p.tiles_m, p.cluster) * p.n_tiles_n;
  const int kblocks = p.num_taps * p.kb_per_tap;
  const uint32_t stage_bytes = (uint32_t)(kABytes + b_bytes);

  if (warp == 0) {
    {
      // ===================== TMA producer (whole warp loops, one elected lane issues) =====================
      int s = 0;
      uint32_t ph = 0;
      bool first = true;
      const int b_part = b_bytes / p.cluster, n_part = p.n_tile / p.cluster;
      const uint32_t lbar0 = kPair ? mapa_u32(smem_u32(&full_bar[0]), 0) : 0u;     // leader's full_bar[0] (pair mode)
      const int nstages = p.stages, kb_per_tap = p.kb_per_tap, num_taps = p.num_taps;
      int plt = 0;
      for (int unit = cluster_id; unit < total_units; unit += num_clusters, ++plt) {
        const TileCoord tc = decode_tile(p, unit, crank);
        const int map0 = p.lv[tc.lvl].map0;
        for (int t = 0; t < num_taps; ++t) {
          const CUtensorMap* am = &p.amap[map0 + p.tap_map[t]];
          const int ax = tc.x0 + p.tap_dx[t], ay = tc.y0 + p.tap_dy[t];
          int kcoord = t * kb_per_tap * 64;
          for (int kc = 0; kc < kb_per_tap; ++kc, kcoord += 64) {
            if ((p.debug_mode & 3) != 2) {
              if (first) { TS(2); first = false; }
              mbar_wait(&empty_bar[s], ph ^ 1);    // every CTA of the cluster has finished reading stage s
              if (t == 0 && kc == 0) TR(0, plt, 0);
              if (elect_one()) {
                if constexpr (kPair) {
                  // each CTA loads its own 128 x 64 activation tile and its half of the weight tile; all bytes are
                  // accounted on the leader's barrier (the single MMA issuer waits there)
                  const uint32_t lbar = lbar0 + (uint32_t)s * 8u;
                  if (crank == 0) mbar_expect_tx(&full_bar[s], 2 * stage_bytes);
                  else mbar_arrive_cluster(lbar);
                  tma_load_4d_2sm(sA + (size_t)s * kABytes, am, lbar, kc * 64, ax, ay, tc.img);
                  tma_load_2d_2sm(sB + (size_t)s * b_bytes, &p.bmap, lbar, kcoord, tc.n0 + crank * (p.n_tile / 2));
                } else {
                  mbar_expect_tx(&full_bar[s], stage_bytes);
                  tma_load_4d(sA + (size_t)s * kABytes, am, &full_bar[s], kc * 64, ax, ay, tc.img);
                  if (p.cluster == 1) {
                    tma_load_2d(sB + (size_t)s * b_bytes, &p.bmap, &full_bar[s], kcoord, tc.n0);
                  } else {
                    // this CTA fetches 1/cluster of the weight tile and multicasts it into every CTA of the cluster
                    tma_load_2d_mc(sB + (size_t)s * b_bytes + (size_t)crank * b_part, &p.bmap, &full_bar[s], kcoord,
                                   tc.n0 + crank * n_part, cmask);
                  }
                }
              }
              __syncwarp();
              if (t == 0 && kc == 0) TR(0, plt, 1);
            }
            if (++s == nstages) { s = 0; ph ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    if (!kPair || crank == 0) {
      // ===================== MMA issuer (pair mode: the leader CTA issues for both SMs) =====================
      const uint32_t idesc = make_idesc(kPair ? 256 : 128, p.n_tile);
      int s = 0;
      uint32_t ph = 0, lt = 0;
      int acc = 0;
      uint32_t acc_ph = 0;
      const int nstages = p.stages, num_acc = p.num_acc;
      const uint32_t sA0 = smem_u32(sA), sB0 = smem_u32(sB);
      for (int unit = cluster_id; unit < total_units; unit += num_clusters, ++lt) {
        if (lt == 0) TS(3);
        mbar_wait(&tempty_bar[acc], acc_ph ^ 1);
        TR(1, lt, 0);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * p.n_tile);
        for (int kb = 0; kb < kblocks; ++kb) {
          if ((p.debug_mode & 3) != 2) mbar_wait(&full_bar[s], ph);
          if (lt == 0 && kb == 0) TS(4);
          if (kb == 0) TR(1, lt, 1);
          tc_fence_after();
          if (elect_one()) {
            if ((p.debug_mode & 3) == 1) {
              mbar_arrive(&empty_bar[s]);
            } else {
              const uint64_t adesc = make_sdesc(sA0 + (uint32_t)s * kABytes);
              const uint64_t bdesc = make_sdesc(sB0 + (uint32_t)s * (uint32_t)b_bytes);
#pragma unroll
              for (int k = 0; k < 4; ++k) {
                // advance 16 elements (32 B) along K inside the 128-byte swizzle atom: +2 in the >>4 start field
                if constexpr (kPair) umma2_f16(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) ? 1u : 0u);
                else umma_f16(d_tmem, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) ? 1u : 0u);
              }
              if constexpr (kPair) umma_commit2_mc(&empty_bar[s], 3);       // frees stage s in both CTAs of the pair
              else if (p.cluster == 1) umma_commit(&empty_bar[s]); // frees the smem stage when these MMAs retire
              else umma_commit_mc(&empty_bar[s], cmask);          // ... in every CTA of the cluster (peers write into it)
            }
          }
          __syncwarp();
          if (++s == nstages) { s = 0; ph ^= 1; }
        }
        if (lt == 0) TS(8);
        if (elect_one()) {
          if constexpr (kPair) umma_commit2_mc(&tfull_bar[acc], 3);      // accumulator halves complete in both CTAs
          else umma_commit(&tfull_bar[acc]);                   // accumulator complete
        }
        __syncwarp();
        TR(1, lt, 2);
        if (++acc == num_acc) { acc = 0; acc_ph ^= 1; }
      }
    }
  } else if (warp == kStoreWarp) {
    // ===================== staging-ring warp: TMA stores + residual prefetch =====================
    if (p.out_tma) {
      const int nch = p.n_tile >> 6, nslots = p.stage_slots;
      const int my_tiles = cluster_id < total_units ? (total_units - cluster_id + num_clusters - 1) / num_clusters : 0;
      const int total_chunks = (p.debug_mode & 256) ? 0 : my_tiles * nch;   // 256: epilogue skips the chunk loop
      // residual request for chunk g (tile g / nch of this CTA, 64-channel chunk g % nch) into slot g % nslots
      auto request_residual = [&](int g) {
        const int t = g / nch, c = g - t * nch;
        const TileCoord tr = decode_tile(p, cluster_id + t * num_clusters, crank);
        const int sl = g % nslots;
        if (tr.active) {
          mbar_expect_tx(&rfull_bar[sl], 16384);
          tma_load_4d(s_stage + (size_t)sl * 16384, &p.rmap[tr.lvl], &rfull_bar[sl], tr.n0 + c * 64, tr.x0, tr.y0, tr.img);
        } else {
          mbar_arrive(&rfull_bar[sl]);
        }
      };
      if (p.res_tma && elect_one()) {
        for (int g = 0; g < nslots && g < total_chunks; ++g) request_residual(g);
      }
      __syncwarp();
      int slot = 0, c = 0, t = 0;
      uint32_t slot_ph = 0;
      TileCoord tc = decode_tile(p, cluster_id, crank);
      for (int g = 0; g < total_chunks; ++g) {
        mbar_wait(&sfull_bar[slot], slot_ph);
        if (c == 0) TR(3, t, 0);
        if (c == nch - 1) TR(3, t, 2);
        if (elect_one()) {
          if (tc.active && !(p.debug_mode & 8))
            tma_store_4d(&p.omap[tc.lvl], s_stage + (size_t)slot * 16384, tc.n0 + c * 64, tc.x0, tc.y0, tc.img);
          bulk_commit();
          // release a slot once its store has been read out: the previous chunk's (this chunk's own store keeps running),
          // or this chunk's at once when the ring has a single slot
          // (a deeper lag - more stores in flight - was measured slower: it delays the residual requests, r01 run 42)
          int h = -1;
          if (nslots == 1) { bulk_wait_read<0>(); h = g; }
          else if (g >= p.store_lag) {
            // keep `store_lag` stores in flight: recycle the slot of chunk g - lag once its store has been read out
            switch (p.store_lag) {
              case 1: bulk_wait_read<1>(); break;
              case 2: bulk_wait_read<2>(); break;
              case 3: bulk_wait_read<3>(); break;
              default: bulk_wait_read<4>(); break;
            }
            h = g - p.store_lag;
          }
          if (h >= 0) {
            if (p.res_tma) {
              if (h + nslots < total_chunks) { fence_async_smem(); request_residual(h + nslots); }
            } else {
              mbar_arrive(&sfree_bar[h % nslots]);
            }
          }
        }
        __syncwarp();
        if (c == 0) TR(3, t, 1);
        if (c == nch - 1) TR(3, t, 3);
        if (++slot == nslots) { slot = 0; slot_ph ^= 1; }
        if (++c == nch) {
          c = 0;
          ++t;
          if (g + 1 < total_chunks) tc = decode_tile(p, cluster_id + t * num_clusters, crank);
        }
      }
      if (elect_one()) bulk_wait_read<0>();          // staging slots must outlive their TMA stores
      __syncwarp();
    }
  } else if (p.epi_split) {
    // ===================== epilogue warps (2..9), split groups =====================
    const uint32_t stage_a = smem_u32(s_stage);
    const uint32_t rfull_a = smem_u32(rfull_bar), sfull_a = smem_u32(sfull_bar), sfree_a = smem_u32(sfree_bar);
    if (p.res_tma) {
      if (p.relu) epilogue_split<kPair, true, true>(p, cluster_id, num_clusters, total_units, crank, tmem_base, tfull_bar, tempty_bar,
                                                    stage_a, rfull_a, sfull_a, sfree_a, warp, lane);
      else epilogue_split<kPair, true, false>(p, cluster_id, num_clusters, total_units, crank, tmem_base, tfull_bar, tempty_bar,
                                              stage_a, rfull_a, sfull_a, sfree_a, warp, lane);
    } else {
      if (p.relu) epilogue_split<kPair, false, true>(p, cluster_id, num_clusters, total_units, crank, tmem_base, tfull_bar, tempty_bar,
                                                     stage_a, rfull_a, sfull_a, sfree_a, warp, lane);
      else epilogue_split<kPair, false, false>(p, cluster_id, num_clusters, total_units, crank, tmem_base, tfull_bar, tempty_bar,
                                               stage_a, rfull_a, sfull_a, sfree_a, warp, lane);
    }
  } else {
    // ===================== epilogue warps (2..9) =====================
    // Two warps per TMEM lane quadrant (a warp may only touch lanes 32*(warp%4)..+31); the pair splits the tile's
    // columns, which doubles the loads/stores in flight of this latency-bound phase.
    const int lane_grp = warp & 3;
    const int col_half = (warp - 2) >> 2;
    const int row = lane_grp * 32 + lane;
    const int et = threadIdx.x - 64;                 // 0..255 within the epilogue group
    int split = ((p.n_tile / 2 + 31) / 32) * 32;
    if (split > p.n_tile) split = p.n_tile;
    const int c_begin = col_half ? split : 0, c_end = col_half ? p.n_tile : split;
    uint32_t lt = 0;
    int acc = 0;
    uint32_t acc_ph = 0;
    int slot = 0;                                    // staging ring position of the next chunk, and its use parity
    uint32_t slot_ph = 0;
    const int nslots = p.stage_slots;
    const bool single_n = p.n_tiles_n == 1;
    // loop-invariant parameters and shared addresses of the chunk loop, pinned in registers
    const int o_flags = opaque((p.bias ? 1 : 0) | (p.relu ? 2 : 0) | (p.res_tma ? 4 : 0) | (p.gn_group ? 8 : 0) |
                               (p.alpha != 1.0f ? 16 : 0));
    const int o_dbg = opaque(p.debug_mode);
    const float o_alpha = __int_as_float(opaque(__float_as_int(p.alpha)));
    const uint32_t stage_a = smem_u32(s_stage), bias_a = smem_u32(s_bias);
    const uint32_t rfull_a = smem_u32(rfull_bar), sfull_a = smem_u32(sfull_bar), sfree_a = smem_u32(sfree_bar);
    for (int unit = cluster_id; unit < total_units; unit += num_clusters, ++lt) {
      const TileCoord tc = decode_tile(p, unit, crank);
      const LevelDesc& L = p.lv[tc.lvl];
#define TS2(slot) do { if (lt == 1 && warp == 2) TS(slot); } while (0)
#ifdef SMB_TS_FINE                                   // per-chunk stamps (tools/conv_timeline.py; build with -DSMB_TS_FINE)
#define TS3(slot) TS2(slot)
#else
#define TS3(slot) do { } while (0)
#endif
      TS2(16);
      if (warp == 2) TR(2, lt, 0);
      const int bw_shift = 31 - __clz(L.BW);            // BW is a power of two (choose_patch)
      const int iy = row >> bw_shift, ix = row & (L.BW - 1);
      const int x = tc.x0 + ix, y = tc.y0 + iy, n0 = tc.n0;
      const bool valid = tc.active && (x < L.W_out) && (y < L.H_out);
      const size_t pix = ((size_t)tc.img * L.H_out + y) * L.W_out + x;
      const __half* res_row = nullptr;
      if (valid) {
        if (p.res_mode == 1) {
          res_row = L.residual + pix * p.res_pitch;
        } else if (p.res_mode == 2) {
          // F.interpolate(mode='nearest', size=...) : src = min(floor(dst * in/out), in-1)   (fpn.py:149-152)
          const int sy = min((int)floorf((float)y * ((float)L.res_h / (float)L.H_out)), L.res_h - 1);
          const int sx = min((int)floorf((float)x * ((float)L.res_w / (float)L.W_out)), L.res_w - 1);
          res_row = L.residual + (((size_t)tc.img * L.res_h + sy) * L.res_w + sx) * p.res_pitch;
        }
      }
      // residual prefetch (one 32-channel chunk ahead of the accumulator drain)
      uint4 rcur[4], rnext[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) { rcur[j] = make_uint4(0u, 0u, 0u, 0u); rnext[j] = make_uint4(0u, 0u, 0u, 0u); }
      if (res_row && c_begin < c_end && !p.out_tma) {
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (n0 + c_begin + j * 8 + 8 <= p.Cout && c_begin + j * 8 < c_end)
            rcur[j] = __ldg(reinterpret_cast<const uint4*>(res_row + n0 + c_begin + j * 8));
      }
      TS2(17);
      // stage this tile's bias slice in shared memory (double-buffered; one named barrier per tile).  With a single N
      // tile the slice never changes: staged once, before the first tile.
      float* sb = s_bias + (single_n ? 0 : (lt & 1) * 256);
      if (!single_n || lt == 0) {
        if (p.bias) {
          for (int c = et; c < p.n_tile; c += kEpiThreads) sb[c] = (n0 + c < p.Cout) ? __ldg(p.bias + n0 + c) : 0.f;
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");
      }
      TS2(18);
      mbar_wait(&tfull_bar[acc], acc_ph);
      TS2(19);
      if (warp == 2) TR(2, lt, 1);
      if (lt == 0 && warp == 2 && lane == 0) TS(9);
      tc_fence_after();
      const uint32_t t_base = tmem_base + ((uint32_t)(lane_grp * 32) << 16) + (uint32_t)(acc * p.n_tile);
      if (p.out_tma && (o_dbg & 256)) {
        // profiling: accumulator released untouched (bare main-loop period)
      } else if (p.out_tma) {
        // ---------- staged epilogue: TMEM -> registers -> swizzled smem tile (128 px x 64 ch) -> TMA store ----------
        // All 8 warps work on the same 64-channel chunk (warp pair = two 32-channel halves of a lane quadrant); the
        // scattered per-thread 16-byte global stores of the direct path become one coalesced, bounds-clipped TMA store.
        const int nch = p.n_tile >> 6;
        uint4 rc[4], rn[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { rc[j] = make_uint4(0u, 0u, 0u, 0u); rn[j] = make_uint4(0u, 0u, 0u, 0u); }
        const bool res_smem = p.res_tma && tc.active;
        if (res_row && !res_smem) {
#pragma unroll
          for (int j = 0; j < 4; ++j) rc[j] = __ldg(reinterpret_cast<const uint4*>(res_row + n0 + col_half * 32 + j * 8));
        }
        // Half-chunk software pipeline: while 16 accumulator columns are being turned into fp16, the tcgen05.ld of the next
        // 16 is in flight (same register budget as one 32-column load).
        uint32_t va[16], vb[16];
        tmem_ld16(t_base + (uint32_t)(col_half * 32), va);
        // The chunk loop is rolled (the body is ~400 SASS instructions instead of ~3000 straight-line ones per tile, and
        // the GroupNorm partials need no dynamically indexed array).  NOTE: rolling it did NOT change the measured
        // epilogue time (profiles/r01_conv_concurrency_h.txt, run 45); why a chunk still costs ~1.1-1.4k cycles with all
        // of its work disabled (profiles/r01_epilogue_ablation_debug_bits.txt) is not yet attributed - see DESIGN.md 7.
#pragma unroll 1
        for (int c64 = 0; c64 < nch; ++c64) {
          {
            const int cc = c64 * 64 + col_half * 32;     // first of this thread's 32 columns inside the tile
            float gv[8];                                   // GroupNorm partials of this chunk: [group of 8 ch][sum, sumsq]
#pragma unroll
            for (int j = 0; j < 8; ++j) gv[j] = 0.f;
            if (res_row && !res_smem && c64 + 1 < nch) {
#pragma unroll
              for (int j = 0; j < 4; ++j) rn[j] = __ldg(reinterpret_cast<const uint4*>(res_row + n0 + cc + 64 + j * 8));
            }
            const uint32_t srow = stage_a + (uint32_t)slot * 16384u + (uint32_t)row * 128u;   // this thread's staging row
            if (o_flags & 4) {
              // the slot's previous store has been read out AND this chunk's residual has landed in it (inactive tiles:
              // the store warp arrives without a load)
              mbar_wait_a(rfull_a + (uint32_t)slot * 8u, slot_ph);
              if (res_smem) {
#pragma unroll
                for (int j = 0; j < 4; ++j) rc[j] = lds128(srow + (uint32_t)(((col_half * 4 + j) ^ (row & 7)) * 16));
              }
            } else {
              mbar_wait_a(sfree_a + (uint32_t)slot * 8u, slot_ph ^ 1);       // the slot's previous TMA store has been read out
            }
            TS3(20 + 4 * c64);
            if (warp == 2 && lt == 2) TR(4, c64, 0);
            if (!(o_dbg & 512)) {
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              uint32_t* v = h ? vb : va;
              if (!(o_dbg & 128)) {
                tmem_ld_wait16(v);
                if (h == 0) tmem_ld16(t_base + (uint32_t)(cc + 16), vb);
                else if (c64 + 1 < nch) tmem_ld16(t_base + (uint32_t)(cc + 64), va);
              }
              if (h == 0) TS3(21 + 4 * c64);
              if (h == 0 && warp == 2 && lt == 2) TR(4, c64, 1);
              if (h == 1 && warp == 2 && lt == 2) TR(5, c64, 0);
              float f[16];
#pragma unroll
              for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[j]);
              if ((o_flags & 1) && !(o_dbg & 64)) {
                const uint32_t ba = bias_a + (uint32_t)((single_n ? 0 : (int)(lt & 1) * 256) + cc + h * 16) * 4u;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  const uint4 b = lds128(ba + (uint32_t)j * 16u);
                  fadd2(f[4 * j], f[4 * j + 1], __uint_as_float(b.x), __uint_as_float(b.y));
                  fadd2(f[4 * j + 2], f[4 * j + 3], __uint_as_float(b.z), __uint_as_float(b.w));
                }
              }
              if (o_flags & 16) {
#pragma unroll
                for (int j = 0; j < 16; ++j) f[j] *= o_alpha;
              }
              if ((res_row || res_smem) && !(o_dbg & 64)) {
#pragma unroll
                for (int j = 0; j < 2; ++j) {
                  const __half2* hh = reinterpret_cast<const __half2*>(&rc[h * 2 + j]);
#pragma unroll
                  for (int e = 0; e < 4; ++e) {
                    const float2 a = __half22float2(hh[e]);
                    fadd2(f[j * 8 + 2 * e], f[j * 8 + 2 * e + 1], a.x, a.y);
                  }
                }
              }
              if ((o_flags & 8) && valid && !(o_dbg & 4)) {
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                  float sg = 0.f, qg = 0.f;
#pragma unroll
                  for (int e = 0; e < 8; ++e) { sg += f[g * 8 + e]; qg += f[g * 8 + e] * f[g * 8 + e]; }
                  gv[(h * 2 + g) * 2] = sg;
                  gv[(h * 2 + g) * 2 + 1] = qg;
                }
              }
              // swizzled staging write: row = pixel, 16-byte chunk index ^= (row & 7); ReLU on the packed halves
              // (max(round(x), 0) == round(max(x, 0)): rounding is monotonic and 0 is exact)
#pragma unroll
              for (int j = 0; j < 2; ++j) {
                uint4 o;
                uint32_t* ho = reinterpret_cast<uint32_t*>(&o);
                if (o_flags & 2) {
#pragma unroll
                  for (int e = 0; e < 4; ++e) ho[e] = pack_f16x2_relu(f[j * 8 + 2 * e], f[j * 8 + 2 * e + 1]);
                } else {
#pragma unroll
                  for (int e = 0; e < 4; ++e) ho[e] = pack_f16x2(f[j * 8 + 2 * e], f[j * 8 + 2 * e + 1]);
                }
                const int chunk = (col_half * 4 + h * 2 + j) ^ (row & 7);
                if (!(o_dbg & 32)) sts128(srow + (uint32_t)(chunk * 16), o);
              }
              if (h == 0 && warp == 2 && lt == 2) TR(5, c64, 1);
            }
            }
            if ((o_flags & 8) && !(o_dbg & 4)) {
              // 32 lanes x 8 partials -> lane j (j < 8) ends up with the warp total of partial j (recursive halving over
              // lane bits 2..0, then two full exchanges over bits 3, 4: 9 shuffles), then ONE 64-bit fixed-point atomic
              // per partial (integer adds are associative: bit-reproducible statistics).
#pragma unroll
              for (int off = 4; off >= 1; off >>= 1) {
                const bool up = (lane & off) != 0;
#pragma unroll
                for (int i = 0; i < off; ++i) {
                  const float send = up ? gv[i] : gv[i + off];
                  const float keep = up ? gv[i + off] : gv[i];
                  gv[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
                }
              }
              gv[0] += __shfl_xor_sync(0xffffffffu, gv[0], 8);
              gv[0] += __shfl_xor_sync(0xffffffffu, gv[0], 16);
              if (lane < 8 && tc.active) {
                // lane partial g covers 8 channels; with 16-channel groups two adjacent partials add into one slot
                const int g = lane >> 1, kind = lane & 1;
                int grp = ((n0 + cc) >> 3) + g;
                if (p.gn_group == 16) grp >>= 1;
                const int ngroups = p.Cout / p.gn_group;
                unsigned long long* st = reinterpret_cast<unsigned long long*>(L.gn_stats) + ((size_t)tc.img * ngroups + grp) * 2 + kind;
                atomicAdd(st, (unsigned long long)__float2ll_rn(gv[0] * (kind ? kGnSqScale : kGnSumScale)));
              }
            }
            TS3(41);
            if (warp == 2 && lt == 2) TR(4, c64, 2);
            if (!(o_dbg & 16)) fence_async_smem();         // generic-proxy writes -> visible to the TMA store
            if (warp == 2 && lt == 2) TR(5, c64, 2);
            __syncwarp();
            if (lane == 0) mbar_arrive_a(sfull_a + (uint32_t)slot * 8u);  // 8 warps -> the store warp ships the slot
            TS3(22 + 4 * c64);
            if (warp == 2 && lt == 2) TR(4, c64, 3);
            if (++slot == nslots) { slot = 0; slot_ph ^= 1; }
#pragma unroll
            for (int j = 0; j < 4; ++j) rc[j] = rn[j];
          }
        }
      } else
      for (int c0 = c_begin; c0 < c_end; c0 += 32) {
        if (res_row && c0 + 32 < c_end) {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (n0 + c0 + 32 + j * 8 + 8 <= p.Cout && c0 + 32 + j * 8 < c_end)
              rnext[j] = __ldg(reinterpret_cast<const uint4*>(res_row + n0 + c0 + 32 + j * 8));
        }
        uint32_t v[32];
        if (c0 + 32 <= c_end) {
          tmem_ld32(t_base + (uint32_t)c0, v);
        } else {                                     // 16-column tail
          tmem_ld16(t_base + (uint32_t)c0, v);
#pragma unroll
          for (int j = 16; j < 32; ++j) v[j] = 0u;
        }
        tmem_ld_wait();
#pragma unroll
        for (int h = 0; h < 2; ++h) {                // two 16-channel halves
          const int ch0 = n0 + c0 + h * 16;
          if (c0 + h * 16 >= c_end || ch0 >= p.Cout) continue;     // warp-uniform
          float f[16];
#pragma unroll
          for (int j = 0; j < 16; ++j) f[j] = __uint_as_float(v[h * 16 + j]);
          if (p.bias) {
            const float4* b4 = reinterpret_cast<const float4*>(sb + c0 + h * 16);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 b = b4[j];
              f[4 * j] += b.x; f[4 * j + 1] += b.y; f[4 * j + 2] += b.z; f[4 * j + 3] += b.w;
            }
          }
          if (p.alpha != 1.0f) {
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] *= p.alpha;
          }
          if (res_row) {
            const __half2* ha = reinterpret_cast<const __half2*>(&rcur[2 * h]);
            const __half2* hb = reinterpret_cast<const __half2*>(&rcur[2 * h + 1]);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float2 a = __half22float2(ha[j]), b = __half22float2(hb[j]);
              f[2 * j] += a.x; f[2 * j + 1] += a.y;
              f[8 + 2 * j] += b.x; f[8 + 2 * j + 1] += b.y;
            }
          }
          if (p.gn_group && !(p.debug_mode & 4)) {
            // per-(image, group) sum / sum of squares of the conv output (pre-activation), fp32 in-warp, then
            // 64-bit fixed-point integer atomics (associative -> bit-reproducible run to run).
            float s0 = 0.f, q0 = 0.f, s1 = 0.f, q1 = 0.f;
            if (valid) {
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                s0 += f[j]; q0 += f[j] * f[j];
                s1 += f[8 + j]; q1 += f[8 + j] * f[8 + j];
              }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
              s0 += __shfl_xor_sync(0xffffffffu, s0, o);
              q0 += __shfl_xor_sync(0xffffffffu, q0, o);
              s1 += __shfl_xor_sync(0xffffffffu, s1, o);
              q1 += __shfl_xor_sync(0xffffffffu, q1, o);
            }
            if (lane == 0) {
              const int ngroups = p.Cout / p.gn_group;
              unsigned long long* st = reinterpret_cast<unsigned long long*>(L.gn_stats) + (size_t)tc.img * ngroups * 2;
              if (p.gn_group == 8) {
                const int g = ch0 >> 3;
                atomicAdd(st + g * 2, (unsigned long long)__float2ll_rn(s0 * kGnSumScale));
                atomicAdd(st + g * 2 + 1, (unsigned long long)__float2ll_rn(q0 * kGnSqScale));
                atomicAdd(st + g * 2 + 2, (unsigned long long)__float2ll_rn(s1 * kGnSumScale));
                atomicAdd(st + g * 2 + 3, (unsigned long long)__float2ll_rn(q1 * kGnSqScale));
              } else {
                const int g = ch0 >> 4;
                atomicAdd(st + g * 2, (unsigned long long)__float2ll_rn((s0 + s1) * kGnSumScale));
                atomicAdd(st + g * 2 + 1, (unsigned long long)__float2ll_rn((q0 + q1) * kGnSqScale));
              }
            }
          }
          if (p.relu) {
#pragma unroll
            for (int j = 0; j < 16; ++j) f[j] = fmaxf(f[j], 0.f);
          }
          if (valid && !(p.debug_mode & 8)) {
            if (p.out_f32) {
              float4* o = reinterpret_cast<float4*>(reinterpret_cast<float*>(L.out) + pix * p.out_pitch + ch0);
#pragma unroll
              for (int j = 0; j < 4; ++j) o[j] = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
            } else {
              uint4 oa, ob;
              __half2* ha = reinterpret_cast<__half2*>(&oa);
              __half2* hb = reinterpret_cast<__half2*>(&ob);
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                ha[j] = __floats2half2_rn(f[2 * j], f[2 * j + 1]);
                hb[j] = __floats2half2_rn(f[8 + 2 * j], f[8 + 2 * j + 1]);
              }
              uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<__half*>(L.out) + pix * p.out_pitch + ch0);
              o[0] = oa;
              o[1] = ob;
            }
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) rcur[j] = rnext[j];
      }
      if (lt == 0 && warp == 2 && lane == 0) TS(10);
      TS2(36);
      // this warp has drained its share of the accumulator
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (kPair && crank != 0) mbar_arrive_cluster(mapa_u32(smem_u32(&tempty_bar[acc]), 0));
        else mbar_arrive(&tempty_bar[acc]);
      }
      if (warp == 2) TR(2, lt, 2);
      if (++acc == p.num_acc) { acc = 0; acc_ph ^= 1; }
    }
  }

  if (threadIdx.x == 0) TS(11);
  tc_fence_before();
  if (p.cluster > 1) cluster_sync_all();             // no CTA may exit while peers can still multicast to / arrive on it
  else __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if constexpr (kPair) tmem_dealloc2(tmem_base, (uint32_t)p.tmem_cols);
    else tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Short-K 1x1 convolutions (ResNet conv1 / conv3 / shortcut with K <= 256): ONE 128 x 128 tile per CTA, no persistent loop,
// no staging ring, several CTAs resident per SM.
//
// Why a second kernel: for these shapes the persistent kernel above spends ~3.3 us per 128-pixel tile even with its whole
// epilogue switched off (profiles/r02_conv_diag_short_k.txt: 39.7 -> 35.8 us with TMEM loads, math, staging writes, fence and
// stores disabled) - the tile time is the latency of the load -> MMA -> commit -> epilogue -> recycle chain of ONE CTA per
// SM, which a K = 64 tile (one k-block) cannot amortise.  Here the chain is still there, but 2-3 independent CTAs per SM
// (64-96 KB shared memory, 128 TMEM columns, 160 threads each) overlap each other's latencies.
//
//   warp 0      : TMEM alloc, TMA loads (A k-blocks, weight k-blocks, residual tile) and tcgen05.mma issue (one elected lane)
//   warps 1..4  : epilogue, one TMEM lane quadrant each: tcgen05.ld 32 columns -> +bias (+residual from the staging tile)
//                 -> ReLU -> fp16 -> back into the swizzled staging tile; then two 64-channel TMA stores.
constexpr int kSmallThreads = 160;
constexpr int kSmallN = 128;

__global__ void __launch_bounds__(kSmallThreads) conv1x1_small_kernel(const __grid_constant__ ConvParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nst = p.stages;                                   // 1 or 2 operand stages
  uint8_t* sA = smem;                                         // [nst][128 px x 64 ch]
  uint8_t* sB = smem + (size_t)nst * kABytes;                 // [nst][128 co x 64 k]
  uint8_t* s_stage = sB + (size_t)nst * kABytes;              // [2][128 px x 64 ch]: residual in, result out
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_stage + 2 * 16384);
  uint64_t* empty_bar = full_bar + 2;
  uint64_t* tfull_bar = empty_bar + 2;
  uint64_t* rfull_bar = tfull_bar + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rfull_bar + 1);

  if (warp == 0) {
    if (lane == 0) {
      tma_prefetch_desc(&p.amap[0]);
      tma_prefetch_desc(&p.bmap);
      tma_prefetch_desc(&p.omap[0]);
      for (int i = 0; i < 2; ++i) { mbar_init(&full_bar[i], 1); mbar_init(&empty_bar[i], 1); }
      mbar_init(tfull_bar, 1);
      mbar_init(rfull_bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    tmem_alloc(tmem_slot, (uint32_t)kSmallN);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");

  // tile of this CTA: N tiles of one M tile are adjacent in the grid (they read the same activation patch: L2 reuse)
  const LevelDesc& L = p.lv[0];
  int nt;
  int mt = fast_divmod((int)blockIdx.x, p.n_tiles_n, nt);
  int tx, ty;
  mt = fast_divmod(mt, L.tiles_x, tx);
  const int img = fast_divmod(mt, L.tiles_y, ty);
  const int x0 = tx * L.BW, y0 = ty * L.BH, n0 = nt * kSmallN;
  const int kblocks = p.kb_per_tap;                            // one tap (1x1), Cin / 64 k-blocks

  if (warp == 0) {
    const uint32_t idesc = make_idesc(128, kSmallN);
    const uint32_t sA0 = smem_u32(sA), sB0 = smem_u32(sB);
    const int ax = x0 + p.tap_dx[0], ay = y0 + p.tap_dy[0];
    if (elect_one()) {
      if (p.res_tma) {                                       // residual tile: two 64-channel boxes into the staging tile
        mbar_expect_tx(rfull_bar, 2 * 16384);
        tma_load_4d(s_stage, &p.rmap[0], rfull_bar, n0, x0, y0, img);
        tma_load_4d(s_stage + 16384, &p.rmap[0], rfull_bar, n0 + 64, x0, y0, img);
      }
      for (int kb = 0; kb < nst && kb < kblocks; ++kb) {
        mbar_expect_tx(&full_bar[kb], 2 * kABytes);
        tma_load_4d(sA + (size_t)kb * kABytes, &p.amap[p.tap_map[0]], &full_bar[kb], kb * 64, ax, ay, img);
        tma_load_2d(sB + (size_t)kb * kABytes, &p.bmap, &full_bar[kb], kb * 64, n0);
      }
    }
    __syncwarp();
    int s = 0;
    uint32_t ph = 0;
    for (int kb = 0; kb < kblocks; ++kb) {
      mbar_wait(&full_bar[s], ph);
      tc_fence_after();
      if (elect_one()) {
        const uint64_t adesc = make_sdesc(sA0 + (uint32_t)s * kABytes);
        const uint64_t bdesc = make_sdesc(sB0 + (uint32_t)s * kABytes);
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_f16(tmem_base, adesc + (uint64_t)(k * 2), bdesc + (uint64_t)(k * 2), idesc, (kb | k) ? 1u : 0u);
        umma_commit(&empty_bar[s]);
      }
      __syncwarp();
      if (kb + nst < kblocks) {                                // refill this stage with k-block kb + nst once its MMAs retired
        mbar_wait(&empty_bar[s], ph);
        if (elect_one()) {
          mbar_expect_tx(&full_bar[s], 2 * kABytes);
          tma_load_4d(sA + (size_t)s * kABytes, &p.amap[p.tap_map[0]], &full_bar[s], (kb + nst) * 64, ax, ay, img);
          tma_load_2d(sB + (size_t)s * kABytes, &p.bmap, &full_bar[s], (kb + nst) * 64, n0);
        }
        __syncwarp();
      }
      if (++s == nst) { s = 0; ph ^= 1; }
    }
    if (elect_one()) umma_commit(tfull_bar);
    __syncwarp();
  } else {
    // ---------------- epilogue: warps 1..4 <-> TMEM lane quadrants (warp & 3)
    const int lane_grp = warp & 3;
    const int row = lane_grp * 32 + lane;
    const uint32_t stage_a = smem_u32(s_stage);
    if (p.res_tma) mbar_wait(rfull_bar, 0);
    mbar_wait(tfull_bar, 0);
    tc_fence_after();
    const uint32_t t_base = tmem_base + ((uint32_t)(lane_grp * 32) << 16);
#pragma unroll 1
    for (int c = 0; c < kSmallN / 32; ++c) {
      uint32_t v[32];
      tmem_ld32(t_base + (uint32_t)(c * 32), v);
      const uint32_t srow = stage_a + (uint32_t)(c >> 1) * 16384u + (uint32_t)row * 128u;
      uint4 rc[4];
      if (p.res_tma) {
#pragma unroll
        for (int j = 0; j < 4; ++j) rc[j] = lds128(srow + (uint32_t)((((c & 1) * 4 + j) ^ (row & 7)) * 16));
      }
      tmem_ld_wait();
      float f[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) f[j] = __uint_as_float(v[j]);
      if (p.bias) {
        const float4* b4 = reinterpret_cast<const float4*>(p.bias + n0 + c * 32);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 b = __ldg(b4 + j);
          fadd2(f[4 * j], f[4 * j + 1], b.x, b.y);
          fadd2(f[4 * j + 2], f[4 * j + 3], b.z, b.w);
        }
      }
      if (p.res_tma) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const __half2* hh = reinterpret_cast<const __half2*>(&rc[j]);
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const float2 a = __half22float2(hh[e]);
            fadd2(f[j * 8 + 2 * e], f[j * 8 + 2 * e + 1], a.x, a.y);
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint4 o;
        uint32_t* ho = reinterpret_cast<uint32_t*>(&o);
        if (p.relu) {
#pragma unroll
          for (int e = 0; e < 4; ++e) ho[e] = pack_f16x2_relu(f[j * 8 + 2 * e], f[j * 8 + 2 * e + 1]);
        } else {
#pragma unroll
          for (int e = 0; e < 4; ++e) ho[e] = pack_f16x2(f[j * 8 + 2 * e], f[j * 8 + 2 * e + 1]);
        }
        sts128(srow + (uint32_t)((((c & 1) * 4 + j) ^ (row & 7)) * 16), o);
      }
    }
    fence_async_smem();                                        // generic-proxy writes -> visible to the TMA store
    asm volatile("bar.sync 1, 128;" ::: "memory");
    if (warp == 1 && elect_one()) {
      tma_store_4d(&p.omap[0], s_stage, n0, x0, y0, img);
      tma_store_4d(&p.omap[0], s_stage + 16384, n0 + 64, x0, y0, img);
      bulk_commit();
      bulk_wait_read<0>();                                     // the staging tile must outlive the stores' read-out
    }
    __syncwarp();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)kSmallN);
  }
}

// ------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

static int encode_map(CUtensorMap* m, void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                      const uint32_t* box) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return SMB_ECUDA; }
  cuuint64_t d[5]; cuuint64_t s[4]; cuuint32_t b[5]; cuuint32_t es[5];
  for (int i = 0; i < rank; ++i) { d[i] = dims[i]; b[i] = box[i]; es[i] = 1; }
  for (int i = 0; i < rank - 1; ++i) s[i] = strides_bytes[i];
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, (cuuint32_t)rank, base, d, s, b, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): rank=%d dims=[%llu,%llu,%llu,%llu] strides=[%llu,%llu,%llu] box=[%u,%u,%u,%u]",
              (int)r, rank, (unsigned long long)d[0], (unsigned long long)d[1], (unsigned long long)(rank > 2 ? d[2] : 0),
              (unsigned long long)(rank > 3 ? d[3] : 0), (unsigned long long)s[0], (unsigned long long)(rank > 2 ? s[1] : 0),
              (unsigned long long)(rank > 3 ? s[2] : 0), b[0], b[1], rank > 2 ? b[2] : 0, rank > 3 ? b[3] : 0);
    return SMB_ECUDA;
  }
  return SMB_OK;
}

}  // namespace smb

using namespace smb;

struct smb_conv_plan {
  ConvParams p;
  int grid;
  size_t smem_bytes;
  int has_bias, has_residual, gn_stats;
  int omap_ok;                    // output tensor maps encoded (fp16 output, Cout % 64 == 0)
  int rmap_ok;                    // residual tensor maps encoded (same-shape fp16 residual)
  const void* rmap_ptr;           // single-level plans: residual pointer rmap[0] is currently encoded for (lazy, smb_conv_run)
  int small;                      // 1: conv1x1_small_kernel (one 128 x 128 tile per CTA), else the persistent conv_gemm_kernel
};

static int g_min_tiles = 48;
extern "C" int smb_conv_set_min_tiles(int min_tiles) {
  const int prev = g_min_tiles;
  g_min_tiles = min_tiles > 0 ? min_tiles : 48;
  return prev;
}

static int g_num_sms = 0;
static int num_sms() {
  if (!g_num_sms) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
  }
  return g_num_sms;
}

// choose the BH x BW = 128 patch with the fewest tiles (ties -> wider rows, better store coalescing)
static void choose_patch(int H, int W, int* BH, int* BW) {
  const int cand[5][2] = {{1, 128}, {2, 64}, {4, 32}, {8, 16}, {16, 8}};
  long best = -1;
  for (int i = 0; i < 5; ++i) {
    const long t = (long)cdiv(H, cand[i][0]) * cdiv(W, cand[i][1]);
    if (best < 0 || t < best) { best = t; *BH = cand[i][0]; *BW = cand[i][1]; }
  }
}

static int finish_plan(smb_conv_plan* pl, int Cout, int Ktotal, const void* weight) {
  ConvParams& p = pl->p;
  pl->small = 0;
  {
    // short-K 1x1 convolutions (K <= 256, fp16 TMA-storable output, no GroupNorm statistics, same-shape residual or none):
    // one tile per CTA, several CTAs per SM (conv1x1_small_kernel)
    // Measured (profiles/r02_conv_times_small1x1_*.txt): not faster than the persistent kernel - layer1.conv3 19.7 us with
    // either - so it is OFF by default (SMB_CONV_SMALL=1 selects it; tests/test_gpu_conv.py keeps it validated).
    const char* envs = getenv("SMB_CONV_SMALL");
    const int want = envs ? atoi(envs) : 0;
    const int kb = Ktotal / 64;
    if (want && p.num_levels == 1 && p.num_taps == 1 && kb >= 1 && kb <= 4 && Cout % kSmallN == 0 && pl->omap_ok && !p.out_f32 &&
        p.gn_group == 0 && (p.res_mode == 0 || (p.res_mode == 1 && pl->rmap_ok)) && !getenv("SMB_CONV_DEBUG")) {
      pl->small = 1;
      p.n_tile = kSmallN;
      p.n_tiles_n = Cout / kSmallN;
      p.num_acc = 1;
      p.tmem_cols = kSmallN;
      p.pair = 0;
      p.cluster = 1;
      p.debug_mode = 0;
      p.out_tma = 1;
      p.res_tma = (p.res_mode == 1) ? 1 : 0;
      p.stage_slots = 2;
      p.store_lag = 1;
      p.stages = kb < 2 ? kb : 2;
      pl->smem_bytes = (size_t)p.stages * 2 * kABytes + 2 * 16384 + 256 + 1024;
      uint64_t dims[2] = {(uint64_t)Ktotal, (uint64_t)Cout};
      uint64_t strides[1] = {(uint64_t)Ktotal * 2};
      uint32_t box[2] = {64, (uint32_t)kSmallN};
      const int rc = encode_map(&p.bmap, const_cast<void*>(weight), 2, dims, strides, box);
      if (rc) return rc;
      pl->grid = p.tiles_m * p.n_tiles_n;
      return SMB_OK;
    }
  }
  // N tile: the largest of {Cout (<=256, rounded to 16) | 256, 128, 64} that still yields >= ~one wave of tiles.
  // Small feature maps (few M tiles) are latency-bound per tile, so they are split along N to occupy more SMs.
  int cand[3], nc = 0;
  if (Cout <= 256) cand[nc++] = (Cout + 15) / 16 * 16;
  else if (Cout % 256 == 0) cand[nc++] = 256;
  if (Cout > 128 && Cout % 128 == 0) cand[nc++] = 128;
  if (Cout > 64 && Cout % 64 == 0) cand[nc++] = 64;
  if (nc == 0) { set_error("conv plan: unsupported Cout=%d", Cout); return SMB_EINVAL; }
  int n_tile = cand[nc - 1];
  const char* envt = getenv("SMB_CONV_MIN_TILES");
  const long min_tiles = envt ? atol(envt) : g_min_tiles;
  for (int i = 0; i < nc; ++i)
    if ((long)p.tiles_m * cdiv(Cout, cand[i]) >= min_tiles) { n_tile = cand[i]; break; }
  p.n_tile = n_tile;
  p.n_tiles_n = cdiv(Cout, n_tile);
  p.num_acc = (2 * n_tile <= 512) ? 2 : 1;
  int tc = 32;
  while (tc < p.num_acc * n_tile) tc <<= 1;
  p.tmem_cols = tc;
  // pair mode (tcgen05 cta_group::2): two SMs compute one 256-row x n_tile tile and each ingests only half of the
  // weight tile - the L2 -> SM ingress (the bound for these K-major 128-row tiles) drops from 16K+n*128 to 16K+n*64
  // bytes per k-block per SM.
  const char* envp = getenv("SMB_CONV_PAIR");
  const int want_pair = envp ? atoi(envp) : 1;
  p.pair = (want_pair && p.tiles_m >= 2 && n_tile % 32 == 0 && n_tile >= 32) ? 1 : 0;
  const char* envd = getenv("SMB_CONV_DEBUG");
  p.debug_mode = envd ? atoi(envd) : 0;
  if (p.debug_mode & 3) p.pair = 0;
  const size_t stage = (size_t)kABytes + (size_t)(p.pair ? n_tile / 2 : n_tile) * 128;
  p.out_tma = (pl->omap_ok && !p.out_f32 && n_tile % 64 == 0 && !getenv("SMB_CONV_NO_TMA_STORE")) ? 1 : 0;
  p.res_tma = (p.out_tma && p.res_mode == 1 && pl->rmap_ok && !getenv("SMB_CONV_NO_TMA_RES")) ? 1 : 0;
  size_t stage_out = p.out_tma ? (size_t)(n_tile / 64) * 16384 : 0;      // result / residual staging tiles
  // Staging ring of the TMA-store epilogue: one tile's worth of 64-channel chunks, or two when shared memory allows it
  // without starving the operand pipeline (short-K tiles - the bottleneck output / shortcut 1x1 convs - are epilogue-bound:
  // with two tiles of slots the residual of the next tile lands and the stores of the previous tile drain meanwhile).
  p.stage_slots = n_tile / 64;
  p.store_lag = 1;
  {
    const int kblocks = Ktotal / 64;
    const char* envs = getenv("SMB_CONV_STAGE_SETS");
    const int want2 = envs ? atoi(envs) == 2 : 1;
    const int st2 = (int)((194 * 1024 - 2 * (long)stage_out) / (long)stage);
    // operand stages that must remain: min(kblocks, 3), and never fewer than the two the pipeline needs (a one-k-block
    // tile of 256 channels without pair mode would otherwise be left with a single stage and no plan)
    const int min_st = kblocks < 2 ? 2 : (kblocks < 3 ? kblocks : 3);
    if (p.out_tma && want2 && 2 * stage_out <= 128 * 1024 && st2 >= min_st) {
      p.stage_slots *= 2;
      stage_out *= 2;
    }
  }
  {
    const char* envl = getenv("SMB_CONV_STORE_LAG");
    int lag = envl ? atoi(envl) : 1;
    if (lag < 1) lag = 1;
    if (lag > 4) lag = 4;
    if (lag > p.stage_slots - 1) lag = p.stage_slots > 1 ? p.stage_slots - 1 : 1;
    p.store_lag = lag;
  }
  {
    // split-group epilogue (epilogue_split): TMA-store plans without GroupNorm statistics whose residual, if any, is
    // TMA-staged; bias and alpha == 1 are checked at run time.  SMB_CONV_EPI_SPLIT=0 keeps the lockstep epilogue.
    const char* enve = getenv("SMB_CONV_EPI_SPLIT");
    const int want = enve ? atoi(enve) : 1;
    p.epi_split = (want && p.out_tma && p.gn_group == 0 && (p.res_mode == 0 || p.res_tma) && Cout % n_tile == 0 &&
                   p.stage_slots >= 2 && p.stage_slots >= n_tile / 64 && !(p.debug_mode & ~8)) ? 1 : 0;
  }
  const size_t budget = 194 * 1024 - stage_out;
  int stages = (int)(budget / stage);
  if (stages > 8) stages = 8;
  if (stages < 2) { set_error("conv plan: tile too large for shared memory"); return SMB_EINVAL; }
  p.stages = stages;
  pl->smem_bytes = stages * stage + 4096 + stage_out + 1024;    // + barriers/bias (4 KB) + staging + align
  // weights: [Cout, Ktotal] K-major
  uint64_t dims[2] = {(uint64_t)Ktotal, (uint64_t)Cout};
  uint64_t strides[1] = {(uint64_t)Ktotal * 2};
  // cluster size: pair mode is a 2-CTA cluster; otherwise optionally multicast the weight tile (SMB_CONV_CLUSTER)
  int cluster = 1;
  if (p.pair) {
    cluster = 2;
  } else {
    const char* env = getenv("SMB_CONV_CLUSTER");
    const int want = env ? atoi(env) : 1;
    if ((want == 2 || want == 4) && p.tiles_m >= num_sms() && (n_tile / want) % 8 == 0) cluster = want;
  }
  p.cluster = cluster;
  uint32_t box[2] = {64, (uint32_t)(n_tile / cluster)};
  int rc = encode_map(&p.bmap, const_cast<void*>(weight), 2, dims, strides, box);
  if (rc) return rc;
  const int units = cdiv(p.tiles_m, cluster) * p.n_tiles_n;
  const char* envc = getenv("SMB_CONV_MAX_CTAS");            // experiments: leave SMs free for a concurrent stream
  int sm_cap = num_sms();
  if (envc && atoi(envc) > 0 && atoi(envc) < sm_cap) sm_cap = atoi(envc);
  const int max_clusters = (cluster == 4 && sm_cap > 132 ? 132 : sm_cap) / cluster;
  const int clusters = units < max_clusters ? units : max_clusters;
  pl->grid = clusters * cluster;
  return SMB_OK;
}

extern "C" int smb_conv_plan_create_multi(const smb_conv_desc_t* d, int num_levels, const smb_conv_level_t* levels,
                                          const void* weight, smb_conv_plan_t** plan_out) {
  SMB_CHECK_ARG(d && levels && weight && plan_out, "smb_conv_plan_create: null pointer");
  SMB_CHECK_ARG(num_levels >= 1 && num_levels <= kMaxLevels, "smb_conv_plan_create: num_levels=%d outside [1,%d]", num_levels, kMaxLevels);
  SMB_CHECK_ARG(d->Cin % 64 == 0 && d->Cin > 0, "smb_conv_plan_create: Cin=%d must be a multiple of 64", d->Cin);
  SMB_CHECK_ARG(d->Cout % 16 == 0 && d->Cout > 0, "smb_conv_plan_create: Cout=%d must be a multiple of 16", d->Cout);
  SMB_CHECK_ARG((d->kh == 1 && d->kw == 1 && d->pad == 0) || (d->kh == 3 && d->kw == 3 && d->pad == 1),
                "smb_conv_plan_create: only 1x1/p0 and 3x3/p1 kernels (got %dx%d pad %d)", d->kh, d->kw, d->pad);
  SMB_CHECK_ARG(d->stride == 1 || d->stride == 2, "smb_conv_plan_create: stride %d", d->stride);
  SMB_CHECK_ARG(d->stride == 1 || num_levels == 1, "smb_conv_plan_create: strided convolutions are single-level");
  const int in_pitch = d->in_pitch ? d->in_pitch : d->Cin;
  const int out_pitch = d->out_pitch ? d->out_pitch : d->Cout;
  SMB_CHECK_ARG(in_pitch % 8 == 0 && out_pitch % 4 == 0, "smb_conv_plan_create: bad pitches");
  SMB_CHECK_ARG(((uintptr_t)weight % 16) == 0, "smb_conv_plan_create: weight must be 16-byte aligned");
  smb_conv_plan* pl = new smb_conv_plan();
  memset(&pl->p, 0, sizeof(ConvParams));
  pl->omap_ok = 0;
  pl->rmap_ok = 0;
  pl->rmap_ptr = nullptr;
  ConvParams& p = pl->p;
  const int k = d->kh, s = d->stride;
  p.n_img = d->N;
  p.num_levels = num_levels;
  p.num_taps = k * k; p.kb_per_tap = d->Cin / 64;
  p.Cout = d->Cout;
  p.out_pitch = out_pitch; p.out_f32 = (d->out_dtype == SMB_F32);
  p.alpha = 1.0f; p.relu = d->relu;
  p.res_mode = d->has_residual ? (d->residual_upsample ? 2 : 1) : 0;
  p.res_pitch = d->Cout;
  p.gn_group = d->gn_stats ? d->Cout / 32 : 0;
  pl->has_bias = d->has_bias; pl->has_residual = d->has_residual; pl->gn_stats = d->gn_stats;
  if (d->gn_stats && !(p.gn_group == 8 || p.gn_group == 16)) {
    set_error("smb_conv_plan_create: gn_stats needs Cout/32 in {8,16}");
    delete pl;
    return SMB_EINVAL;
  }
  const uint64_t px = (uint64_t)in_pitch * 2;       // bytes per pixel
  int rc = SMB_OK;
  int tile_start = 0;
  for (int l = 0; l < num_levels && rc == SMB_OK; ++l) {
    const smb_conv_level_t& lv = levels[l];
    LevelDesc& L = p.lv[l];
    const int H = lv.H, W = lv.W;
    if (!lv.in || !lv.out || H <= 0 || W <= 0 || ((uintptr_t)lv.in % 16) || ((uintptr_t)lv.out % 16) ||
        (d->has_residual && !lv.residual) || (d->gn_stats && !lv.gn_stats)) {
      set_error("smb_conv_plan_create: level %d has a null / misaligned pointer or empty shape", l);
      rc = SMB_EINVAL;
      break;
    }
    const int Ho = (H + 2 * d->pad - k) / s + 1, Wo = (W + 2 * d->pad - k) / s + 1;
    L.H_out = Ho; L.W_out = Wo;
    choose_patch(Ho, Wo, &L.BH, &L.BW);
    L.tiles_x = cdiv(Wo, L.BW); L.tiles_y = cdiv(Ho, L.BH);
    L.tile_start = tile_start;
    tile_start += d->N * L.tiles_x * L.tiles_y;
    L.out = lv.out; L.residual = (const __half*)lv.residual; L.gn_stats = (long long*)lv.gn_stats;
    L.res_h = lv.res_h; L.res_w = lv.res_w;
    const uint32_t box[4] = {64, (uint32_t)L.BW, (uint32_t)L.BH, 1};
    if (rc == SMB_OK && d->out_dtype == SMB_F16 && d->Cout % 64 == 0 && out_pitch % 8 == 0) {
      uint64_t odims[4] = {(uint64_t)d->Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)d->N};
      const uint64_t opx = (uint64_t)out_pitch * 2;
      uint64_t ostr[3] = {opx, opx * Wo, opx * Wo * Ho};
      rc = encode_map(&p.omap[l], lv.out, 4, odims, ostr, box);
      pl->omap_ok = (rc == SMB_OK);
      if (rc != SMB_OK) break;
      if (d->has_residual && !d->residual_upsample && num_levels == 1) pl->rmap_ok = 1;   // encoded lazily in smb_conv_run
      if (d->has_residual && !d->residual_upsample && num_levels > 1) {
        // multi-level plans bake the residual pointer, so its map can be encoded here
        uint64_t rstr[3] = {(uint64_t)d->Cout * 2, (uint64_t)d->Cout * 2 * Wo, (uint64_t)d->Cout * 2 * Wo * Ho};
        rc = encode_map(&p.rmap[l], const_cast<void*>(lv.residual), 4, odims, rstr, box);
        pl->rmap_ok = (rc == SMB_OK);
        if (rc != SMB_OK) break;
      }
    }
    if (s == 1) {
      L.map0 = l;
      uint64_t dims[4] = {(uint64_t)d->Cin, (uint64_t)W, (uint64_t)H, (uint64_t)d->N};
      uint64_t strides[3] = {px, px * W, px * W * H};
      rc = encode_map(&p.amap[l], const_cast<void*>(lv.in), 4, dims, strides, box);
    } else {
      // stride 2: input (2*oy + r - pad, 2*ox + c - pad) -> parity-split views with doubled strides
      L.map0 = 0;
      for (int py = 0; py < 2 && rc == SMB_OK; ++py)
        for (int pxp = 0; pxp < 2 && rc == SMB_OK; ++pxp) {
          const int hp = (H - py + 1) / 2, wp = (W - pxp + 1) / 2;   // rows / cols of this parity
          uint64_t dims[4] = {(uint64_t)d->Cin, (uint64_t)(wp > 0 ? wp : 1), (uint64_t)(hp > 0 ? hp : 1), (uint64_t)d->N};
          uint64_t strides[3] = {px * 2, px * W * 2, px * W * H};
          const char* base = (const char*)lv.in + ((size_t)py * W + pxp) * px;
          rc = encode_map(&p.amap[py * 2 + pxp], const_cast<char*>(base), 4, dims, strides, box);
        }
    }
  }
  if (rc == SMB_OK) {
    p.tiles_m = tile_start;
    for (int i = (s == 1 ? num_levels : 4); i < kMaxMaps; ++i) p.amap[i] = p.amap[0];
    for (int r = 0; r < k; ++r)
      for (int c = 0; c < k; ++c) {
        const int t = r * k + c;
        if (s == 1) {
          p.tap_map[t] = 0; p.tap_dx[t] = c - d->pad; p.tap_dy[t] = r - d->pad;
        } else {
          const int oy = r - d->pad, ox = c - d->pad;            // input offset relative to 2*o
          const int py = ((oy % 2) + 2) % 2, pxp = ((ox % 2) + 2) % 2;
          p.tap_map[t] = py * 2 + pxp;
          p.tap_dy[t] = (oy - py) / 2;                           // exact: oy - py is even
          p.tap_dx[t] = (ox - pxp) / 2;
        }
      }
    rc = finish_plan(pl, d->Cout, k * k * d->Cin, weight);
  }
  if (rc != SMB_OK) { delete pl; return rc; }
  *plan_out = pl;
  return SMB_OK;
}

extern "C" int smb_conv_plan_create(const smb_conv_desc_t* d, const void* in, const void* weight, void* out,
                                    smb_conv_plan_t** plan_out) {
  SMB_CHECK_ARG(d, "smb_conv_plan_create: null desc");
  // single tensor; residual / gn_stats pointers are supplied at run time (placeholders keep the level non-null)
  smb_conv_level_t lv;
  lv.in = in; lv.out = out;
  lv.residual = d->has_residual ? out : nullptr;
  lv.gn_stats = d->gn_stats ? out : nullptr;
  lv.H = d->H; lv.W = d->W; lv.res_h = d->res_h; lv.res_w = d->res_w;
  return smb_conv_plan_create_multi(d, 1, &lv, weight, plan_out);
}

// 7x7/2 stem on the padded NHWC8 image written by smb_image_to_nhwc8:
//   img8 [N, H+6, W+8, 8] fp16 (pixel (y,x) stored at (y+3, x+3)); K = 7 filter rows x (8 pixels x 8 ch).
//   Output pixel (oy,ox), filter row r reads padded row 2*oy + r, pixels 2*ox .. 2*ox+7 (128 contiguous bytes).
extern "C" int smb_stem_plan_create(int N, int H, int W, const void* img_nhwc8, const void* weight448, void* out,
                                    smb_conv_plan_t** plan_out) {
  SMB_CHECK_ARG(img_nhwc8 && weight448 && out && plan_out, "smb_stem_plan_create: null pointer");
  SMB_CHECK_ARG(H % 2 == 0 && W % 2 == 0, "smb_stem_plan_create: H, W must be even (images are padded to /32)");
  smb_conv_plan* pl = new smb_conv_plan();
  memset(&pl->p, 0, sizeof(ConvParams));
  pl->omap_ok = 0;
  pl->rmap_ok = 0;
  pl->rmap_ptr = nullptr;
  ConvParams& p = pl->p;
  LevelDesc& L = p.lv[0];
  const int Ho = H / 2, Wo = W / 2, Hp = H + 6, Wp = W + 8;
  p.n_img = N; p.num_levels = 1;
  L.H_out = Ho; L.W_out = Wo;
  choose_patch(Ho, Wo, &L.BH, &L.BW);
  L.tiles_x = cdiv(Wo, L.BW); L.tiles_y = cdiv(Ho, L.BH);
  L.tile_start = 0; L.map0 = 0; L.out = out;
  p.tiles_m = N * L.tiles_x * L.tiles_y;
  p.num_taps = 7; p.kb_per_tap = 1;
  p.Cout = 64;
  p.out_pitch = 64; p.out_f32 = 0; p.alpha = 1.f; p.relu = 1;
  p.gn_group = 0;
  pl->has_bias = 1;
  const uint64_t rowb = (uint64_t)Wp * 16;
  const uint32_t box[4] = {64, (uint32_t)L.BW, (uint32_t)L.BH, 1};
  int rc = SMB_OK;
  for (int par = 0; par < 2 && rc == SMB_OK; ++par) {
    const int rows = (Hp - par + 1) / 2;
    uint64_t dims[4] = {64, (uint64_t)Wo, (uint64_t)rows, (uint64_t)N};
    uint64_t strides[3] = {32, rowb * 2, rowb * Hp};     // 2-pixel step along x: overlapping 8-pixel windows
    rc = encode_map(&p.amap[par], (char*)const_cast<void*>(img_nhwc8) + par * rowb, 4, dims, strides, box);
  }
  for (int i = 2; i < kMaxMaps; ++i) p.amap[i] = p.amap[i & 1];
  if (rc == SMB_OK) {
    uint64_t odims[4] = {64, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
    uint64_t ostr[3] = {128, (uint64_t)128 * Wo, (uint64_t)128 * Wo * Ho};
    rc = encode_map(&p.omap[0], out, 4, odims, ostr, box);
    pl->omap_ok = (rc == SMB_OK);
  }
  for (int r = 0; r < 7; ++r) { p.tap_map[r] = r & 1; p.tap_dy[r] = r >> 1; p.tap_dx[r] = 0; }
  if (rc == SMB_OK) rc = finish_plan(pl, 64, 448, weight448);
  if (rc != SMB_OK) { delete pl; return rc; }
  *plan_out = pl;
  return SMB_OK;
}

// 7x7/2 stem on the SPACE-TO-DEPTH image written by smb_image_to_s2d16 / smb_preprocess_u8_s2d:
//   q [N, H/2+3, W/2+4, 16] fp16, q(Y, X, (dy*2+dx)*4 + c) = padded pixel (2Y+dy, 2X+dx) channel c.
//   out(oy, ox) = sum_{a,b<4} sum_{dy,dx,c} w[2a+dy][2b+dx][c] * q(oy+a, ox+b, (dy,dx,c)) : a 4x4 stride-1 convolution
//   over 16 channels, K = 4 filter rows x (4 cells x 16 ch = 128 contiguous bytes) = 256 instead of the 448 of the
//   pixel-window form (7 rows x 8 pixels x 8 ch) - 43 % fewer operand bytes and MMAs for the L2->SM-bound N = 64 stem.
extern "C" int smb_stem_plan_create_s2d(int N, int H, int W, const void* img_s2d16, const void* weight256, void* out,
                                        smb_conv_plan_t** plan_out) {
  SMB_CHECK_ARG(img_s2d16 && weight256 && out && plan_out, "smb_stem_plan_create_s2d: null pointer");
  SMB_CHECK_ARG(H % 2 == 0 && W % 2 == 0, "smb_stem_plan_create_s2d: H, W must be even (images are padded to /32)");
  smb_conv_plan* pl = new smb_conv_plan();
  memset(&pl->p, 0, sizeof(ConvParams));
  pl->omap_ok = 0;
  pl->rmap_ok = 0;
  pl->rmap_ptr = nullptr;
  ConvParams& p = pl->p;
  LevelDesc& L = p.lv[0];
  const int Ho = H / 2, Wo = W / 2, Hq = H / 2 + 3, Wq = W / 2 + 4;
  p.n_img = N; p.num_levels = 1;
  L.H_out = Ho; L.W_out = Wo;
  choose_patch(Ho, Wo, &L.BH, &L.BW);
  L.tiles_x = cdiv(Wo, L.BW); L.tiles_y = cdiv(Ho, L.BH);
  L.tile_start = 0; L.map0 = 0; L.out = out;
  p.tiles_m = N * L.tiles_x * L.tiles_y;
  p.num_taps = 4; p.kb_per_tap = 1;
  p.Cout = 64;
  p.out_pitch = 64; p.out_f32 = 0; p.alpha = 1.f; p.relu = 1;
  p.gn_group = 0;
  pl->has_bias = 1;
  const uint64_t rowb = (uint64_t)Wq * 32;
  const uint32_t box[4] = {64, (uint32_t)L.BW, (uint32_t)L.BH, 1};
  uint64_t dims[4] = {64, (uint64_t)Wo, (uint64_t)Hq, (uint64_t)N};
  uint64_t strides[3] = {32, rowb, rowb * Hq};          // 1-cell step along x: overlapping 4-cell (128-byte) windows
  int rc = encode_map(&p.amap[0], const_cast<void*>(img_s2d16), 4, dims, strides, box);
  for (int i = 1; i < kMaxMaps; ++i) p.amap[i] = p.amap[0];
  if (rc == SMB_OK) {
    uint64_t odims[4] = {64, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)N};
    uint64_t ostr[3] = {128, (uint64_t)128 * Wo, (uint64_t)128 * Wo * Ho};
    rc = encode_map(&p.omap[0], out, 4, odims, ostr, box);
    pl->omap_ok = (rc == SMB_OK);
  }
  for (int a = 0; a < 4; ++a) { p.tap_map[a] = 0; p.tap_dy[a] = a; p.tap_dx[a] = 0; }
  if (rc == SMB_OK) rc = finish_plan(pl, 64, 256, weight256);
  if (rc != SMB_OK) { delete pl; return rc; }
  *plan_out = pl;
  return SMB_OK;
}

extern "C" void smb_conv_plan_destroy(smb_conv_plan_t* plan) { delete plan; }

// Cap the persistent grid (e.g. to half the SMs) so that two independent convolutions captured on different streams
// can run side by side and fill each other's partial waves.
extern "C" int smb_conv_plan_set_max_ctas(smb_conv_plan_t* plan, int max_ctas) {
  SMB_CHECK_ARG(plan && max_ctas >= 1, "smb_conv_plan_set_max_ctas: bad argument");
  if (plan->small) return SMB_OK;                   // one tile per CTA: the grid is the tile count
  const int c = plan->p.cluster;
  int g = (max_ctas / c) * c;
  if (g < c) g = c;
  if (g < plan->grid) plan->grid = g;
  return SMB_OK;
}

extern "C" int smb_conv_plan_info(const smb_conv_plan_t* plan, int* out, int n) {
  SMB_CHECK_ARG(plan && out && n >= 0, "smb_conv_plan_info: bad argument");
  const ConvParams& p = plan->p;
  const int v[] = {p.n_tile, p.n_tiles_n, p.tiles_m, p.pair, p.cluster, plan->grid, p.out_tma, p.res_tma, p.stage_slots,
                   p.epi_split, plan->small};
  const int nv = (int)(sizeof(v) / sizeof(v[0]));
  for (int i = 0; i < n && i < nv; ++i) out[i] = v[i];
  return nv;
}

extern "C" int smb_conv_run(const smb_conv_plan_t* plan, const float* bias, const void* residual, void* gn_stats,
                            float alpha, smb_stream_t stream) {
  SMB_CHECK_ARG(plan, "smb_conv_run: null plan");
  SMB_CHECK_ARG(!plan->has_bias || bias, "smb_conv_run: plan expects a bias");
  ConvParams p = plan->p;
  p.bias = plan->has_bias ? bias : nullptr;
  // single-level plans take residual / statistics pointers at run time; multi-level plans bake them per level
  if (p.num_levels == 1) {
    if (plan->has_residual) {
      SMB_CHECK_ARG(residual, "smb_conv_run: plan expects a residual");
      p.lv[0].residual = (const __half*)residual;
      if (p.res_tma) {
        smb_conv_plan* mp = const_cast<smb_conv_plan*>(plan);       // descriptor cache keyed by the residual pointer
        if (mp->rmap_ptr != residual) {
          const LevelDesc& L0 = p.lv[0];
          uint64_t rdims[4] = {(uint64_t)p.Cout, (uint64_t)L0.W_out, (uint64_t)L0.H_out, (uint64_t)p.n_img};
          uint64_t rstr[3] = {(uint64_t)p.Cout * 2, (uint64_t)p.Cout * 2 * L0.W_out, (uint64_t)p.Cout * 2 * L0.W_out * L0.H_out};
          uint32_t rbox[4] = {64, (uint32_t)L0.BW, (uint32_t)L0.BH, 1};
          const int erc = encode_map(&mp->p.rmap[0], const_cast<void*>(residual), 4, rdims, rstr, rbox);
          if (erc) return erc;
          mp->rmap_ptr = residual;
        }
        p.rmap[0] = mp->p.rmap[0];
      }
    }
    if (plan->gn_stats) {
      SMB_CHECK_ARG(gn_stats, "smb_conv_run: plan expects a gn_stats buffer");
      p.lv[0].gn_stats = (long long*)gn_stats;
    }
  }
  p.alpha = alpha;
  if (!plan->has_bias || alpha != 1.0f || ((uintptr_t)bias & 15)) p.epi_split = 0;   // epilogue_split: float4 bias reads, no scaling
  SMB_CHECK_ARG(!plan->small || alpha == 1.0f, "smb_conv_run: the short-K 1x1 plan does not scale its output (alpha must be 1)");
  {
    const char* ets = getenv("SMB_CONV_TS");      // hex device address of a 16 x int64 buffer (profiling only)
    p.dbg_ts = ets ? (long long*)strtoull(ets, nullptr, 16) : nullptr;
  }
  static DeviceOnce attr_once;
  if (attr_once.first()) {
    SMB_CUDA_OK(cudaFuncSetAttribute(conv_gemm_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    SMB_CUDA_OK(cudaFuncSetAttribute(conv_gemm_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    SMB_CUDA_OK(cudaFuncSetAttribute(conv1x1_small_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024));
  }
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3(plan->grid);
  cfg.blockDim = dim3(plan->small ? kSmallThreads : kThreads);
  cfg.dynamicSmemBytes = plan->smem_bytes;
  cfg.stream = (cudaStream_t)stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = p.cluster;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  static int use_pdl = -1;
  if (use_pdl < 0) { const char* e = getenv("SMB_CONV_PDL"); use_pdl = e ? atoi(e) : 1; }
  if (use_pdl) {
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.numAttrs = 2;
  }
  {
    cudaError_t e = plan->small ? cudaLaunchKernelEx(&cfg, conv1x1_small_kernel, p)
                    : p.pair  ? cudaLaunchKernelEx(&cfg, conv_gemm_kernel<true>, p)
                              : cudaLaunchKernelEx(&cfg, conv_gemm_kernel<false>, p);
    if (e != cudaSuccess) {
      set_error("conv_gemm_kernel launch failed: %s (grid=%d cluster=%d pair=%d smem=%zu n_tile=%d stages=%d tiles_m=%d n_tiles_n=%d)",
                cudaGetErrorString(e), plan->grid, p.cluster, p.pair, plan->smem_bytes, p.n_tile, p.stages, p.tiles_m, p.n_tiles_n);
      cudaGetLastError();
      return SMB_ECUDA;
    }
  }
  SMB_LAUNCH_OK("conv_gemm_kernel");
  return SMB_OK;
}
