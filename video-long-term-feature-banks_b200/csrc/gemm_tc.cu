// tcgen05 (5th-gen tensor core) gathered GEMM for sm_100a.
//
//   D[m,n] = epi( sum_k A[m,k] * B[n,k] ),  fp32 storage, kind::tf32 MMA, fp32 accumulate in TMEM.
//
// Persistent kernel: grid = min(#tiles, #SMs), one CTA per SM walks a static sequence of 128 x BN output
// tiles (UMMA M=128, N=BN, cta_group::1), 544 threads:
//   warps 0-7  PRODUCERS -- the A/B K-chunks (32 fp32 = one 128-byte swizzle row) go straight from NDHWC
//              tensors into the UMMA canonical swizzled shared-memory layouts, never through an im2col
//              buffer: dense operands by TMA tiled boxes (SWIZZLE_128B K-major, SWIZZLE_128B_ATOM_32B
//              MN-major), convolution gathers by TMA im2col copies (conv fwd, unit-stride dgrad, wgrad;
//              one thread issues), and what TMA cannot express (conv1 stem with 16-byte pixels, strided
//              dgrad, unaligned operands) by 16-byte cp.async with zero-fill = padding (all 8 warps);
//   warp 8     TMEM allocator + single-thread tcgen05.mma issuer; tcgen05.commit releases each smem
//              stage back to the producers and hands finished accumulators to the epilogue;
//   warps 9-16 EPILOGUE -- tcgen05.ld TMEM -> registers -> smem transpose -> fused affine / residual /
//              ReLU / TF32 rounding -> coalesced 128-bit global stores (or atomics for split-K).
// The smem ring (full[s]/empty[s] mbarriers) runs continuously across tiles and the accumulator is double
// buffered in TMEM (tmem_full[a]/tmem_empty[a]), so the epilogue of one tile overlaps the loads and MMAs
// of the next.
//
// Operand kinds are described in include/vlfb.h; their element-level definition is
// operand_elem() in common.cuh, which the SIMT engine evaluates literally and the tests
// compare this kernel against.
#include <cuda.h>
#include <stdlib.h>
#include <string.h>

#include <type_traits>

#include "common.cuh"

#ifndef VLFB_EPI_DEPTH
#define VLFB_EPI_DEPTH 2
#endif
namespace vlfb {
namespace tc {

constexpr int BM = 128;        // tile rows (UMMA M)
constexpr int KC = 32;         // fp32 per K chunk (128 B)
constexpr int NPROD = 256;     // 8 producer warps = 2 per scheduler, so the address-generation latency of one warp
                               // hides behind the other (ncu r01: with one producer warp per scheduler 'wait' +
                               // 'selected' stalls dominated).  Measured alternatives (profiles/r01_perf_log.md):
                               // 7 producer warps (16 warps total -> 128 instead of 96 registers, no spills) lose
                               // 3-5% of the step on the gather-bound convs; 4 epilogue warps lose ~4%.
constexpr int NPW = NPROD / 32;
// TMA-only builds: warps whose lane 0 issues the TMA boxes of a K chunk (box b by warp b % NTMAW).  The wgrad chunk is 4
// (dY^T atoms) + 8 (im2col atoms of 32 columns) small boxes and its K loop runs at 33-37 % of the tensor pipe (ncu call M),
// so round 2 tried 2 and 3 issuing warps: parity-green and MUCH slower (call Q: step 16.6 ms instead of 12.7, wgrad 5.7 ms
// instead of 3.1, every other kind slower too) -- the boxes are not limited by the issuing thread but by the TMA unit's
// per-box cost, and concurrent issuers only interleave the boxes of different stages.  Kept as a build parameter with the
// measured default of ONE issuer; the remedy is fewer, larger boxes (one 4-D box per MN-major operand tile, below).
#ifndef VLFB_TMA_WARPS
#define VLFB_TMA_WARPS 1
#endif
constexpr int NTMAW = VLFB_TMA_WARPS;
constexpr int RSTEP = NPROD / 8;   // rows covered by one pass of the K-major loaders
constexpr int NEPI = 256;          // 8 epilogue warps (two per TMEM lane quarter, splitting the column blocks)
constexpr int EPC = 16;            // accumulator columns per epilogue step (tcgen05.ld.32x32b.x16)
constexpr int EPITCH = EPC + 4;    // padded staging row (floats)
constexpr int EPI_COLV = 2 * 128;     // per-warp column scale + bias of its 128 columns (floats)
constexpr int EPI_WARP_FLOATS = 32 * EPITCH + EPI_COLV;
constexpr int EPI_STAGE_BYTES = (NEPI / 32) * EPI_WARP_FLOATS * 4;
constexpr int A_TILE_BYTES = BM * KC * 4;  // 16 KB
constexpr int MAX_STAGES = 8;

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
// Bounded wait: a protocol bug traps (kernel error) instead of hanging the GPU.  The clock is only read
// every 4096 polls so that the spin loop stays 3 instructions long (try_wait suspends in hardware).
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = 0;
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0xFFFu) == 0) {
      const long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 8000000000LL) {
        printf("vlfb gemm_tc: mbarrier timeout (block %d thread %d)\n", blockIdx.x, threadIdx.x);
        __trap();
      }
    }
  }
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool valid) {
  // ignore-src predicate => 16 bytes of zeros (conv padding / tails); one LDGSTS.ZFILL, no size arithmetic
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.eq.u32 p, %2, 0;\n\t"
      "cp.async.cg.shared.global [%0], [%1], 16, p;\n\t}"
      ::"r"(dst), "l"(src), "r"((uint32_t)valid) : "memory");
}
// TMA: one thread arms the stage barrier with the byte count, then issues the bulk tensor copy; the copy
// engine writes the box into shared memory in the SWIZZLE_128B pattern and completes the transaction.
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, int c3, int c4,
                                            uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5, %6}], [%7];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void cp_async_wait_dyn(int n) {
  switch (n) {
    case 0: cp_async_wait<0>(); break;
    case 1: cp_async_wait<1>(); break;
    case 2: cp_async_wait<2>(); break;
    case 3: cp_async_wait<3>(); break;
    case 4: cp_async_wait<4>(); break;
    default: cp_async_wait<5>(); break;
  }
}
__device__ __forceinline__ void fence_proxy_async() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
// ---- cta_group::2 (CTA pair) variants.  Protocol (DESIGN.md 4.1): both CTAs of a (2,1,1) cluster allocate TMEM and
// stage their half of the operands; the barriers that order the pipeline live at the SAME shared-memory offsets in
// both CTAs; the leader (cluster rank 0) issues the MMAs and publishes their completion to both CTAs with a
// multicast commit; the peer's TMA loads and epilogue warps signal the LEADER's barriers (mapa address).
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t mapa_rank(uint32_t saddr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_tf32_2(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of all prior MMAs of the pair -> one arrival on the barrier at this offset in BOTH CTAs
__device__ __forceinline__ void umma_commit2(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(bar), "h"((uint16_t)3) : "memory");
}
// TMA loads issued by either CTA of the pair; the transaction bytes land on `bar`, which may be the peer's barrier
__device__ __forceinline__ void tma_load_3d_2(uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(c2), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void red_add_f4(float* p, const float4& v) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 ld_cg_f4(const float* p) {
  float4 v;
  asm volatile("ld.global.cg.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// residual / accumulate reads: plain (coherent) 128-bit loads -- D may have been written by an earlier launch
// on the same stream, never by this one
__device__ __forceinline__ float4 ld_nc_f4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ uint32_t ld_nc_u16(const unsigned short* p) {
  unsigned short v;
  asm volatile("ld.global.nc.u16 %0, [%1];" : "=h"(v) : "l"(p));
  return (uint32_t)v;
}
__device__ __forceinline__ void prefetch_l2(const void* p) {
  asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// UMMA shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout), SWIZZLE_128B.
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                 uint32_t layout_type = 2) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);                 // [0,14)  start address
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;        // [16,30) leading byte offset
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;        // [32,46) stride byte offset
  d |= (uint64_t)1 << 46;                                  // [46,48) descriptor version 1 (sm_100)
  d |= (uint64_t)layout_type << 61;                        // [61,64) 2 = SWIZZLE_128B, 1 = SWIZZLE_128B_BASE32B
  return d;
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): tf32 x tf32 -> f32, M=128, N=bn.
__host__ __device__ inline uint32_t make_idesc(int bn, int a_mn_major, int b_mn_major, int m = BM) {
  uint32_t d = 0;
  d |= 1u << 4;                          // c_format  = F32
  d |= 2u << 7;                          // a_format  = TF32
  d |= 2u << 10;                         // b_format  = TF32
  d |= (uint32_t)(a_mn_major & 1) << 15; // a_major
  d |= (uint32_t)(b_mn_major & 1) << 16; // b_major
  d |= (uint32_t)(bn >> 3) << 17;        // n_dim
  d |= (uint32_t)(m >> 4) << 24;         // m_dim (128, or 256 = a CTA pair with cta_group::2)
  return d;
}

__host__ __device__ constexpr bool is_mn(int kind) { return kind == VLFB_OP_DENSE_MN || kind == VLFB_OP_CONV_MN || kind == VLFB_OP_STEM_MN; }

// ---------------------------------------------------------------- fast integer division
// q = x / d for 0 <= x < 2^31 with a precomputed multiplier (the gather loaders decode an output
// position per 16-byte copy; 64-bit hardware division there cost more than the copy itself).
struct FastDiv { uint32_t mul, shr, d; };
inline FastDiv make_fastdiv(int d) {
  FastDiv f;
  f.d = (uint32_t)d;
  if (d <= 1) { f.mul = 0; f.shr = 0; return f; }
  int lg = 31 - __builtin_clz((unsigned)d);
  if (d & (d - 1)) ++lg;                       // ceil(log2 d)
  const int p = 31 + lg;
  f.mul = (uint32_t)(((1ull << p) + (uint64_t)d - 1) / (uint64_t)d);
  f.shr = (uint32_t)(p - 32);
  return f;
}
__device__ __forceinline__ void fd_divmod(uint32_t x, const FastDiv& f, uint32_t& q, uint32_t& r) {
  q = (f.d <= 1) ? x : (__umulhi(x, f.mul) >> f.shr);
  r = x - q * f.d;
}
struct PosDiv { FastDiv w, h, t; };
__device__ __forceinline__ Pos4 decode_pos_fast(uint32_t idx, const PosDiv& pd) {
  Pos4 p;
  uint32_t q, r;
  fd_divmod(idx, pd.w, q, r); p.w = (int)r;
  fd_divmod(q, pd.h, q, r); p.h = (int)r;
  fd_divmod(q, pd.t, q, r); p.t = (int)r;
  p.n = (int)q;
  return p;
}

// TMA im2col mode (measured semantics: profiles/r01_im2col_probe.txt): the 5-D map of an NDHWC tensor walks
// `pixelsPerColumn` window origins in W -> H -> D -> N order inside the bounding box [lower, dim-1+upper] with the
// convolution strides as traversal strides; {w,h,d} = origin of the first window (= out*stride - pad), the u16
// offsets select the filter tap (tap*dilation); out-of-range pixels (padding, tensor tail) read as zeros.
__device__ __forceinline__ void tma_load_im2col(uint32_t dst, const CUtensorMap* tm, int c, int w, int h, int d, int n,
                                                int ow, int oh, int od, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%2, %3, %4, %5, %6}], [%7], {%8, %9, %10};"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c), "r"(w), "r"(h), "r"(d), "r"(n), "r"(bar),
        "h"((uint16_t)ow), "h"((uint16_t)oh), "h"((uint16_t)od)
      : "memory");
}

__device__ __forceinline__ void tma_load_im2col_2(uint32_t dst, const CUtensorMap* tm, int c, int w, int h, int d, int n,
                                                  int ow, int oh, int od, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.tensor.5d.im2col.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes "
      "[%0], [%1, {%2, %3, %4, %5, %6}], [%7], {%8, %9, %10};"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tm)), "r"(c), "r"(w), "r"(h), "r"(d), "r"(n), "r"(bar),
        "h"((uint16_t)ow), "h"((uint16_t)oh), "h"((uint16_t)od)
      : "memory");
}

// ---------------------------------------------------------------- K-major loaders
// Tile = `rows` rows x 128 B.  Thread t copies the 16-byte chunk (t & 7) of rows (t >> 3) + RSTEP j.
template <int KIND, int MAXR>
struct KLoader {
  const float* base;
  int64_t ld;
  int nrow;          // rows of this tile handled per thread (rows / RSTEP)
  int kend;          // DENSE_K: K limit for the 16-byte tail predicate
  int row0;
  // per owned row: decoded position (conv kinds) and the swizzled shared-memory offset of its 16-byte chunk
  int s_n[MAXR], s_t[MAXR], s_hw[MAXR];
  uint32_t dst[MAXR];
  uint32_t rowmask;  // DENSE_K: bit j set when row j is inside the matrix
  // Filter-tap cursor.  Chunks are issued in order, so the tap advances incrementally (no division per
  // chunk) and the gathered element offset / validity of every owned row is recomputed only when the
  // tap changes (ncu r01: the per-chunk divisions and 64-bit address math made the producers
  // instruction-bound at ~330 instructions per chunk per warp).
  int cpt, tc, kt, kh, kw;
  int off[MAXR];
  uint32_t okmask;

  __device__ __forceinline__ void init(const vlfb_gemm_params_t& p, const vlfb_operand_t& op, int row0_, int rows,
                                       int limit, int batch, const PosDiv& pdo, const PosDiv& pdi, int kc_first) {
    const int tid = threadIdx.x;
    const int c = tid & 7;
    nrow = rows / RSTEP;
    base = op.ptr;
    ld = op.ld;
    if (KIND == VLFB_OP_STEM_K && ld <= 0) ld = p.g.W;
    kend = p.K;
    rowmask = 0;
    row0 = row0_;
    const vlfb_conv_geom_t& g = p.g;
    if (KIND == VLFB_OP_DENSE_K) base += (int64_t)batch * op.batch_stride;
#pragma unroll
    for (int j = 0; j < MAXR; ++j) {
      if (j >= nrow) break;
      const int r = (tid >> 3) + RSTEP * j;
      const int row = row0 + r;
      const bool ok = row < limit;
      dst[j] = (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4));
      if (KIND == VLFB_OP_DENSE_K) {
        if (ok) rowmask |= 1u << j;
      } else if (KIND == VLFB_OP_CONV_K || KIND == VLFB_OP_STEM_K) {
        Pos4 o = decode_pos_fast(ok ? (uint32_t)row : 0u, pdo);
        s_n[j] = o.n * g.T;
        s_t[j] = ok ? o.t * g.sT - g.pT : -100000;
        s_hw[j] = ((o.h * g.sH - g.pH) << 16) | ((o.w * g.sW - g.pW) & 0xFFFF);
      } else {  // DGRAD_K: rows are input positions
        Pos4 i = decode_pos_fast(ok ? (uint32_t)row : 0u, pdi);
        s_n[j] = i.n * g.To;
        s_t[j] = ok ? i.t + g.pT : -100000;
        s_hw[j] = ((i.h + g.pH) << 16) | ((i.w + g.pW) & 0xFFFF);
      }
    }
    if (KIND == VLFB_OP_CONV_K || KIND == VLFB_OP_DGRAD_K) {
      cpt = (KIND == VLFB_OP_CONV_K ? g.C : g.Co) / KC;
      const int tap = kc_first / cpt;              // one division per tile
      tc = kc_first - tap * cpt;
      decode_tap(tap, g.kH, g.kW, kt, kh, kw);
      compute_tap(g);
    } else if (KIND == VLFB_OP_STEM_K) {
      kt = kc_first / g.kH;
      kh = kc_first - kt * g.kH;
    }
  }

  __device__ __forceinline__ void compute_tap(const vlfb_conv_geom_t& g) {
    okmask = 0;
    const int dt = kt * g.dT, dh = kh * g.dH, dw = kw * g.dW;
#pragma unroll
    for (int j = 0; j < MAXR; ++j) {
      if (j >= nrow) break;
      if (KIND == VLFB_OP_CONV_K) {
        const int ti = s_t[j] + dt, hi = (s_hw[j] >> 16) + dh, wi = (int)(short)(s_hw[j] & 0xFFFF) + dw;
        const bool ok = (unsigned)ti < (unsigned)g.T && (unsigned)hi < (unsigned)g.H && (unsigned)wi < (unsigned)g.W;
        off[j] = ok ? (((s_n[j] + ti) * g.H + hi) * g.W + wi) * g.C : 0;
        if (ok) okmask |= 1u << j;
      } else {  // DGRAD_K
        const int a = s_t[j] - dt, b = (s_hw[j] >> 16) - dh, cc = (int)(short)(s_hw[j] & 0xFFFF) - dw;
        bool ok = a >= 0 && b >= 0 && cc >= 0;
        int to = a, ho = b, wo = cc;
        if (g.sT != 1) { ok = ok && (a % g.sT == 0); to = a / g.sT; }
        if (g.sH != 1) { ok = ok && (b % g.sH == 0); ho = b / g.sH; }
        if (g.sW != 1) { ok = ok && (cc % g.sW == 0); wo = cc / g.sW; }
        ok = ok && to < g.To && ho < g.Ho && wo < g.Wo;
        off[j] = ok ? (((s_n[j] + to) * g.Ho + ho) * g.Wo + wo) * g.Co : 0;
        if (ok) okmask |= 1u << j;
      }
    }
  }

  // Issue the cp.asyncs of the NEXT K chunk (`kc` = its global index, used by DENSE_K only) into `tile`.
  __device__ __forceinline__ void issue(const vlfb_gemm_params_t& p, int kc, uint32_t tile) {
    const int c = threadIdx.x & 7;
    const vlfb_conv_geom_t& g = p.g;
    if (KIND == VLFB_OP_DENSE_K) {
      const int k = kc * KC + c * 4;
      const bool kok = k < kend;
      const int r0 = threadIdx.x >> 3;
#pragma unroll
      for (int j = 0; j < MAXR; ++j) {
        if (j >= nrow) break;
        const bool ok = kok && ((rowmask >> j) & 1u);
        const float* src = ok ? base + (int64_t)(row0 + r0 + RSTEP * j) * ld + k : base;
        cp_async16(tile + dst[j], src, ok);
      }
    } else if (KIND == VLFB_OP_CONV_K || KIND == VLFB_OP_DGRAD_K) {
      const int c0 = tc * KC + c * 4;
#pragma unroll
      for (int j = 0; j < MAXR; ++j) {
        if (j >= nrow) break;
        const bool ok = (okmask >> j) & 1u;
        cp_async16(tile + dst[j], base + (off[j] + c0), ok);
      }
      if (++tc == cpt) {          // next tap
        tc = 0;
        if (++kw == g.kW) { kw = 0; if (++kh == g.kH) { kh = 0; ++kt; } }
        compute_tap(g);
      }
    } else {  // STEM_K: chunk = one (kt,kh) filter row of 8 pixels x 4 channels; this thread's pixel = c
#pragma unroll
      for (int j = 0; j < MAXR; ++j) {
        if (j >= nrow) break;
        const int ti = s_t[j] + kt, hi = (s_hw[j] >> 16) + kh, wi = (int)(short)(s_hw[j] & 0xFFFF) + c;
        const bool ok = (unsigned)ti < (unsigned)g.T && (unsigned)hi < (unsigned)g.H && (unsigned)wi < (unsigned)g.W;
        const int o = ok ? (((s_n[j] + ti) * g.H + hi) * (int)ld + wi) * 4 : 0;      // ld = row pitch in pixels
        cp_async16(tile + dst[j], base + o, ok);
      }
      if (++kh == g.kH) { kh = 0; ++kt; }
    }
  }
};

// ---------------------------------------------------------------- MN-major loaders
// Tile = 32 k-rows, each `rows`*4 bytes of the m (or n) extent, stored as
// [atom of 32 elements][32 k-rows][128 B] (UMMA canonical MN-major SWIZZLE_128B_BASE32B: LBO = 4096 between
// atoms, SBO = 512 between groups of 4 k-rows).
template <int KIND>
struct MNLoader {
  static constexpr int MAXS = (32 * 64) / NPROD;   // copies per thread per chunk at the widest tile (256 cols)
  const float* base;
  int64_t ld;
  int tapz, nslot;
  // A thread copies the SAME 16-byte column chunk c of the k-rows kk0, kk0 + kstep, ... (NPROD is a multiple of
  // the chunks per k-row), so everything that depends on the column -- bounds, filter tap (kh,kw), channel,
  // swizzled shared-memory offset -- is one scalar per tile, and the per-chunk work per copy is two shuffles,
  // a bit test and an add (ncu r01: the previous per-slot arrays cost ~100 instructions per 16-byte copy).
  int mn, kk0, kstep;
  bool colok;
  uint32_t dst0, dstep;
  int slotoff;       // conv kinds: element offset of (kh,kw,ci) relative to the k-row's window origin
  int sh, sw;        // bit positions of this column's kh / kw in the k-row's validity word

  __device__ __forceinline__ void init(const vlfb_gemm_params_t& p, const vlfb_operand_t& op, int row0, int rows,
                                       int limit, int batch, int tap, const FastDiv& cdiv, const FastDiv& kwdiv) {
    const vlfb_conv_geom_t& g = p.g;
    base = op.ptr;
    if (KIND == VLFB_OP_DENSE_MN) base += (int64_t)batch * op.batch_stride;
    ld = op.ld;
    tapz = tap;
    const int cpr = rows >> 2;            // 16-byte chunks per k-row (8, 16, 32 or 64)
    const int lcpr = 31 - __clz(cpr);
    nslot = (KC * cpr) / NPROD;
    kstep = NPROD >> lcpr;
    kk0 = threadIdx.x >> lcpr;
    const int c = threadIdx.x & (cpr - 1);
    mn = row0 + c * 4;
    colok = mn < limit;
    // atom-major tile [atom of 32 elements][32 k-rows][128 B] in the SWIZZLE_128B_BASE32B pattern (32-byte
    // units XOR (k & 3)); plain SWIZZLE_128B returns zeros for tf32 MN-major operands (measured,
    // profiles/r01_gemm_layout_diag.txt).  Same image as a TMA box with SWIZZLE_128B_ATOM_32B.
    // kstep is a multiple of 4 whenever a thread owns more than one copy, so the XOR term is per-thread.
    const int r = kk0 & 3, cc8 = c & 7;
    dst0 = (uint32_t)((c >> 3) * 4096 + kk0 * 128 + ((((cc8 >> 1) ^ r) << 5) | ((cc8 & 1) << 4)));
    dstep = (uint32_t)(kstep * 128);
    slotoff = 0; sh = 0; sw = 8;
    if (KIND == VLFB_OP_CONV_MN) {
      uint32_t tap_hw, cc, qh, qw;
      fd_divmod((uint32_t)(colok ? mn : 0), cdiv, tap_hw, cc);     // n = (kh*kW + kw) * C + ci
      fd_divmod(tap_hw, kwdiv, qh, qw);
      slotoff = ((int)qh * g.dH * g.W + (int)qw * g.dW) * g.C + (int)cc;
      sh = (int)qh; sw = 8 + (int)qw;
    } else if (KIND == VLFB_OP_STEM_MN) {            // n = kh*32 + px*4 (+ch); ld = row pitch in pixels (0 = W)
      if (ld <= 0) ld = g.W;
      const int qh = mn >> 5, qw = (mn & 31) >> 2;
      slotoff = (qh * (int)ld + qw) * 4;
      sh = qh; sw = 8 + qw;
    }
  }

  // k0 = first k of this chunk, kend = exclusive k limit of this CTA's K range.
  // Conv kinds (wgrad B operand): the N extent spans ALL (kh,kw) taps of one kt slice, so one pass over dY
  // feeds up to 256 (tap, ci) columns.  Each lane decodes ONE of the 32 k-rows (output positions) of the
  // chunk into (element offset of its window origin, validity bits per kh and per kw); the copies fetch the
  // row they need with warp shuffles.
  __device__ __forceinline__ void issue(const vlfb_gemm_params_t& p, const PosDiv& pd, int k0, int kend, uint32_t tile) const {
    const vlfb_conv_geom_t& g = p.g;
    int info_a = 0, info_b = 0;
    if (KIND != VLFB_OP_DENSE_MN) {
      const int k = k0 + (threadIdx.x & 31);
      const bool okr = k < kend;
      const Pos4 o = decode_pos_fast(okr ? (uint32_t)k : 0u, pd);
      const int t0 = o.t * g.sT - g.pT + tapz * g.dT;          // z slice = temporal tap
      const bool okt = okr && (unsigned)t0 < (unsigned)g.T;
      const int h0 = o.h * g.sH - g.pH, w0 = o.w * g.sW - g.pW;
      info_a = (((o.n * g.T + t0) * g.H + h0) * (KIND == VLFB_OP_STEM_MN ? (int)ld : g.W) + w0) * g.C;
      const int nh = g.kH, nw = (KIND == VLFB_OP_STEM_MN) ? 8 : g.kW;
      const int dh = (KIND == VLFB_OP_STEM_MN) ? 1 : g.dH, dw = (KIND == VLFB_OP_STEM_MN) ? 1 : g.dW;
      int hm = 0, wm = 0;
      for (int q = 0, h = h0; q < nh; ++q, h += dh) hm |= ((unsigned)h < (unsigned)g.H) ? (1 << q) : 0;
      for (int q = 0, w = w0; q < nw; ++q, w += dw) wm |= ((unsigned)w < (unsigned)g.W) ? (256 << q) : 0;
      info_b = okt ? (hm | wm) : 0;
    }
    int lane_src = kk0;
    uint32_t d = tile + dst0;
#pragma unroll
    for (int j = 0; j < MAXS; ++j) {
      if (j >= nslot) break;
      bool ok = colok;
      const float* src = base;
      if (KIND == VLFB_OP_DENSE_MN) {
        const int k = k0 + lane_src;
        ok = ok && k < kend;
        if (ok) src = base + (int64_t)k * ld + mn;
      } else {
        const int ra = __shfl_sync(0xffffffffu, info_a, lane_src);
        const int rb = __shfl_sync(0xffffffffu, info_b, lane_src);
        ok = ok && (((rb >> sh) & (rb >> sw) & 1) != 0);
        if (ok) src = base + (ra + slotoff);
      }
      // columns beyond the matrix are never copied: whatever shared memory holds there only reaches accumulator
      // columns >= N, which the epilogue does not store (k tails of real columns ARE zero-filled)
      if (colok) cp_async16(d, src, ok);
      lane_src += kstep;
      d += dstep;
    }
  }
};

// ---------------------------------------------------------------- the kernel
// Timeline instrumentation of the diagnostic build (-DVLFB_TRACE, scripts/trace_gemm.py): per CTA 64 clock64 slots.
//   0 entry, 1 globaltimer at entry, 2 prologue done, 3 exit; producer 8+2i / 9+2i = work item i first / last copy issued;
//   MMA 16+2i first chunk landed, 17+2i last MMA issued; epilogue warp 0: 24+4i accumulator ready, 25+4i blocks done,
//   26+4i piece counted, 27+4i fix-up done.
#ifdef VLFB_TRACE
unsigned long long* g_trace_buf = nullptr;
#define TR(slot) do { if (L.trace) L.trace[(size_t)blockIdx.x * 64 + (slot)] = (unsigned long long)clock64(); } while (0)
#else
#define TR(slot) do { } while (0)
#endif
constexpr int MAX_UNITS = 160;       // >= #SMs: CTAs (or CTA pairs) of the persistent grid
constexpr int SK_CNT_INTS = 16384;   // arrival counters at the head of the stream-K workspace (tile x rank x epilogue warp)

// the lean epilogue addresses D / residual / sign bits with 32-bit element offsets
__host__ __device__ inline bool span32_ok(const vlfb_gemm_params_t& p) {
  const long long z = p.taps > 1 ? (long long)(p.taps - 1) * p.d_tap_stride : (long long)(p.batch - 1) * p.d_batch_stride;
  return z >= 0 && p.ldd > 0 && (long long)p.M * p.ldd + z < (1ll << 32);
}

struct ParCls { short nh, nw, rh, rw, ph, pw; int nk; };   // taps per dim, first tap, parity, K chunks of the class

struct Launch {
  int bn;        // tile N (32/64/128/256) = UMMA N = TMEM columns
  int stages;
  PosDiv out;    // fast divisors of the conv OUTPUT extents (Wo, Ho, To)
  PosDiv in;     // ... and of the INPUT extents (W, H, T) for the dgrad row decode
  FastDiv cdiv;  // input channels C (wgrad: n -> (tap, ci))
  FastDiv kwdiv; // kW
  int tma_a, tma_b;  // operand fetched by TMA instead of cp.async: 1 = dense tiled boxes, 2 = im2col (conv gathers),
                     // 3 = conv1 stem rows: {8 px x 4 ch = 128 B, 16 output positions} boxes of the overlapping-window
                     //     view of a W-padded clip (make_tmap_stem)
  int lag;           // cp.async groups kept in flight before a stage is published (< stages)
  int tiles_m, tiles_n, total_tiles;
  int tile_rows;     // output rows per tile: 128, or 256 when a CTA pair shares the tile (cta_group::2)
  int stem_patch;    // conv1 forward: an M tile = a 16 (wo) x 8 (ho) patch of one output frame instead of 128 consecutive
                     // positions, so that ONE strided TMA box stages the whole A tile of a K chunk (tile row r =
                     // (ho0 + r / 16, wo0 + r % 16)); the fast epilogue maps rows back (patch_row)
  int patch_wb, patch_hb;   // patches per output row / per frame column: Wo / 16, Ho / 8 (forward), Ho / 2 (wgrad)
                            // conv1 WGRAD (B = STEM_MN) with stem_patch: K chunk = the 32 output positions of a
                            // 16 (wo) x 2 (ho) patch; ONE box stages the sH + kH input rows all kH filter-row atoms need
                            // ([input row][16 windows][128 B] slabs; atom kh of output row j = slab j*sH + kh, so the UMMA
                            // descriptor's atom stride is one slab) and one 4-D box per 32 channels stages dY^T
  // Strided conv dgrad (A = DGRAD_K, sH / sW = 2) as sH * sW PARITY CLASSES: the input positions (h, w) = (sH h' + ph,
  // sW w' + pw) of one class receive only the filter taps kh = rh + sH j, kw = rw + sW i (rh = (ph + pH) % sH ...), i.e.
  // each class is a unit-stride convolution over dY with nh x nw taps (3x3 stride 2: 1 + 2 + 2 + 4 = 9 taps for the four
  // classes instead of 4 x 9 with three quarters of the gathered operand zero).  The class is the tile's z index: M
  // tiles run over the class's sub-grid (W / sW, H / sH, T, N), A is one im2col box over dY per chunk, B the chunk of
  // the transposed weights at the ORIGINAL tap, and the epilogue maps sub-grid rows back to dX rows (par_row).
  int par;           // number of parity classes (0 = off)
  int par_m;         // rows of one class = N T (H / sH) (W / sW)
  int par_lo[2];     // im2col origin offset (w, h) shared by the classes: (p + ph) / s - (taps - 1)
  PosDiv sub;        // fast divisors of the sub-grid extents
  ParCls par_cls[4];
  // Stream-K: the linear space (tile, K chunk) is cut into one contiguous range per unit (CTA or CTA pair), so every
  // SM gets the same number of chunks whatever the tile count.  A tile whose chunks span several units is reduced
  // through the workspace by the LAST unit to arrive at its counter (no unit ever waits for another).
  int sk;
  int nkt;           // K chunks per tile
  float* ws_tiles;   // partial-sum slots: [unit][2][rank][128][bn]
  int* ws_cnt;       // arrival counters [tile][rank][epilogue warp], zero between launches
  unsigned long long* trace;   // diagnostic build only
  int bounds[MAX_UNITS + 1];
};

struct TileInfo {
  int m0, n0, batch, tap, k_begin, k_end, nk;
  int tile;          // linear tile index
  // stream-K: units sharing this tile, packed to keep the epilogue's register budget:
  //   bits 0-7 npieces (1 = whole tile here), 8-15 first unit, 16 = workspace slot (0/1) of that first unit's piece
  //   (every later piece is in slot 0), 17 = this unit's slot
  int pinfo;
  __device__ __forceinline__ int npieces() const { return pinfo & 0xFF; }
  __device__ __forceinline__ int ufirst() const { return (pinfo >> 8) & 0xFF; }
  __device__ __forceinline__ int first_slot() const { return (pinfo >> 16) & 1; }
  __device__ __forceinline__ int slot() const { return (pinfo >> 17) & 1; }
};

// Linear tile index -> (m tile fastest, n tile, z = batch|tap x split): CTAs that run concurrently share the
// same weight (B) tile in L2.
__device__ __forceinline__ void decode_tile(const vlfb_gemm_params_t& p, const Launch& L, int t, int rank, int split_k,
                                            TileInfo& ti) {
  const int mt = t % L.tiles_m;
  const int r = t / L.tiles_m;
  const int nt = r % L.tiles_n;
  const int z = r / L.tiles_n;
  const int split = z % split_k, zz = z / split_k;
  ti.batch = (p.taps > 1) ? 0 : zz;
  ti.tap = (p.taps > 1) ? zz : 0;
  ti.m0 = mt * L.tile_rows + rank * BM;
  ti.n0 = nt * L.bn;
  int kper = (p.K + split_k - 1) / split_k;
  kper = (kper + KC - 1) / KC * KC;
  ti.k_begin = split * kper;
  ti.k_end = min(p.K, ti.k_begin + kper);
  ti.nk = (ti.k_end > ti.k_begin) ? (ti.k_end - ti.k_begin + KC - 1) / KC : 0;
  if (L.par) {                     // z = parity class: its own K extent (possibly zero: epilogue-only tiles)
    ti.k_begin = 0;
    ti.nk = L.par_cls[zz].nk;
    ti.k_end = ti.nk * KC;
  }
  ti.tile = t;
  ti.pinfo = 1;
}

// strided-dgrad parity classes: dX row of sub-grid row m of class c
__device__ __forceinline__ int par_row(const vlfb_gemm_params_t& p, const Launch& L, int cls, int m) {
  const Pos4 o = decode_pos_fast((uint32_t)m, L.sub);
  const ParCls& c = L.par_cls[cls];
  return ((o.n * p.g.T + o.t) * p.g.H + o.h * p.g.sH + c.ph) * p.g.W + o.w * p.g.sW + c.pw;
}

// conv1 patch tiles: linear output position of tile row r of M tile `mt`
__device__ __forceinline__ int patch_row(const vlfb_gemm_params_t& p, const Launch& L, int mt, int r) {
  const int wb = mt % L.patch_wb, q = mt / L.patch_wb;
  const int hb = q % L.patch_hb, rest = q / L.patch_hb;            // rest = n * To + to
  return (rest * p.g.Ho + hb * 8 + (r >> 4)) * p.g.Wo + wb * 16 + (r & 15);
}

// Every role of a CTA (and both CTAs of a pair) walks the same work sequence.  cur/lim = next tile index / tile
// count (static loop, stride = #units) or next / end position in the (tile, K chunk) space (stream-K).
struct Sched { int cur, lim; };
__device__ __forceinline__ void sched_init(Sched& s, const Launch& L, int unit) {
  s.cur = L.sk ? L.bounds[unit] : unit;
  s.lim = L.sk ? L.bounds[unit + 1] : L.total_tiles;
}
__device__ __forceinline__ bool sched_next(const vlfb_gemm_params_t& p, const Launch& L, Sched& s, int unit, int nunits,
                                           int rank, TileInfo& ti) {
  if (L.sk) {
    if (s.cur >= s.lim) return false;
    const int tile = s.cur / L.nkt;
    const int c0 = s.cur - tile * L.nkt;
    const int len = min(L.nkt - c0, s.lim - s.cur);
    decode_tile(p, L, tile, rank, 1, ti);
    ti.k_begin = c0 * KC;
    ti.k_end = min(p.K, (c0 + len) * KC);
    ti.nk = len;
    if (len != L.nkt && L.ws_tiles != nullptr) {
      const int s0 = tile * L.nkt, e0 = s0 + L.nkt;
      int uf = unit, ul = unit;
      while (L.bounds[uf] > s0) --uf;
      while (L.bounds[ul + 1] < e0) ++ul;
      const int first_slot = (L.bounds[uf] < s0) ? 1 : 0;
      const int slot = (unit == uf) ? first_slot : 0;
      ti.pinfo = (ul - uf + 1) | (uf << 8) | (first_slot << 16) | (slot << 17);
    }
    s.cur += len;
    return true;
  }
  while (s.cur < s.lim) {
    decode_tile(p, L, s.cur, rank, p.split_k, ti);
    s.cur += nunits;
    if (ti.nk != 0 || L.par) return true;
  }
  return false;
}

// Persistent, warp-specialised: grid = min(#tiles, #SMs) CTAs (PAIR: 2 x #pairs in clusters of two); every role walks
// the same work sequence (Sched).  The smem ring (full/empty) runs continuously across tiles and the TMEM accumulator
// is double-buffered (tmem_full/tmem_empty), so the epilogue of tile i overlaps the loads and MMAs of tile i+1.
// PAIR (both operands staged by TMA only): the two CTAs of a cluster own one 256 x bn tile; CTA r stages A rows
// [m0 + 128 r, +128) and B rows [n0 + (bn/2) r, +bn/2); the leader issues tcgen05.mma.cta_group::2 (M = 256) which
// reads both CTAs' shared memory and writes 128 accumulator lanes x bn columns into EACH CTA's TMEM, so every SM
// receives (128 + bn/2) x 128 B per K chunk instead of (128 + bn) x 128 B for the same MACs.
// CP = false: both operands are staged by TMA, so ONE producer warp suffices and the CTA is 10 warps (producer, MMA
// issuer, 8 epilogue warps) with up to 168 registers per thread -- the 17-warp CP = true build (8 cp.async gather
// warps: conv1 stem, strided dgrad, operands TMA cannot address) is capped at 96 and spills in the epilogue.
template <int AK, int BK, bool MASK, bool PAIR, bool CP>
__global__ void __launch_bounds__((CP ? NPROD : 32 * NTMAW) + 32 + NEPI, 1) gemm_tc_kernel(const vlfb_gemm_params_t p, const Launch L,
                                                              const __grid_constant__ CUtensorMap tmA,
                                                              const __grid_constant__ CUtensorMap tmB) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const int bn = L.bn, S = L.stages;
  const int bnh = PAIR ? (bn >> 1) : bn;                    // B rows (columns of D) staged by this CTA
  const uint32_t b_tile_bytes = (uint32_t)bnh * KC * 4;
  const uint32_t stage_bytes = A_TILE_BYTES + b_tile_bytes;
  const uint32_t epi_base = smem_base + S * stage_bytes;                  // per-epilogue-warp transpose tiles
  const uint32_t bar_base = epi_base + EPI_STAGE_BYTES;
  const uint32_t full0 = bar_base, empty0 = bar_base + 8 * MAX_STAGES;
  const uint32_t tfull0 = bar_base + 16 * MAX_STAGES, tempty0 = tfull0 + 16;
  const uint32_t tptr_addr = tempty0 + 16;
  volatile uint32_t* tptr_generic =
      reinterpret_cast<volatile uint32_t*>(smem_raw + (tptr_addr - smem_u32(smem_raw)));

  static_assert(!(PAIR && CP), "CTA pairs need both operands staged by TMA");
  constexpr int NPRODT = CP ? NPROD : 32 * NTMAW;   // producer threads of this build
  constexpr int NPWT = NPRODT / 32;
  constexpr int NTHR = NPRODT + 32 + NEPI;
  const int tid = threadIdx.x, warp = tid >> 5;
  const int rank = PAIR ? (int)cluster_ctarank() : 0;
  const int unit = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int nunits = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  const bool tma_a = L.tma_a != 0, tma_b = L.tma_b != 0;
  const bool cp_any = CP && !(tma_a && tma_b);

#ifdef VLFB_TRACE
  if (tid == 0 && L.trace) {
    unsigned long long gt;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
    L.trace[(size_t)blockIdx.x * 64 + 1] = gt;
    TR(0);
  }
#endif
  if (tid == 0) {
    for (int s = 0; s < S; ++s) {
      mbar_init(full0 + 8 * s, (cp_any ? NPROD : 0) + ((tma_a || tma_b) ? 1 : 0));
      mbar_init(empty0 + 8 * s, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull0 + 8 * a, 1);
      mbar_init(tempty0 + 8 * a, PAIR ? 2 * (NEPI / 32) : NEPI / 32);       // one arrival per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  uint32_t tmem_cols = 32;              // tcgen05.alloc takes a power of two >= 32; two accumulators of bn columns
  while (tmem_cols < (uint32_t)(2 * bn)) tmem_cols <<= 1;
  if (warp == NPWT) {
    if (PAIR) tmem_alloc2(tptr_addr, tmem_cols); else tmem_alloc(tptr_addr, tmem_cols);
  }
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();     // PAIR: the peer's barriers exist before anything signals them
  tc_fence_after();
  const uint32_t tmem = *tptr_generic;
  if (tid == 0) TR(2);

  if (warp < NPWT) {
    // ============================ PRODUCERS (8 cp.async warps / NTMAW TMA issuers) ============================
    // TMA issuers: thread 0 in a CP build; lane 0 of every producer warp in a TMA-only build.  All issuers walk the same
    // tile / chunk sequence with their own copy of the (deterministic) gather state and wait for the free stage
    // themselves; issuer `hid` launches the boxes b with b % NISS == hid; issuer 0 posts the expected byte count.
    constexpr int NISS = CP ? 1 : NTMAW;
    const int hid = CP ? 0 : (tid >> 5);
    const bool issuer = CP ? (tid == 0) : ((tid & 31) == 0);
    if (cp_any || issuer) {
      KLoader<is_mn(AK) ? VLFB_OP_DENSE_K : AK, BM / RSTEP> ka;
      MNLoader<is_mn(AK) ? AK : VLFB_OP_DENSE_MN> ma;
      KLoader<is_mn(BK) ? VLFB_OP_DENSE_K : BK, 256 / RSTEP> kb;
      MNLoader<is_mn(BK) ? BK : VLFB_OP_DENSE_MN> mb;
      const int LAG = L.lag;
      // compile-time gates keep the im2col state out of the instantiations that cannot use it (registers)
      const bool im2col_a = (AK == VLFB_OP_CONV_K || AK == VLFB_OP_DGRAD_K) && L.tma_a == 2;
      const bool im2col_b = BK == VLFB_OP_CONV_MN && L.tma_b == 2;
      constexpr int NATOM = BK == VLFB_OP_CONV_MN ? 8 : 1;
      // im2col state of the issuing thread: window origin of the tile's first row + filter-tap cursor (A), and
      // per 32-column atom the channel slice / tap offsets of the wgrad B tile
      int ia_w = 0, ia_h = 0, ia_d = 0, ia_n = 0, ic_t = 0, ic_h = 0, ic_w = 0, ic_c = 0, icpt = 1;
      int ib_c[NATOM], ib_off[NATOM], ib_atoms = 0;
      // conv1 stem rows (tma 3): the 128 tile rows = 8 groups of 16 consecutive output positions (16 | Wo, so a group
      // never crosses an output row): per group the window origin (wo, hi0 = ho sH - pH, ti0 = to sT - pT, n)
      const bool stem_a = !PAIR && AK == VLFB_OP_STEM_K && L.tma_a == 3;
      const bool stem_b = !PAIR && BK == VLFB_OP_STEM_MN && L.tma_b == 3;
      constexpr int NSG = AK == VLFB_OP_STEM_K ? 8 : 1;
      int sg_w[NSG], sg_ht[NSG], sg_n[NSG];
      // chunk counter over the CTA's whole work sequence; ring slot / phase / lagged slot advance
      // incrementally (S is a run-time value: `it % S` cost three integer divisions per chunk per thread)
      int it = 0, s = 0, sl = 0;
      uint32_t ph = 0;
      // PAIR: every copy of either CTA completes on the LEADER's stage barrier
      const uint32_t fullx = PAIR ? mapa_rank(full0, 0) : full0;
      auto ld3 = [&](uint32_t dst, const CUtensorMap* tm, int c0, int c1, int c2, uint32_t bar) {
        if (PAIR) tma_load_3d_2(dst, tm, c0, c1, c2, bar); else tma_load_3d(dst, tm, c0, c1, c2, bar);
      };
      auto ldi = [&](uint32_t dst, const CUtensorMap* tm, int c, int w, int h, int d, int n, int ow, int oh, int od,
                     uint32_t bar) {
        if (PAIR) tma_load_im2col_2(dst, tm, c, w, h, d, n, ow, oh, od, bar);
        else tma_load_im2col(dst, tm, c, w, h, d, n, ow, oh, od, bar);
      };
      Sched sc;
      sched_init(sc, L, unit);
      TileInfo ti;
      int witem = 0;
      while (sched_next(p, L, sc, unit, nunits, rank, ti)) {
        if (tid == 0 && witem < 4) TR(8 + 2 * witem);
        const int nb0 = ti.n0 + rank * bnh;              // first D column whose B rows this CTA stages
        if (cp_any) {
          if (!tma_a) { if (is_mn(AK)) ma.init(p, p.a, ti.m0, BM, p.M, ti.batch, ti.tap, L.cdiv, L.kwdiv); else { ka.init(p, p.a, ti.m0, BM, p.M, ti.batch, L.out, L.in, ti.k_begin / KC); ka.kend = ti.k_end; } }
          if (!tma_b) { if (is_mn(BK)) mb.init(p, p.b, ti.n0, bn, p.N, ti.batch, ti.tap, L.cdiv, L.kwdiv); else { kb.init(p, p.b, ti.n0, bn, p.N, ti.batch, L.out, L.in, ti.k_begin / KC); kb.kend = ti.k_end; } }
        }
        const int kc0 = ti.k_begin / KC;
        // bytes the stage barrier expects: this CTA's copies (PAIR: both CTAs', posted by the leader)
        uint32_t tma_bytes = (tma_a ? (uint32_t)A_TILE_BYTES : 0u) + (tma_b ? b_tile_bytes : 0u);
        if (PAIR) tma_bytes *= 2u;
        if (issuer && stem_a && L.stem_patch) {
          const vlfb_conv_geom_t& g = p.g;
          const int mt = ti.m0 / BM;
          const int wb = mt % L.patch_wb, q = mt / L.patch_wb;
          const int hb = q % L.patch_hb, rest = q / L.patch_hb;
          const int to = rest % g.To, n = rest / g.To;
          sg_w[0] = wb * 16;
          sg_ht[0] = ((hb * 8 * g.sH - g.pH) << 16) | ((to * g.sT - g.pT) & 0xFFFF);
          sg_n[0] = n;
          ic_t = kc0 / g.kH;
          ic_h = kc0 - ic_t * g.kH;
        } else if (issuer && stem_a) {
          const vlfb_conv_geom_t& g = p.g;
          Pos4 o = decode_pos_fast((uint32_t)ti.m0, L.out);
#pragma unroll
          for (int q = 0; q < NSG; ++q) {
            sg_w[q] = o.w;
            sg_ht[q] = ((o.h * g.sH - g.pH) << 16) | ((o.t * g.sT - g.pT) & 0xFFFF);
            sg_n[q] = (ti.m0 + 16 * q < p.M) ? o.n : g.N;          // rows past M: out of bounds in N -> zeros
            o.w += 16;
            if (o.w >= g.Wo) { o.w = 0; if (++o.h == g.Ho) { o.h = 0; if (++o.t == g.To) { o.t = 0; ++o.n; } } }
          }
          ic_t = kc0 / g.kH;
          ic_h = kc0 - ic_t * g.kH;
        }
        if (issuer && im2col_a) {
          const vlfb_conv_geom_t& g = p.g;
          if (AK == VLFB_OP_CONV_K) {
            const Pos4 o = decode_pos_fast((uint32_t)ti.m0, L.out);
            ia_w = o.w * g.sW - g.pW; ia_h = o.h * g.sH - g.pH; ia_d = o.t * g.sT - g.pT; ia_n = o.n;
            icpt = g.C / KC;
          } else if (L.par) {   // parity class of a strided dgrad: unit-stride gather over dY with the class's taps
            const Pos4 o = decode_pos_fast((uint32_t)ti.m0, L.sub);
            ia_w = o.w + L.par_lo[0]; ia_h = o.h + L.par_lo[1];
            ia_d = o.t + g.pT - (g.kT - 1) * g.dT; ia_n = o.n;
            icpt = g.Co / KC;
          } else {  // DGRAD_K, unit strides: dx[i] = sum_tap dy[i + pad - tap*dil] -> origin i + pad - (k-1)*dil
            const Pos4 o = decode_pos_fast((uint32_t)ti.m0, L.in);
            ia_w = o.w + g.pW - (g.kW - 1) * g.dW; ia_h = o.h + g.pH - (g.kH - 1) * g.dH;
            ia_d = o.t + g.pT - (g.kT - 1) * g.dT; ia_n = o.n;
            icpt = g.Co / KC;
          }
          const int tap = kc0 / icpt;
          ic_c = kc0 - tap * icpt;
          decode_tap(tap, g.kH, g.kW, ic_t, ic_h, ic_w);     // (par: kc0 = 0 -> all zero; ic_h / ic_w count the class's taps)
        }
        if (issuer && im2col_b) {
          const vlfb_conv_geom_t& g = p.g;
          ib_atoms = 0;
          int peer_atoms = 0;
#pragma unroll
          for (int a = 0; a < NATOM; ++a) {
            const int ncol = nb0 + a * 32;
            if (a * 32 < bnh && ncol < p.N) {
              uint32_t tap_hw, ci, qh, qw;
              fd_divmod((uint32_t)ncol, L.cdiv, tap_hw, ci);       // n = (kh*kW + kw) * C + ci
              fd_divmod(tap_hw, L.kwdiv, qh, qw);
              ib_c[a] = (int)ci;
              ib_off[a] = ((int)qh * g.dH << 16) | ((int)qw * g.dW);
              ib_atoms = a + 1;
            }
            if (PAIR && a * 32 < bnh && ti.n0 + (rank ^ 1) * bnh + a * 32 < p.N) peer_atoms = a + 1;
          }
          tma_bytes = (PAIR ? 2u : 1u) * (tma_a ? (uint32_t)A_TILE_BYTES : 0u) + 4096u * (uint32_t)(ib_atoms + peer_atoms);
        }
        if (issuer && stem_b) {
          ib_atoms = 0;                                             // atoms = filter rows kh of this N tile
          for (int a = 0; a * 32 < bn && ti.n0 + a * 32 < p.N; ++a) ib_atoms = a + 1;
          tma_bytes = (tma_a ? (uint32_t)A_TILE_BYTES : 0u) + 4096u * (uint32_t)ib_atoms;
          if (L.stem_patch) {
            int a_atoms = 0;
            for (int a = 0; a * 32 < p.M && a < BM / 32; ++a) a_atoms = a + 1;
            tma_bytes = 4096u * (uint32_t)a_atoms + 2048u * (uint32_t)(p.g.sH + p.g.kH);
          }
        }
        for (int i = 0; i < ti.nk; ++i, ++it) {
          // Helper issuers (hid > 0) wait for the free stage LAZILY, right before their first box of the chunk: an issuer
          // without a box in a chunk (2-box chunks on 3 issuers) must not wait at all -- nothing would depend on it, the
          // others would lap it by two phases of the stage barrier and its parity wait would then never return (call P:
          // exactly that hang, 4 s later the watchdog trap, in the full-size captured step).
          const bool need_wait = it >= S;
          const uint32_t wpar = ph ^ 1u;
          const int s_cur = s;
          if (need_wait && (NISS == 1 || hid == 0 || cp_any)) mbar_wait(empty0 + 8 * s_cur, wpar);
          if (++s == S) { s = 0; ph ^= 1u; }
          const uint32_t a_tile = smem_base + s_cur * stage_bytes;
          const uint32_t b_tile = a_tile + A_TILE_BYTES;
          const uint32_t fbar = fullx + 8 * s_cur;
          if (issuer && tma_bytes) {
            if (hid == 0 && (!PAIR || rank == 0)) mbar_expect_tx(full0 + 8 * s_cur, tma_bytes);
            int box = 0;                                  // boxes of this chunk, in issue order
            bool waited = NISS == 1 || hid == 0;
            auto mine = [&]() {
              const bool m = NISS == 1 || (box % NISS) == hid;
              ++box;
              if (m && !waited) {
                if (need_wait) mbar_wait(empty0 + 8 * s_cur, wpar);
                waited = true;
              }
              return m;
            };
            if (stem_a) {
              const vlfb_conv_geom_t& g = p.g;
              if (L.stem_patch) {                     // one {128 B x 16 wo x 8 rows (stride sH)} box = the whole A tile
                if (mine()) tma_load_5d(a_tile, &tmA, 0, sg_w[0], (sg_ht[0] >> 16) + ic_h, (int)(short)(sg_ht[0] & 0xFFFF) + ic_t, sg_n[0], fbar);
              } else {
#pragma unroll
                for (int q = 0; q < NSG; ++q)
                  if (mine()) tma_load_5d(a_tile + q * 2048, &tmA, 0, sg_w[q], (sg_ht[q] >> 16) + ic_h, (int)(short)(sg_ht[q] & 0xFFFF) + ic_t,
                              sg_n[q], fbar);
              }
              if (++ic_h == g.kH) { ic_h = 0; ++ic_t; }
            } else if (im2col_a) {
              const vlfb_conv_geom_t& g = p.g;
              if (AK == VLFB_OP_CONV_K) {
                if (mine()) ldi(a_tile, &tmA, ic_c * KC, ia_w, ia_h, ia_d, ia_n, ic_w * g.dW, ic_h * g.dH, ic_t * g.dT, fbar);
              } else if (AK == VLFB_OP_DGRAD_K && L.par) {
                // tap (kt, rh + sH ic_h, rw + sW ic_w) of the class: dY offset (taps - 1 - index), weights at the original tap
                const ParCls& c = L.par_cls[ti.batch];
                if (mine()) ldi(a_tile, &tmA, ic_c * KC, ia_w, ia_h, ia_d, ia_n, c.nw - 1 - ic_w, c.nh - 1 - ic_h, (g.kT - 1 - ic_t) * g.dT, fbar);
                const int tap = (ic_t * g.kH + c.rh + g.sH * ic_h) * g.kW + c.rw + g.sW * ic_w;
                if (mine()) ld3(b_tile, &tmB, tap * g.Co + ic_c * KC, nb0, 0, fbar);
                if (++ic_c == icpt) {
                  ic_c = 0;
                  if (++ic_w == c.nw) { ic_w = 0; if (++ic_h == c.nh) { ic_h = 0; ++ic_t; } }
                }
              } else {
                if (mine()) ldi(a_tile, &tmA, ic_c * KC, ia_w, ia_h, ia_d, ia_n, (g.kW - 1 - ic_w) * g.dW,
                    (g.kH - 1 - ic_h) * g.dH, (g.kT - 1 - ic_t) * g.dT, fbar);
              }
              if (!(AK == VLFB_OP_DGRAD_K && L.par) && ++ic_c == icpt) {
                ic_c = 0;
                if (++ic_w == g.kW) { ic_w = 0; if (++ic_h == g.kH) { ic_h = 0; ++ic_t; } }
              }
            } else if (tma_a && !(stem_b && L.stem_patch)) {
              if (is_mn(AK) && L.tma_a == 4) {            // all atoms of the tile in one box
                if (mine()) tma_load_4d(a_tile, &tmA, 0, ti.k_begin + i * KC, ti.m0 >> 5, ti.batch, fbar);
              } else if (is_mn(AK)) {
                for (int a = 0; a < BM / 32; ++a)
                  if (mine()) ld3(a_tile + a * 4096, &tmA, ti.m0 + a * 32, ti.k_begin + i * KC, ti.batch, fbar);
              } else {
                if (mine()) ld3(a_tile, &tmA, (kc0 + i) * KC, ti.m0, ti.batch, fbar);
              }
            }
            if (stem_b && L.stem_patch) {
              const vlfb_conv_geom_t& g = p.g;
              const int q = ti.k_begin / KC + i;                     // chunk -> patch (wb, row pair, frame)
              const int wb = q % L.patch_wb, q2 = q / L.patch_wb;
              const int hp = q2 % L.patch_hb, rest = q2 / L.patch_hb;
              const int to = rest % g.To, n = rest / g.To;
              if (mine()) tma_load_5d(b_tile, &tmB, 0, wb * 16, hp * 2 * g.sH - g.pH, to * g.sT - g.pT + ti.tap, n, fbar);
              for (int a = 0; a * 32 < p.M && a < BM / 32; ++a)      // dY^T: {32 channels, 16 wo, 2 ho} per atom
                if (mine()) tma_load_4d(a_tile + a * 4096, &tmA, ti.m0 + a * 32, wb * 16, hp * 2, rest, fbar);
            } else if (stem_b) {
              // conv1 wgrad B tile: 32 output positions (k rows) = 2 groups of 16; per filter row kh one 32-column atom
              // (8 px x 4 ch) = two {128 B x 16 positions} boxes of the overlapping-window view
              const vlfb_conv_geom_t& g = p.g;
              const int kh0 = ti.n0 >> 5;
#pragma unroll
              for (int hf = 0; hf < 2; ++hf) {
                const int kpos = ti.k_begin + i * KC + 16 * hf;
                const Pos4 o = decode_pos_fast((uint32_t)(kpos < p.K ? kpos : 0), L.out);
                const int bn_ = kpos < p.K ? o.n : g.N;
                const int bh = o.h * g.sH - g.pH + kh0, bt = o.t * g.sT - g.pT + ti.tap;
                for (int a = 0; a < ib_atoms; ++a)
                  if (mine()) tma_load_5d(b_tile + a * 4096 + hf * 2048, &tmB, 0, o.w, bh + a, bt, bn_, fbar);
              }
            } else if (BK == VLFB_OP_CONV_MN && L.tma_b == 5) {
              // wgrad B tile of a convolution without spatial taps: 32 consecutive positions of one clip, shifted by whole
              // frames for the temporal tap, all channel atoms of the tile in ONE box (make_tmap_conv_flat)
              const vlfb_conv_geom_t& g = p.g;
              const uint32_t hw = (uint32_t)(g.H * g.W), thw = (uint32_t)g.T * hw;
              const uint32_t kpos = (uint32_t)(ti.k_begin + i * KC);
              const uint32_t n = kpos / thw;
              const int pos = (int)(kpos - n * thw) + (ti.tap * g.dT - g.pT) * (int)hw;
              if (mine()) tma_load_4d(b_tile, &tmB, 0, pos, nb0 >> 5, (int)n, fbar);
            } else if (im2col_b) {
              // wgrad B tile: 32 output positions (k rows) x one (kh, kw, 32-channel) atom per copy
              const vlfb_conv_geom_t& g = p.g;
              const Pos4 o = decode_pos_fast((uint32_t)(ti.k_begin + i * KC), L.out);
              const int bw = o.w * g.sW - g.pW, bh = o.h * g.sH - g.pH, bd = o.t * g.sT - g.pT;
#pragma unroll
              for (int a = 0; a < NATOM; ++a)
                if (a < ib_atoms)
                  if (mine()) ldi(b_tile + a * 4096, &tmB, ib_c[a], bw, bh, bd, o.n, ib_off[a] & 0xFFFF, ib_off[a] >> 16,
                      ti.tap * g.dT, fbar);
            } else if (tma_b && !(AK == VLFB_OP_DGRAD_K && L.par)) {
              if (is_mn(BK) && L.tma_b == 4) {
                if (mine()) tma_load_4d(b_tile, &tmB, 0, ti.k_begin + i * KC, nb0 >> 5, ti.batch, fbar);
              } else if (is_mn(BK)) {
                for (int a = 0; a < bnh / 32; ++a)
                  if (mine()) ld3(b_tile + a * 4096, &tmB, nb0 + a * 32, ti.k_begin + i * KC, ti.batch, fbar);
              } else {
                if (mine()) ld3(b_tile, &tmB, (kc0 + i) * KC, nb0, ti.batch, fbar);
              }
            }
          }
          if (!cp_any) continue;
          if (!tma_a) {
            if (is_mn(AK)) ma.issue(p, L.out, ti.k_begin + i * KC, ti.k_end, a_tile);
            else ka.issue(p, kc0 + i, a_tile);
          }
          if (!tma_b) {
            if (is_mn(BK)) mb.issue(p, L.out, ti.k_begin + i * KC, ti.k_end, b_tile);
            else kb.issue(p, kc0 + i, b_tile);
          }
          cp_async_commit();
          if (it >= LAG) {
            cp_async_wait_dyn(LAG);
            fence_proxy_async();
            mbar_arrive(full0 + 8 * sl);
            if (++sl == S) sl = 0;
          }
        }
        if (tid == 0 && witem < 4) TR(9 + 2 * witem);
        ++witem;
      }
      if (cp_any) {
        cp_async_wait<0>();
        fence_proxy_async();
        for (int c = (it > LAG ? it - LAG : 0); c < it; ++c) {
          mbar_arrive(full0 + 8 * sl);
          if (++sl == S) sl = 0;
        }
      }
    }
  } else if (warp == NPWT) {
    // ============================ MMA ISSUER (1 thread; PAIR: the leader CTA's) ============================
    if ((tid & 31) == 0 && rank == 0) {
      const uint32_t idesc = make_idesc(bn, is_mn(AK) ? 1 : 0, is_mn(BK) ? 1 : 0, PAIR ? 2 * BM : BM);
      // K-major tile: SWIZZLE_128B, LBO 16, SBO 1024, K step 32 B; MN-major: SWIZZLE_128B_BASE32B, LBO 4096, SBO 512,
      // K step 1024 B (4 k-rows of 128 B per 32-element atom)
      const uint64_t a_d0 = is_mn(AK) ? make_desc(smem_base, 4096, 512, 1) : make_desc(smem_base, 16, 1024);
      const uint64_t b_d0 = is_mn(BK) ? make_desc(smem_base + A_TILE_BYTES, 4096, 512, 1) : make_desc(smem_base + A_TILE_BYTES, 16, 1024);
      const uint32_t a_hi = (uint32_t)(a_d0 >> 32), b_hi = (uint32_t)(b_d0 >> 32);
      const uint32_t a_lo0 = (uint32_t)a_d0, b_lo0 = (uint32_t)b_d0;
      const uint32_t stage_units = stage_bytes >> 4;
      // conv1 wgrad patch chunks: atoms (filter rows) are one 2 KB input-row slab apart (LBO 2048), the second output row
      // of the patch starts sH slabs further
      const bool stem_pb = !PAIR && BK == VLFB_OP_STEM_MN && L.tma_b == 3 && L.stem_patch != 0;
      const uint32_t b_lo0_pb = (uint32_t)make_desc(smem_base + A_TILE_BYTES, 2048, 512, 1);     // LBO lives in the low word
      const uint32_t pb_rowstep = (uint32_t)(p.g.sH * 2048) >> 4;
      constexpr uint32_t a_kstep = is_mn(AK) ? (1024u >> 4) : (32u >> 4), b_kstep = is_mn(BK) ? (1024u >> 4) : (32u >> 4);
      int it = 0, tile_iter = 0, s = 0;
      uint32_t ph = 0;
      Sched sc;
      sched_init(sc, L, unit);
      TileInfo ti;
      while (sched_next(p, L, sc, unit, nunits, rank, ti)) {
        const int acc = tile_iter & 1;
        if (tile_iter >= 2) {                          // wait until the epilogue(s) drained this accumulator
          mbar_wait(tempty0 + 8 * acc, ((tile_iter >> 1) - 1) & 1);
          tc_fence_after();
        }
        const uint32_t d_tmem = tmem + (uint32_t)(acc * bn);
        for (int i = 0; i < ti.nk; ++i, ++it) {
          mbar_wait(full0 + 8 * s, ph);
          if (i == 0 && tile_iter < 4) TR(16 + 2 * tile_iter);
          tc_fence_after();
          // descriptors of the stage: only the 14-bit start-address field moves (by stage, then by the 32-byte /
          // 1024-byte K step of a K-major / MN-major tile), so each MMA costs one 32-bit add per operand instead of
          // re-encoding the descriptor (trace r2b: the issue loop, not the tensor pipe, paced tiles narrower than 256)
          const uint32_t a_lo = a_lo0 + (uint32_t)s * stage_units, b_lo = b_lo0 + (uint32_t)s * stage_units;
#pragma unroll
          for (int j = 0; j < KC / 8; ++j) {          // UMMA K = 8 for tf32
            const uint64_t da = ((uint64_t)a_hi << 32) | (uint64_t)(a_lo + (uint32_t)j * a_kstep);
            uint64_t db = ((uint64_t)b_hi << 32) | (uint64_t)(b_lo + (uint32_t)j * b_kstep);
            if (BK == VLFB_OP_STEM_MN && stem_pb)     // k rows 0-15 = output row 0 (slab kh), 16-31 = output row 1 (slab sH + kh)
              db = ((uint64_t)b_hi << 32) |
                   (uint64_t)(b_lo0_pb + (uint32_t)s * stage_units + (uint32_t)(j >> 1) * pb_rowstep + (uint32_t)(j & 1) * (1024u >> 4));
            if (PAIR) umma_tf32_2(d_tmem, da, db, idesc, (i | j) ? 1u : 0u);
            else umma_tf32(d_tmem, da, db, idesc, (i | j) ? 1u : 0u);
          }
          // frees the smem stage (PAIR: in both CTAs) when these MMAs retire
          if (PAIR) umma_commit2(empty0 + 8 * s); else umma_commit(empty0 + 8 * s);
          if (++s == S) { s = 0; ph ^= 1u; }
        }
        // accumulator complete -> epilogue (PAIR: of both CTAs); a parity class without taps has nothing to wait for
        if (!PAIR && ti.nk == 0) mbar_arrive(tfull0 + 8 * acc);
        else if (PAIR) umma_commit2(tfull0 + 8 * acc); else umma_commit(tfull0 + 8 * acc);
        if (tile_iter < 4) TR(17 + 2 * tile_iter);
        ++tile_iter;
      }
    }
  } else {
    // ============================ EPILOGUE (8 warps) ============================
    // TMEM lane quarter = warp % 4 (hardware rule); the two warps of a quarter take alternate 16-column
    // blocks.  Each 32x16 block is transposed through a padded shared-memory tile so that a warp store /
    // residual load / atomic covers 8 rows x 64 contiguous bytes (whole 32-byte sectors).
    const int ew = warp - NPWT - 1;
    const int quarter = warp & 3;
    const int half = ew >> 2;
    const int lane = tid & 31;
    float* stg = reinterpret_cast<float*>(smem_raw + (epi_base - smem_u32(smem_raw))) + ew * EPI_WARP_FLOATS;
    float* wsc = stg + 32 * EPITCH;      // column scale of this warp's column blocks, then the bias
    float* wbi = wsc + 128;
    int colv_n0 = -1;
    const bool vec_ok = ((p.ldd & 3) == 0) && ((p.d_batch_stride & 3) == 0) && ((p.d_tap_stride & 3) == 0) &&
                        ((reinterpret_cast<uintptr_t>(p.d) & 15) == 0) &&
                        (!p.residual || (reinterpret_cast<uintptr_t>(p.residual) & 15) == 0) &&
                        (!p.relu_mask || (reinterpret_cast<uintptr_t>(p.relu_mask) & 15) == 0) &&
                        !(p.residual && (p.flags & VLFB_EPI_ACCUM));
    const int col = (lane & 3) * 4;
    const bool want_res = (p.residual != nullptr) || (p.flags & VLFB_EPI_ACCUM);
    const float* res_src = p.residual ? p.residual : p.d;
    const uint32_t tempty_x = (PAIR && rank != 0) ? mapa_rank(tempty0, 0) : tempty0;
    const int nrank = PAIR ? 2 : 1;
    const size_t ws_tile_floats = (size_t)BM * bn;
    int tile_iter = 0;
    Sched sc;
    sched_init(sc, L, unit);
    TileInfo ti;
    while (sched_next(p, L, sc, unit, nunits, rank, ti)) {
      const int acc = tile_iter & 1;
      const uint32_t lane_addr = tmem + (uint32_t)(acc * bn) + ((uint32_t)(quarter * 32) << 16);
      const bool par = !PAIR && AK == VLFB_OP_DGRAD_K && L.par != 0;
      const int64_t tile_off = par ? 0 : (int64_t)ti.batch * p.d_batch_stride + (int64_t)ti.tap * p.d_tap_stride;
      if ((want_res || MASK) && !par) {
        // pull the NEXT tile's residual / mask rows into L2 while this tile is being written out
        Sched sn = sc;
        TileInfo tn;
        if (sched_next(p, L, sn, unit, nunits, rank, tn) && tn.npieces() == 1) {
          const int64_t noff = (int64_t)tn.batch * p.d_batch_stride + (int64_t)tn.tap * p.d_tap_stride;
          const int segs = bn >> 5;
          for (int idx = tid - (NPRODT + 32); idx < BM * segs; idx += NEPI) {
            const int row = idx / segs, seg = idx - row * segs;
            const int m = tn.m0 + row, n = tn.n0 + seg * 32;
            if (m < p.M && n < p.N) {
              if (want_res) prefetch_l2(res_src + noff + (int64_t)m * p.ldd + n);
              if (MASK && p.relu_mask) prefetch_l2(p.relu_mask + noff + (int64_t)m * p.ldd + n);
            }
          }
        }
      }
      if (ti.n0 != colv_n0) {
        // per-column affine of this warp's blocks -> shared memory, once per N tile (not per block: the
        // global-load latency used to sit in front of every block's first FFMA)
        colv_n0 = ti.n0;
        for (int i = lane; i < (bn >> 1); i += 32) {
          const int n = ti.n0 + half * EPC + (i >> 4) * (2 * EPC) + (i & 15);
          wsc[i] = (p.col_scale && n < p.N) ? p.col_scale[n] : 1.f;
          wbi[i] = (p.col_bias && n < p.N) ? p.col_bias[n] : 0.f;
        }
        __syncwarp();
      }
      float rs[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int m = ti.m0 + quarter * 32 + (lane >> 2) + 8 * i;
        rs[i] = (p.row_scale && m < p.M) ? p.row_scale[m] : 1.f;
      }
      // One pass over this warp's column blocks.  mode 0: accumulator -> fused epilogue -> D (whole tile here);
      // mode 1 (stream-K piece): raw accumulator -> this unit's workspace slot; mode 2 (last unit to arrive at a
      // shared tile): sum of ALL pieces' slots in piece order (deterministic) -> fused epilogue -> D.
      auto run_blocks = [&](auto mode_c) {
        constexpr int mode = decltype(mode_c)::value;
        const bool wres = want_res && mode != 1;
        // residual / accumulate operands are fetched one column block ahead (register double buffer): with only
        // 8 epilogue warps per SM the loads must be in flight while the previous block is stored, otherwise the
        // epilogue is DRAM-latency bound (Little's law) instead of bandwidth bound
        auto load_res = [&](int c0, float4* r) {
          const int n = ti.n0 + c0 + col;
          const bool ok = wres && vec_ok && c0 < bn && n + 3 < p.N;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int m = ti.m0 + quarter * 32 + (lane >> 2) + 8 * i;
            r[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ok && m < p.M) r[i] = ld_nc_f4(res_src + tile_off + (int64_t)m * p.ldd + n);
          }
        };
        // ReLU mask (backward of the ReLU that produced this GEMM's D-shaped input): fetched one block ahead like
        // the residual, but AFTER the accumulator block has left the registers and packed to 16 bits as soon as
        // it arrives, so that it never coexists with v[] / both residual buffers (register budget of 17 warps;
        // holding it as 4 more float4 spilled the whole epilogue loop -- measured 1.5-2.8x slower).
        auto load_mask = [&](int c0, float4* mk) {
          const int n = ti.n0 + c0 + col;
          const bool ok = mode != 1 && vec_ok && c0 < bn && n + 3 < p.N;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int m = ti.m0 + quarter * 32 + (lane >> 2) + 8 * i;
            mk[i] = make_float4(1.f, 1.f, 1.f, 1.f);
            if (ok && m < p.M) {
              const int64_t e = tile_off + (int64_t)m * p.ldd + n;
              if (p.relu_mask) {
                mk[i] = ld_nc_f4(p.relu_mask + e);
              } else {                                 // sign bits (n % 4 == 0: the four bits sit in one word)
                const uint32_t nib = p.relu_mask_bits[e >> 5] >> (e & 31);
                mk[i] = make_float4((nib & 1u) ? 1.f : 0.f, (nib & 2u) ? 1.f : 0.f, (nib & 4u) ? 1.f : 0.f, (nib & 8u) ? 1.f : 0.f);
              }
            }
          }
        };
        auto pack_mask = [](const float4* mk) {
          uint32_t b = 0;
#pragma unroll
          for (int i = 0; i < 4; ++i)
            b |= ((mk[i].x > 0.f ? 1u : 0u) | (mk[i].y > 0.f ? 2u : 0u) | (mk[i].z > 0.f ? 4u : 0u) |
                  (mk[i].w > 0.f ? 8u : 0u)) << (4 * i);
          return b;
        };
        uint32_t mbits = 0xFFFFu;
        if (MASK) {
          float4 mk[4];
          load_mask(half * EPC, mk);
          mbits = pack_mask(mk);
        }
        // MASK instantiations keep one residual buffer (register budget)
        constexpr bool DB = !MASK;
        float4 rr[4], rn[4];
        if (DB) load_res(half * EPC, rr);          // independent of the accumulator: issued before the wait
        if (mode != 2) {
          mbar_wait(tfull0 + 8 * acc, (tile_iter >> 1) & 1);
          tc_fence_after();
          if (ew == 0 && lane == 0 && tile_iter < 4) TR(24 + 4 * tile_iter);
        }
        for (int c0 = half * EPC; c0 < bn; c0 += 2 * EPC) {
          if (ti.n0 + c0 >= p.N) break;            // warp-uniform
          if (DB) load_res(c0 + 2 * EPC, rn);
          else load_res(c0, rr);                   // L2-resident (tile-ahead prefetch); overlaps the TMEM load
          if (mode != 2) {
            float v[EPC];
            tmem_ld16(lane_addr + c0, v);
            tmem_ld_wait();
#pragma unroll
            for (int q = 0; q < EPC / 4; ++q)
              *reinterpret_cast<float4*>(stg + lane * EPITCH + q * 4) =
                  make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
            __syncwarp();
          }
          float4 mk[4];
          if (MASK) load_mask(c0 + 2 * EPC, mk);
          const int n = ti.n0 + c0 + col;
          const bool nfull = n + 3 < p.N;
          const int cvi = ((c0 - half * EPC) >> 1) + col;
          const float4 cs = *reinterpret_cast<const float4*>(wsc + cvi);
          float4 cb = *reinterpret_cast<const float4*>(wbi + cvi);
          if (mode == 0 && ti.k_begin != 0) cb = make_float4(0.f, 0.f, 0.f, 0.f);      // split-K: bias from the first K slice only
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int row = (lane >> 2) + 8 * i;
            const int m = ti.m0 + quarter * 32 + row;
            float4 a4;
            if (mode == 2) {
              const size_t wso = (size_t)(quarter * 32 + row) * bn + c0 + col;
              a4 = make_float4(0.f, 0.f, 0.f, 0.f);
              for (int j = 0; j < ti.npieces(); ++j) {
                const int sl = (j == 0) ? ti.first_slot() : 0;
                const float4 w4 = ld_cg_f4(L.ws_tiles + ((size_t)((ti.ufirst() + j) * 2 + sl) * nrank + rank) * ws_tile_floats + wso);
                a4.x += w4.x; a4.y += w4.y; a4.z += w4.z; a4.w += w4.w;
              }
            } else {
              a4 = *reinterpret_cast<const float4*>(stg + row * EPITCH + col);
            }
            if (mode == 1) {
              float* const ws_mine = L.ws_tiles + ((size_t)(unit * 2 + ti.slot()) * nrank + rank) * ws_tile_floats;
              *reinterpret_cast<float4*>(ws_mine + (size_t)(quarter * 32 + row) * bn + c0 + col) = a4;
              continue;
            }
            if (m >= p.M || n >= p.N) continue;
            if (nfull && vec_ok) {
              float4 o = make_float4(a4.x * p.alpha, a4.y * p.alpha, a4.z * p.alpha, a4.w * p.alpha);
              o.x = (o.x * cs.x + cb.x) * rs[i]; o.y = (o.y * cs.y + cb.y) * rs[i];
              o.z = (o.z * cs.z + cb.z) * rs[i]; o.w = (o.w * cs.w + cb.w) * rs[i];
              const int64_t off = tile_off + (int64_t)m * p.ldd + n;
              if (want_res) { o.x += rr[i].x; o.y += rr[i].y; o.z += rr[i].z; o.w += rr[i].w; }   // residual or D (ACCUM)
              if (p.flags & VLFB_EPI_RELU) {
                o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f);
              }
              if (MASK) {
                const uint32_t mb = mbits >> (4 * i);
                o.x = (mb & 1u) ? o.x : 0.f; o.y = (mb & 2u) ? o.y : 0.f;
                o.z = (mb & 4u) ? o.z : 0.f; o.w = (mb & 8u) ? o.w : 0.f;
              }
              if (p.flags & VLFB_EPI_TF32) {
                o.x = round_tf32(o.x); o.y = round_tf32(o.y); o.z = round_tf32(o.z); o.w = round_tf32(o.w);
              }
              float* dst = p.d + off;
              if (p.flags & VLFB_EPI_ATOMIC) {
                atomicAdd(dst, o.x); atomicAdd(dst + 1, o.y); atomicAdd(dst + 2, o.z); atomicAdd(dst + 3, o.w);
              } else {
                *reinterpret_cast<float4*>(dst) = o;
              }
            } else {
              const float e4[4] = {a4.x, a4.y, a4.z, a4.w};
#pragma unroll
              for (int e = 0; e < 4; ++e)
                if (n + e < p.N) epilogue_store(p, ti.batch, ti.tap, m, n + e, e4[e], mode != 0 || ti.k_begin == 0);
            }
          }
          __syncwarp();
          if (MASK) mbits = pack_mask(mk);
          if (DB) {
#pragma unroll
            for (int i = 0; i < 4; ++i) rr[i] = rn[i];
          }
        }
      };
      // The same pass, lean: for tiles whose rows are 16-byte addressable and whose N extent is a whole number of
      // 16-column blocks (every layer of the networks).  run_blocks spends ~830 instructions per 32 x 16 block
      // (ncu r2b: per-float4 flag tests, 64-bit address arithmetic and bounds checks) -- 6.3 us for a 128 x 256 tile,
      // longer than the K loop of most res2 / res3 / res4 layers; here every run-time switch is tested once per tile
      // (warp-uniform), rows are four precomputed pointers and the column offset is one add per block.
      auto run_fast = [&](auto mode_c, auto atomic_c, auto wres_c, auto bits_c) {
        constexpr int mode = decltype(mode_c)::value;
        constexpr bool ATOMIC = decltype(atomic_c)::value && mode != 1;
        constexpr bool WRES = decltype(wres_c)::value && mode != 1;
        constexpr bool BITS = decltype(bits_c)::value && mode != 1 && !ATOMIC;      // emit the ReLU sign bits of the result
        const int r0 = quarter * 32 + (lane >> 2);                         // tile rows r0 + 8 i of this lane
        const int cbase = half * EPC + col;
        const bool patch = !PAIR && AK == VLFB_OP_STEM_K && L.stem_patch != 0;
        const int mrows = par ? L.par_m : p.M;
        uint32_t rowok = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) rowok |= (patch || ti.m0 + r0 + 8 * i < mrows) ? (1u << i) : 0u;
        const int ncols = min(bn, p.N - ti.n0);                            // multiple of 16
        // ONE 32-bit element offset per row, shared by every stream (D, residual, sign bits: same addressing), advanced by
        // one block (32 columns) per step; 64-bit row pointers per stream cost 24 registers, which the look-ahead
        // buffers need (the host / fast_tile test guarantees offsets < 2^32)
        uint32_t eo[4];
        float* wsp = nullptr;                  // mode 1: this unit's workspace slot (rows 8 bn apart)
        unsigned short* bout = nullptr;        // relu_bits_out group of tile row r0 + 8 (lane & 3) (this lane stores that row's)
        constexpr bool emit_bits = BITS;
        if (mode == 1)
          wsp = L.ws_tiles + ((size_t)(unit * 2 + ti.slot()) * nrank + rank) * ws_tile_floats + (size_t)r0 * bn + cbase;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          int64_t row = ti.m0 + r0 + 8 * i;
          if (patch) row = patch_row(p, L, ti.m0 / BM, r0 + 8 * i);      // conv1 patch tile: row -> (ho, wo) of the patch
          if (par && ((rowok >> i) & 1u)) row = par_row(p, L, ti.batch, ti.m0 + r0 + 8 * i);   // parity class: sub-grid row -> dX row
          eo[i] = (uint32_t)(tile_off + row * p.ldd + ti.n0 + cbase);
        }
        if (emit_bits) {
          const int rb = r0 + 8 * (lane & 3);
          int64_t row = ti.m0 + rb;
          if (patch) row = patch_row(p, L, ti.m0 / BM, rb);
          bout = reinterpret_cast<unsigned short*>(p.relu_bits_out) + ((tile_off + row * p.ldd + ti.n0 + half * EPC) >> 4);
        }
        const unsigned short* mbase = reinterpret_cast<const unsigned short*>(p.relu_mask_bits);
        const bool relu = (p.flags & VLFB_EPI_RELU) != 0, tf32 = (p.flags & VLFB_EPI_TF32) != 0;
        const bool has_rs = p.row_scale != nullptr;
        const bool nobias = mode == 0 && ti.k_begin != 0;                  // split-K: bias from the first K slice only
        const float alpha = p.alpha;
        // residual / accumulate / mask operands of the block `ahead` blocks after the current one.  ReLU-backward mask
        // (MASK builds): the sign bits of the activation that gates this gradient, one 16-bit group per row and block.
        auto load_ahead = [&](bool valid, int ahead, float4* r, uint32_t* m) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const uint32_t e = eo[i] + (uint32_t)(ahead * 2 * EPC);
            if (WRES) {
              r[i] = make_float4(0.f, 0.f, 0.f, 0.f);
              if (valid && ((rowok >> i) & 1u)) r[i] = ld_nc_f4(res_src + e);
            }
            if (MASK && mode != 1) {
              m[i] = 0xFFFFu;
              if (valid && ((rowok >> i) & 1u)) m[i] = ld_nc_u16(mbase + ((e - (uint32_t)col) >> 4));
            }
          }
        };
        // Residual / mask operands are fetched VLFB_EPI_DEPTH blocks ahead into a ring of register buffers; the loop is
        // unrolled over the ring so that no buffer is ever copied (a `cur = next` move at the end of an iteration waits
        // for the load it copies: the first version's look-ahead was worth less than one block, call G).
        constexpr int NBUF = VLFB_EPI_DEPTH + 1;
        float4 rbuf[NBUF][4];
        uint32_t mbuf[NBUF][4];
        load_ahead(half * EPC < ncols, 0, rbuf[0], mbuf[0]);
        if (NBUF == 3) load_ahead(half * EPC + 2 * EPC < ncols, 1, rbuf[1], mbuf[1]);
        if (mode != 2) {
          mbar_wait(tfull0 + 8 * acc, (tile_iter >> 1) & 1);
          tc_fence_after();
          if (ew == 0 && lane == 0 && tile_iter < 4) TR(24 + 4 * tile_iter);
        }
        // one 32 x 16 block: operands of block c0 in (rc, mc); the block VLFB_EPI_DEPTH ahead is fetched into (rl, ml)
        auto step = [&](int c0, int cofs, const float4* rc, const uint32_t* mc, float4* rl, uint32_t* ml) {
          load_ahead(c0 + 2 * EPC * VLFB_EPI_DEPTH < ncols, VLFB_EPI_DEPTH, rl, ml);
          float4 a4[4];
          uint32_t obits = 0;
          if (mode != 2) {
            float v[EPC];
            tmem_ld16(lane_addr + c0, v);
            tmem_ld_wait();
#pragma unroll
            for (int q = 0; q < EPC / 4; ++q)
              *reinterpret_cast<float4*>(stg + lane * EPITCH + q * 4) =
                  make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
            __syncwarp();
#pragma unroll
            for (int i = 0; i < 4; ++i)
              a4[i] = *reinterpret_cast<const float4*>(stg + ((lane >> 2) + 8 * i) * EPITCH + col);
            __syncwarp();
            if (par && ti.nk == 0) {                                        // class without taps: dX = finish(0)
#pragma unroll
              for (int i = 0; i < 4; ++i) a4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) a4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int j = 0; j < ti.npieces(); ++j) {                        // piece order: deterministic sum
              const int sl = (j == 0) ? ti.first_slot() : 0;
              const float* w = L.ws_tiles + ((size_t)((ti.ufirst() + j) * 2 + sl) * nrank + rank) * ws_tile_floats +
                               (size_t)r0 * bn + cbase + cofs;
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float4 w4 = ld_cg_f4(w + (size_t)i * 8 * bn);
                a4[i].x += w4.x; a4[i].y += w4.y; a4[i].z += w4.z; a4[i].w += w4.w;
              }
            }
          }
          if (mode == 1) {
#pragma unroll
            for (int i = 0; i < 4; ++i) *reinterpret_cast<float4*>(wsp + (size_t)i * 8 * bn) = a4[i];
            wsp += 2 * EPC;
            return;
          }
          const int cvi = ((c0 - half * EPC) >> 1) + col;
          float4 cs = *reinterpret_cast<const float4*>(wsc + cvi);
          float4 cb = *reinterpret_cast<const float4*>(wbi + cvi);
          cs.x *= alpha; cs.y *= alpha; cs.z *= alpha; cs.w *= alpha;
          if (nobias) cb = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            float4 o;
            o.x = fmaf(a4[i].x, cs.x, cb.x); o.y = fmaf(a4[i].y, cs.y, cb.y);
            o.z = fmaf(a4[i].z, cs.z, cb.z); o.w = fmaf(a4[i].w, cs.w, cb.w);
            if (has_rs) { o.x *= rs[i]; o.y *= rs[i]; o.z *= rs[i]; o.w *= rs[i]; }
            if (WRES) { o.x += rc[i].x; o.y += rc[i].y; o.z += rc[i].z; o.w += rc[i].w; }
            if (relu) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
            if (MASK) {
              const uint32_t nib = mc[i] >> ((lane & 3) * 4);
              o.x = (nib & 1u) ? o.x : 0.f; o.y = (nib & 2u) ? o.y : 0.f;
              o.z = (nib & 4u) ? o.z : 0.f; o.w = (nib & 8u) ? o.w : 0.f;
            }
            if (tf32) { o.x = round_tf32(o.x); o.y = round_tf32(o.y); o.z = round_tf32(o.z); o.w = round_tf32(o.w); }
            if ((rowok >> i) & 1u) {
              if (ATOMIC) red_add_f4(p.d + eo[i], o);
              else *reinterpret_cast<float4*>(p.d + eo[i]) = o;
            }
            eo[i] += 2 * EPC;
            if (emit_bits) {             // the row's 16 sign bits: 4 lanes x 4 columns (warp-uniform branch)
              uint32_t nb = (o.x > 0.f ? 1u : 0u) | (o.y > 0.f ? 2u : 0u) | (o.z > 0.f ? 4u : 0u) | (o.w > 0.f ? 8u : 0u);
              nb <<= (lane & 3) * 4;
              nb |= __shfl_xor_sync(0xffffffffu, nb, 1);
              nb |= __shfl_xor_sync(0xffffffffu, nb, 2);
              if ((lane & 3) == i) obits = nb;
            }
          }
          if (emit_bits) {
            if ((rowok >> (lane & 3)) & 1u) *bout = (unsigned short)obits;
            bout += 2 * EPC / 16;
          }
        };
        {
          int c0 = half * EPC, cofs = 0;                                    // cofs: column offset of the block from cbase (mode 2)
          while (c0 < ncols) {
#pragma unroll
            for (int b = 0; b < NBUF; ++b) {
              if (c0 < ncols) step(c0, cofs, rbuf[b], mbuf[b], rbuf[(b + NBUF - 1) % NBUF], mbuf[(b + NBUF - 1) % NBUF]);
              c0 += 2 * EPC; cofs += 2 * EPC;
            }
          }
        }
      };
      // run-time epilogue flavour -> compile-time flags (atomic accumulate; residual / D-accumulate stream)
      auto call_fast = [&](auto mode_c) {
        using T = std::true_type;
        using F = std::false_type;
        const bool atomic = (p.flags & VLFB_EPI_ATOMIC) != 0;
        if (decltype(mode_c)::value == 1) run_fast(mode_c, F{}, F{}, F{});
        else if (atomic) { if (want_res) run_fast(mode_c, T{}, T{}, F{}); else run_fast(mode_c, T{}, F{}, F{}); }
        else if (!MASK && p.relu_bits_out != nullptr) { if (want_res) run_fast(mode_c, F{}, T{}, T{}); else run_fast(mode_c, F{}, F{}, T{}); }
        else { if (want_res) run_fast(mode_c, F{}, T{}, F{}); else run_fast(mode_c, F{}, F{}, F{}); }
      };
      // (the 17-warp cp.async builds never take the fix-up path: the host plans stream-K fix-ups for TMA-fed launches only)
      const bool split_tile = !CP && ti.npieces() > 1;
      // (MASK builds: the lean path reads the mask as sign bits; a float mask takes the general path)
      const bool bits_ok = (p.ldd & 15) == 0 && (p.d_batch_stride & 15) == 0 && (p.d_tap_stride & 15) == 0;
      const bool fast_tile = !CP && vec_ok && (p.N & 15) == 0 && span32_ok(p) && !(MASK && (p.relu_mask != nullptr || !bits_ok));
      if constexpr (!CP) {
        if (fast_tile) {
          if (split_tile) call_fast(std::integral_constant<int, 1>{});
          else call_fast(std::integral_constant<int, 0>{});
        } else {
          if (split_tile) run_blocks(std::integral_constant<int, 1>{});
          else run_blocks(std::integral_constant<int, 0>{});
        }
      } else {
        run_blocks(std::integral_constant<int, 0>{});
      }
      if (ew == 0 && lane == 0 && tile_iter < 4) TR(25 + 4 * tile_iter);
      // every TMEM read of this accumulator has completed (tcgen05.wait::ld above): hand it back to the MMA warp
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR && rank != 0) mbar_arrive_cluster(tempty_x + 8 * acc);
        else mbar_arrive(tempty0 + 8 * acc);
      }
      ++tile_iter;
      if constexpr (!CP) if (split_tile) {
        // publish this piece, count it; the warp that arrives last owns the reduction of its sub-blocks
        __threadfence();
        __syncwarp();
        int* cnt = L.ws_cnt + ((size_t)ti.tile * nrank + rank) * (NEPI / 32) + ew;
        int old = 0;
        if (lane == 0) old = atomicAdd(cnt, 1);
        old = __shfl_sync(0xffffffffu, old, 0);
        if (ew == 0 && lane == 0 && tile_iter <= 4) TR(26 + 4 * (tile_iter - 1));
        if (old == ti.npieces() - 1) {
          __threadfence();
          if (fast_tile) call_fast(std::integral_constant<int, 2>{});
          else run_blocks(std::integral_constant<int, 2>{});
          if (lane == 0) *cnt = 0;                 // counters are zero again when the launch ends
          if (ew == 0 && lane == 0 && tile_iter <= 4) TR(27 + 4 * (tile_iter - 1));
        }
      }
    }
  }
  if (tid == 0) TR(3);
  tc_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();       // PAIR: no CTA exits (or frees TMEM) while its peer can still signal it
  if (warp == NPWT) {
    tc_fence_after();
    if (PAIR) tmem_dealloc2(tmem, tmem_cols); else tmem_dealloc(tmem, tmem_cols);
  }
}

// ---------------------------------------------------------------- host dispatch
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
    const char* e = getenv("VLFB_TMA");
    if (e && atoi(e) == 0) fn = nullptr;
  }
  return fn;
}

// 3-D tensor map {K, rows, batch} of a dense K-major fp32 matrix; box = {32 floats (one 128-byte swizzle
// row), box_rows, 1}; out-of-range rows / K tail read as zeros.
static bool make_tmap(CUtensorMap* tm, const vlfb_operand_t& op, int rows, int K, int batch, int box_rows) {
  EncodeTiledFn enc = encode_fn();
  if (!enc || op.kind != VLFB_OP_DENSE_K || K < KC || rows < box_rows) return false;
  cuuint64_t dims[3] = {(cuuint64_t)K, (cuuint64_t)rows, (cuuint64_t)(batch > 1 ? batch : 1)};
  cuuint64_t strides[2] = {(cuuint64_t)op.ld * 4,
                           (cuuint64_t)(batch > 1 ? op.batch_stride : (int64_t)rows * op.ld) * 4};
  if ((strides[0] & 15) || (strides[1] & 15) || strides[1] == 0) return false;
  cuuint32_t box[3] = {(cuuint32_t)KC, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(op.ptr), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Dense MN-major fp32 matrix [K rows][extent] (+batch): box = {32 elements, 32 k-rows, 1} written in the
// SWIZZLE_128B_ATOM_32B pattern = one UMMA MN-major atom column (4 KB) per copy.
static bool make_tmap_mn(CUtensorMap* tm, const vlfb_operand_t& op, int extent, int K, int batch) {
  EncodeTiledFn enc = encode_fn();
  if (!enc || op.kind != VLFB_OP_DENSE_MN || K < KC || extent < 32) return false;
  cuuint64_t dims[3] = {(cuuint64_t)extent, (cuuint64_t)K, (cuuint64_t)(batch > 1 ? batch : 1)};
  cuuint64_t strides[2] = {(cuuint64_t)op.ld * 4, (cuuint64_t)(batch > 1 ? op.batch_stride : (int64_t)K * op.ld) * 4};
  if ((strides[0] & 15) || (strides[1] & 15) || strides[1] == 0) return false;
  cuuint32_t box[3] = {32, (cuuint32_t)KC, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(op.ptr), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// The same operand as ONE box per tile: a 4-D view {32 elements of an atom, K rows, atom index, batch} -- the atom
// dimension has the SMALLEST stride (128 B), which a tiled map may have -- with box {32, 32 k-rows, natoms, 1}: the copy
// writes atom after atom, i.e. exactly the [atom][k][32] layout the per-atom copies produce, in one instruction instead
// of 4 (A) / 8 (B).  The TMA unit's cost is per BOX: the 12 small boxes of a wgrad K chunk took 0.72 us against 0.27 us
// of MMAs (tensor pipe 33-37 % active in every wgrad launch, ncu call M).  Needs whole atoms (extent % 32 == 0).
static bool make_tmap_mn4(CUtensorMap* tm, const vlfb_operand_t& op, int extent, int K, int batch, int natoms) {
  EncodeTiledFn enc = encode_fn();
  if (!enc || op.kind != VLFB_OP_DENSE_MN || K < KC || extent < 32 || (extent & 31) || natoms < 1 || natoms > 8) return false;
  cuuint64_t dims[4] = {32, (cuuint64_t)K, (cuuint64_t)(extent / 32), (cuuint64_t)(batch > 1 ? batch : 1)};
  cuuint64_t strides[3] = {(cuuint64_t)op.ld * 4, 128, (cuuint64_t)(batch > 1 ? op.batch_stride : (int64_t)K * op.ld) * 4};
  if ((strides[0] & 15) || (strides[2] & 15) || strides[2] == 0) return false;
  cuuint32_t box[4] = {32, (cuuint32_t)KC, (cuuint32_t)natoms, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(op.ptr), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// wgrad activation operand of a convolution WITHOUT spatial taps (1x1x1 and kTx1x1, unit strides, no spatial padding --
// two thirds of the convolutions of the nets): the k rows of a chunk are 32 consecutive positions of one clip, shifted by
// whole frames for the temporal tap, so the gather is a dense 4-D view {32 channels of an atom, T*H*W positions of a
// clip, atom index, clip}; frames outside the clip are out of range in the position dimension and read as zeros.
// ONE box per K chunk instead of up to 8 im2col copies.  Needs T*H*W % 32 == 0 (a chunk never straddles two clips).
static bool make_tmap_conv_flat(CUtensorMap* tm, const float* x, const vlfb_conv_geom_t& g, int natoms) {
  EncodeTiledFn enc = encode_fn();
  const int64_t thw = (int64_t)g.T * g.H * g.W;
  if (!enc || g.kH != 1 || g.kW != 1 || g.sT != 1 || g.sH != 1 || g.sW != 1 || g.pH != 0 || g.pW != 0) return false;
  if ((g.C & 31) || (thw & 31) || g.To != g.T || g.Ho != g.H || g.Wo != g.W || natoms < 1 || natoms > 8) return false;
  cuuint64_t dims[4] = {32, (cuuint64_t)thw, (cuuint64_t)(g.C / 32), (cuuint64_t)g.N};
  cuuint64_t strides[3] = {(cuuint64_t)g.C * 4, 128, (cuuint64_t)thw * g.C * 4};
  cuuint32_t box[4] = {32, (cuuint32_t)KC, (cuuint32_t)natoms, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(x), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// 5-D im2col map of an NDHWC fp32 tensor [N, D, H, W, C]: `pixels` window origins x 32 channels per copy.
// lower/upper = bounding-box corners {W, H, D}; strides = traversal strides {W, H, D}.
typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*,
                                   CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                   CUtensorMapFloatOOBfill);
static bool make_tmap_im2col(CUtensorMap* tm, const float* base, int N, int D, int H, int W, int C, const int lower[3],
                             const int upper[3], const int strides[3], int pixels, CUtensorMapSwizzle swz,
                             int chan = KC) {
  static EncodeIm2colFn enc = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (encode_fn() && cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      enc = reinterpret_cast<EncodeIm2colFn>(ptr);
  }
  if (!enc || (C % chan) != 0 || (reinterpret_cast<uintptr_t>(base) & 15)) return false;
  for (int i = 0; i < 3; ++i)
    if (lower[i] < -16 || lower[i] > 15 || upper[i] < -16 || upper[i] > 15 || strides[i] < 1 || strides[i] > 8) return false;
  cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)N};
  cuuint64_t gstr[4] = {(cuuint64_t)C * 4, (cuuint64_t)C * 4 * W, (cuuint64_t)C * 4 * W * H, (cuuint64_t)C * 4 * W * H * D};
  cuuint32_t estr[5] = {1, (cuuint32_t)strides[0], (cuuint32_t)strides[1], (cuuint32_t)strides[2], 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<float*>(base), dims, gstr, lower, upper,
             (cuuint32_t)chan, (cuuint32_t)pixels, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// conv1 stem (C padded to 4, 16-byte pixels): overlapping-window view of a clip whose rows are stored with `pitch`
// >= pW + W + right pad pixels, the pad pixels zero.  dim0 = the 8 px x 4 ch = 32 floats of one filter row starting
// at padded pixel wo * sW (i.e. real pixel wo * sW - pW), dim1 = wo (stride sW pixels: consecutive windows OVERLAP),
// dim2 / dim3 = input row / frame (their out-of-range coordinates read as zeros = the H / T padding), dim4 = clip.
// One box = 16 consecutive output positions of one output row.
static bool make_tmap_stem(CUtensorMap* tm, const float* ptr, const vlfb_conv_geom_t& g, int64_t pitch, CUtensorMapSwizzle swz,
                           int box_rows = 1) {
  EncodeTiledFn enc = encode_fn();
  if (!enc || g.C != 4 || (g.Wo & 15) || g.dT != 1 || g.dH != 1 || g.dW != 1 || g.kW > 8) return false;
  if (pitch < g.pW + g.W || pitch < (int64_t)(g.Wo - 1) * g.sW + 8 || (reinterpret_cast<uintptr_t>(ptr) & 15)) return false;
  const float* base = ptr - (int64_t)g.pW * 4;                     // padded pixel 0 of row 0
  cuuint64_t dims[5] = {32, (cuuint64_t)g.Wo, (cuuint64_t)g.H, (cuuint64_t)g.T, (cuuint64_t)g.N};
  cuuint64_t gstr[4] = {(cuuint64_t)g.sW * 16, (cuuint64_t)pitch * 16, (cuuint64_t)pitch * 16 * g.H,
                        (cuuint64_t)pitch * 16 * g.H * g.T};
  // box_rows > 1: that many input rows `sH` apart (= consecutive OUTPUT rows) in one box: boxDim = rows * stride with
  // elementStride = stride loads ceil(boxDim / stride) = rows elements (cuTensorMapEncodeTiled)
  // box_rows < 0: -box_rows CONSECUTIVE input rows (conv1 wgrad: the sH + kH rows two output rows' filter windows span)
  cuuint32_t box[5] = {32, 16, (cuuint32_t)(box_rows > 1 ? box_rows * g.sH : (box_rows < 0 ? -box_rows : 1)), 1, 1};
  cuuint32_t estr[5] = {1, 1, (cuuint32_t)(box_rows > 1 ? g.sH : 1), 1, 1};
  if (box[2] > 256 || estr[2] > 8) return false;
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 5, const_cast<float*>(base), dims, gstr, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// conv1 wgrad A operand in patch order: dY [N*To][Ho][Wo][Co] as a 4-D map; box {32 channels, 16 wo, 2 ho} = the 32 k-rows
// of a patch chunk for one 32-channel atom, in the MN-major atom layout (SWIZZLE_128B_ATOM_32B).
static bool make_tmap_dy4(CUtensorMap* tm, const float* dy, const vlfb_conv_geom_t& g) {
  EncodeTiledFn enc = encode_fn();
  if (!enc || (g.Co & 3) || (reinterpret_cast<uintptr_t>(dy) & 15)) return false;
  cuuint64_t dims[4] = {(cuuint64_t)g.Co, (cuuint64_t)g.Wo, (cuuint64_t)g.Ho, (cuuint64_t)g.N * g.To};
  cuuint64_t gstr[3] = {(cuuint64_t)g.Co * 4, (cuuint64_t)g.Co * 4 * g.Wo, (cuuint64_t)g.Co * 4 * g.Wo * g.Ho};
  cuuint32_t box[4] = {32, 16, 2, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(dy), dims, gstr, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// tuning overrides, read once (scripts/tune_gemm.py); the per-call fields of vlfb_gemm_params_t take precedence
struct Env { int bn, stages, lag, pair, sk, debug, no_patch, no_par; bool tma_mn, im2col, fuse_atoms; };
static Env read_env() {
  Env e;
  auto geti = [](const char* name, int dflt) { const char* v = getenv(name); return v ? atoi(v) : dflt; };
  e.bn = geti("VLFB_BN", 0);
  e.stages = geti("VLFB_STAGES", 0);
  e.lag = geti("VLFB_LAG", 0);
  e.pair = geti("VLFB_PAIR", 0);
  e.sk = geti("VLFB_SK", 0);
  e.debug = geti("VLFB_DEBUG", 0);
  e.no_patch = geti("VLFB_NO_PATCH", 0);
  e.no_par = geti("VLFB_NO_PAR", 0);
  e.tma_mn = geti("VLFB_TMA_MN", 1) != 0;
  e.im2col = geti("VLFB_IM2COL", 1) != 0;
  e.fuse_atoms = geti("VLFB_FUSE_ATOMS", 1) != 0;
  return e;
}
static const Env& env() {
  static const Env e = read_env();
  return e;
}

// ---- plan: tile width x CTA pairing x schedule, chosen together by a cycle model of one SM -----------------
// A K chunk (32 fp32 of K) of a 128 x bn tile costs max(tensor pipe, operand delivery):
//   tensor   = 4 MMAs x (128 x bn x 8 MACs) / 2048 MAC/clk = 2 bn clocks (kind::tf32 issues at half the bf16 rate);
//   delivery = (128 + bn) x 128 B, or (128 + bn/2) x 128 B for a CTA pair, at ~58 B/clk through the SM's
//              L2 port (ncu r01: 694 MB -> 98 SMs in 70.9 us on res5 branch2b).
// A tile adds a fixed fill + epilogue cost (~8 chunks' worth); a stream-K launch adds the fix-up of the shared tiles.
static double chunk_cost(int bn, bool pair) {
  const double tensor = 2.0 * bn;
  const double port = (16384.0 + (pair ? 64.0 : 128.0) * bn) / 58.0;
  return tensor > port ? tensor : port;
}

struct Plan { int bn, split_k, pair, sk; int tiles, units; double cost; };

static constexpr bool kind_pair_capable(int kind) { return kind != VLFB_OP_STEM_K && kind != VLFB_OP_STEM_MN; }
static constexpr bool kind_tma_capable(int) { return true; }

size_t gemm_tc_workspace_bytes();

// An accumulating (atomic) product whose split the library chooses is not split into K slices that add into D in
// arrival order when the caller provides a workspace and allows stream-K: the run-to-run result would depend on that
// order.  It runs as whole tiles or as stream-K pieces summed from the workspace in a fixed order by the last arriving
// unit, which then adds the tile to D once.  Otherwise plain split-K (atomic, order-dependent) stays available.
static bool det_split_of(const vlfb_gemm_params_t& p) {
  const int want_sk = p.stream_k != 0 ? p.stream_k : env().sk;
  return (p.flags & VLFB_EPI_ATOMIC) && p.split_k == 0 && want_sk >= 0 && p.workspace != nullptr &&
         p.workspace_bytes >= gemm_tc_workspace_bytes();
}

// `pairs` = co-resident CTA pairs (0: pairing unavailable); pair_ok / sk_ok = what the operands / workspace allow.
static Plan make_plan(const vlfb_gemm_params_t& p, int num_sms, int pairs, bool pair_ok, bool sk_ok) {
  const int zbase = p.taps > 1 ? p.taps : p.batch;
  const bool atomic = (p.flags & VLFB_EPI_ATOMIC) != 0;
  const bool det_split = det_split_of(p);
  const int want_bn = p.tile_n > 0 ? p.tile_n : env().bn;
  const int want_pair = p.pair != 0 ? p.pair : env().pair;
  const int want_sk = p.stream_k != 0 ? p.stream_k : env().sk;
  Plan best, best_sk;
  best.cost = 1e30; best.bn = 32; best.split_k = p.split_k > 0 ? p.split_k : 1; best.pair = 0; best.sk = 0;
  best.tiles = 0; best.units = 0;
  best_sk = best;
  static const int kWidths[] = {256, 192, 128, 96, 64, 32};
  for (int pr = 0; pr < 2; ++pr) {
    // CTA pairs and stream-K are opt-in (p.pair / p.stream_k = 1, VLFB_PAIR / VLFB_SK): measured on B200 (profiles/
    // r02_gemm_variants.txt, r02_trace_*.txt) the K loop of a 128 x 256 tf32 tile already runs at the tensor-pipe
    // rate (0.287 us per 32-deep chunk = 4 x 128-cycle MMAs), so halving the operand bytes per SM buys nothing, and
    // the stream-K fix-up costs more than the idle SMs of a 98-tile launch.
    const bool can_pair = pair_ok && pairs >= 1 && p.M > BM;
    if (pr == 1 && (!can_pair || want_pair <= 0)) continue;
    if (pr == 0 && want_pair > 0 && can_pair) continue;
    const int U = pr ? pairs : num_sms;
    for (int wi = 0; wi < 6; ++wi) {
      const int bn = kWidths[wi];
      if (want_bn > 0 ? bn != want_bn : ((bn & (bn - 1)) != 0)) continue;       // 96 / 192 only on request
      if (pr && (bn & 63)) continue;                                            // each CTA of a pair stages whole 32-column atoms
      if (want_bn <= 0 && bn > 32 && p.N <= bn / 2) continue;                   // do not pad N by 2x
      const int tiles_m = ceil_div(p.M, pr ? 2 * BM : BM);
      const int64_t T = (int64_t)tiles_m * ceil_div(p.N, bn) * zbase;
      const int nkt = ceil_div(p.K, KC);
      const double cc = chunk_cost(bn, pr != 0);
      const double fixed = 8.0 * cc;
      // (a) static tile loop, optional plain split-K (atomic epilogues only)
      const int smax = p.split_k > 0 ? p.split_k : (atomic && !det_split && p.K >= 512 ? (p.K / 256 < 128 ? p.K / 256 : 128) : 1);
      for (int sp = (p.split_k > 0 ? p.split_k : 1); sp <= smax; ++sp) {
        const int64_t tiles = T * sp;
        const double rounds = (double)((tiles + U - 1) / U);
        const double cost = rounds * (ceil_div(ceil_div(p.K, sp), KC) * cc + fixed);
        if (cost < best.cost * 0.999) {
          best.cost = cost; best.bn = bn; best.split_k = sp; best.pair = pr; best.sk = 0;
          best.tiles = (int)tiles; best.units = (int)(tiles < U ? tiles : U);
        }
      }
      // (b) stream-K: equal chunk ranges; shared tiles reduced through the workspace (or by atomics)
      const int64_t total = T * nkt;
      const bool fixup = sk_ok && (!atomic || det_split);
      const bool sk_legal = (det_split ? sk_ok : ((atomic ? p.split_k != 1 : (sk_ok && p.split_k <= 1)) && want_sk > 0)) &&
                            nkt >= 2 && total >= 2 * (int64_t)U && T * (pr ? 2 : 1) * (NEPI / 32) <= SK_CNT_INTS &&
                            U <= MAX_UNITS;
      if (sk_legal && (T % U) != 0) {
        const double per_unit = (double)((total + U - 1) / U);
        const double cost = per_unit * cc + fixed * (double)((T + U - 1) / U) + (fixup ? 2.0 : 1.0) * fixed;
        if (cost < best_sk.cost * 0.999) {
          best_sk.cost = cost; best_sk.bn = bn; best_sk.split_k = 1; best_sk.pair = pr; best_sk.sk = 1;
          best_sk.tiles = (int)T; best_sk.units = U;
        }
      }
    }
  }
  if (best_sk.cost < 1e29 && (want_sk > 0 || best_sk.cost < best.cost * 0.999)) return best_sk;
  return best;
}

// Chunk ranges of the stream-K units.  A boundary that would leave a piece of fewer than `minp` chunks at either end
// of a tile is moved onto the tile boundary.
static void make_bounds(int* b, int U, int64_t T, int nkt) {
  const int64_t total = T * nkt;
  const int minp = nkt >= 16 ? 4 : (nkt >= 8 ? 2 : 1);
  for (int u = 0; u <= U; ++u) {
    int64_t x = (int64_t)u * total / U;
    const int r = (int)(x % nkt);
    if (r && r < minp) x -= r;
    else if (r && nkt - r < minp) x += nkt - r;
    b[u] = (int)x;
  }
  b[0] = 0; b[U] = (int)total;
  bool ok = true;
  for (int u = 0; u < U; ++u) if (b[u + 1] <= b[u]) ok = false;
  if (!ok) for (int u = 0; u <= U; ++u) b[u] = (int)((int64_t)u * total / U);
}

size_t gemm_tc_workspace_bytes() {
  return (size_t)SK_CNT_INTS * 4 + (size_t)MAX_UNITS * 2 * BM * 256 * 4;
}

template <int AK, int BK, bool MASK>
static int max_pairs() {
  static int cached = -1;
  if constexpr (!(kind_pair_capable(AK) && kind_pair_capable(BK))) return 0;
  else if (cached < 0) {
    cached = 0;
    if (cudaFuncSetAttribute(gemm_tc_kernel<AK, BK, MASK, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             227 * 1024) == cudaSuccess) {
      cudaLaunchConfig_t cfg = {};
      cfg.gridDim = dim3(2 * MAX_UNITS);
      cfg.blockDim = dim3(32 + 32 + NEPI);
      cfg.dynamicSmemBytes = 200 * 1024;
      cudaLaunchAttribute attr[1];
      attr[0].id = cudaLaunchAttributeClusterDimension;
      attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
      cfg.attrs = attr;
      cfg.numAttrs = 1;
      int n = 0;
      if (cudaOccupancyMaxActiveClusters(&n, gemm_tc_kernel<AK, BK, MASK, true, false>, &cfg) == cudaSuccess && n > 0)
        cached = n < MAX_UNITS ? n : MAX_UNITS;
    }
    cudaGetLastError();
  }
  return cached;
}

template <int AK, int BK, bool MASK, bool PAIR, bool CP>
static int launch_variant(const cudaLaunchConfig_t& cfg, const vlfb_gemm_params_t& p, const Launch& L, const CUtensorMap& tmA,
                          const CUtensorMap& tmB) {
  static bool attr_done = false;
  cudaError_t e;
  if (!attr_done) {
    e = cudaFuncSetAttribute(gemm_tc_kernel<AK, BK, MASK, PAIR, CP>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) {
      set_error("cudaFuncSetAttribute(smem): %s", cudaGetErrorString(e));
      return VLFB_E_CUDA;
    }
    attr_done = true;
  }
  e = cudaLaunchKernelEx(&cfg, gemm_tc_kernel<AK, BK, MASK, PAIR, CP>, p, L, tmA, tmB);
  if (e != cudaSuccess) {
    set_error("gemm_tc launch: %s", cudaGetErrorString(e));
    return VLFB_E_CUDA;
  }
  VLFB_CHECK_LAUNCH();
  return VLFB_OK;
}

template <int AK, int BK, bool MASK>
int launch(const vlfb_gemm_params_t& p_in, cudaStream_t stream) {
  vlfb_gemm_params_t p = p_in;       // split_k == 0 is resolved below
  const bool det_split = det_split_of(p_in);
  Launch L;
  memset(&L, 0, sizeof(L));
  L.out.w = make_fastdiv(p.g.Wo);
  L.out.h = make_fastdiv(p.g.Ho);
  L.out.t = make_fastdiv(p.g.To);
  L.in.w = make_fastdiv(p.g.W);
  L.in.h = make_fastdiv(p.g.H);
  L.in.t = make_fastdiv(p.g.T);
  L.cdiv = make_fastdiv(p.g.C);
  L.kwdiv = make_fastdiv(p.g.kW);
  static int num_sms = 0;
  if (num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || num_sms <= 0) num_sms = 148;
    if (num_sms > MAX_UNITS) num_sms = MAX_UNITS;
  }
  const Env& ev = env();
  const vlfb_conv_geom_t& g = p.g;
  const bool unit_dgrad = g.sT == 1 && g.sH == 1 && g.sW == 1;
  // can both operands be staged by TMA (the precondition of CTA pairs)?  Decided on the cheap conditions here; the
  // tensor maps themselves are encoded after the plan (their boxes depend on it) and a failure falls back below.
  bool pair_ok = kind_pair_capable(AK) && kind_pair_capable(BK) && encode_fn() != nullptr && ev.im2col &&
                 (ev.tma_mn || !(is_mn(AK) || is_mn(BK))) && !(AK == VLFB_OP_DGRAD_K && !unit_dgrad) && p.K >= KC;
  bool sk_ws = p.workspace != nullptr && p.workspace_bytes >= gemm_tc_workspace_bytes() &&
                     (reinterpret_cast<uintptr_t>(p.workspace) & 15) == 0;
  alignas(64) CUtensorMap tmA, tmB;
  // Strided dgrad as parity classes (see Launch::par): needs whole strides in H / W, unit temporal stride and dilation,
  // both operands addressable by TMA, the lean epilogue (16-byte rows, whole 16-column blocks), and one im2col origin
  // offset shared by all classes that have taps (true for the networks' 3x3 / pad 1 and 1x1 / pad 0 stride-2 layers).
  int par_lo[3] = {0, 0, 0}, par_hi[3] = {0, 0, 0};
  if (AK == VLFB_OP_DGRAD_K && BK == VLFB_OP_DENSE_K && !unit_dgrad && !ev.no_par && ev.im2col && encode_fn() != nullptr &&
      g.sT == 1 && g.sH <= 2 && g.sW <= 2 && g.dT == 1 && g.dH == 1 && g.dW == 1 && (g.H % g.sH) == 0 && (g.W % g.sW) == 0 &&
      (g.Co % KC) == 0 && p.batch == 1 && p.taps <= 1 && p.split_k == 1 && !p.row_scale && !(p.flags & VLFB_EPI_ATOMIC) &&
      (p.N & 15) == 0 && (p.ldd & 3) == 0 && (reinterpret_cast<uintptr_t>(p.d) & 15) == 0 &&
      (!p.residual || ((reinterpret_cast<uintptr_t>(p.residual) & 15) == 0 && !(p.flags & VLFB_EPI_ACCUM))) &&
      !p.relu_mask && (!p.relu_mask_bits || (p.ldd & 15) == 0)) {
    const int Hs = g.H / g.sH, Ws = g.W / g.sW;
    bool ok = true, have_lo = false;
    int ncls = 0;
    ParCls cls[4];
    for (int ph = 0; ph < g.sH; ++ph)
      for (int pw = 0; pw < g.sW; ++pw) {
        ParCls c;
        c.ph = (short)ph; c.pw = (short)pw;
        c.rh = (short)((ph + g.pH) % g.sH); c.rw = (short)((pw + g.pW) % g.sW);
        c.nh = (short)(c.rh < g.kH ? (g.kH - 1 - c.rh) / g.sH + 1 : 0);
        c.nw = (short)(c.rw < g.kW ? (g.kW - 1 - c.rw) / g.sW + 1 : 0);
        if (c.nh == 0 || c.nw == 0) c.nh = c.nw = 0;
        c.nk = g.kT * c.nh * c.nw * (g.Co / KC);
        if (c.nk) {
          const int lw = (pw + g.pW) / g.sW - (c.nw - 1), lh = (ph + g.pH) / g.sH - (c.nh - 1);
          if (have_lo && (lw != par_lo[0] || lh != par_lo[1])) ok = false;
          par_lo[0] = lw; par_lo[1] = lh; have_lo = true;
        }
        cls[ncls++] = c;
      }
    if (ok && have_lo && (int64_t)g.N * g.T * Hs * Ws < (1ll << 31)) {
      // heaviest classes first: the static tile loop hands tiles out round-robin
      for (int i = 0; i < ncls; ++i)
        for (int j = i + 1; j < ncls; ++j)
          if (cls[j].nk > cls[i].nk) { const ParCls t = cls[i]; cls[i] = cls[j]; cls[j] = t; }
      L.par = ncls;
      L.par_m = g.N * g.T * Hs * Ws;
      L.par_lo[0] = par_lo[0]; L.par_lo[1] = par_lo[1];
      for (int i = 0; i < ncls; ++i) L.par_cls[i] = cls[i];
      L.sub.w = make_fastdiv(Ws); L.sub.h = make_fastdiv(Hs); L.sub.t = make_fastdiv(g.T);
      par_lo[2] = g.pT - (g.kT - 1);
      par_hi[0] = par_lo[0] + Ws - g.Wo; par_hi[1] = par_lo[1] + Hs - g.Ho; par_hi[2] = par_lo[2] + g.T - g.To;
      pair_ok = false;
      sk_ws = false;
    }
  }
  Plan plan;
  for (int attempt = 0; attempt < 2; ++attempt) {
    if (L.par) {                       // plan for the class sub-problems: M' rows, one z slice per class
      vlfb_gemm_params_t pp = p;
      pp.M = L.par_m; pp.batch = L.par; pp.K = L.par_cls[0].nk * KC;
      plan = make_plan(pp, num_sms, 0, false, false);
      plan.split_k = 1;
    } else {
      plan = make_plan(p, num_sms, pair_ok ? max_pairs<AK, BK, MASK>() : 0, pair_ok, sk_ws);
    }
    L.bn = plan.bn;
    p.split_k = plan.split_k;
    const int bnh = plan.pair ? L.bn / 2 : L.bn;
    memset(&tmA, 0, sizeof(tmA));
    memset(&tmB, 0, sizeof(tmB));
    const bool mn_tma = ev.tma_mn;
    L.tma_a = (AK == VLFB_OP_DENSE_K && make_tmap(&tmA, p.a, p.M, p.K, p.batch, BM)) ||
              (AK == VLFB_OP_DENSE_MN && mn_tma && make_tmap_mn(&tmA, p.a, p.M, p.K, p.batch)) ? 1 : 0;
    L.tma_b = (BK == VLFB_OP_DENSE_K && make_tmap(&tmB, p.b, p.N, p.K, p.batch, bnh)) ||
              (BK == VLFB_OP_DENSE_MN && mn_tma && make_tmap_mn(&tmB, p.b, p.N, p.K, p.batch)) ? 1 : 0;
    // MN-major tiles as ONE box (all atoms of the tile) instead of one box per 32-element atom
    if (ev.fuse_atoms && !plan.pair) {
      if (AK == VLFB_OP_DENSE_MN && L.tma_a == 1 && make_tmap_mn4(&tmA, p.a, p.M, p.K, p.batch, BM / 32)) L.tma_a = 4;
      if (BK == VLFB_OP_DENSE_MN && L.tma_b == 1 && make_tmap_mn4(&tmB, p.b, p.N, p.K, p.batch, bnh / 32)) L.tma_b = 4;
    }
    if (ev.im2col) {
      // conv gathers as TMA im2col copies: one instruction per K chunk instead of 1024 16-byte cp.asyncs
      const int pad_lo[3] = {-g.pW, -g.pH, -g.pT};
      const int pad_hi[3] = {g.pW - (g.kW - 1) * g.dW, g.pH - (g.kH - 1) * g.dH, g.pT - (g.kT - 1) * g.dT};
      const int cstr[3] = {g.sW, g.sH, g.sT};
      const int ones[3] = {1, 1, 1};
      if (AK == VLFB_OP_CONV_K &&
          make_tmap_im2col(&tmA, p.a.ptr, g.N, g.T, g.H, g.W, g.C, pad_lo, pad_hi, cstr, BM, CU_TENSOR_MAP_SWIZZLE_128B))
        L.tma_a = 2;
      if (AK == VLFB_OP_DGRAD_K && unit_dgrad) {
        const int lo[3] = {g.pW - (g.kW - 1) * g.dW, g.pH - (g.kH - 1) * g.dH, g.pT - (g.kT - 1) * g.dT};
        const int hi[3] = {-g.pW, -g.pH, -g.pT};
        if (make_tmap_im2col(&tmA, p.a.ptr, g.N, g.To, g.Ho, g.Wo, g.Co, lo, hi, ones, BM, CU_TENSOR_MAP_SWIZZLE_128B))
          L.tma_a = 2;
      }
      if (AK == VLFB_OP_DGRAD_K && L.par) {
        if (L.tma_b && make_tmap_im2col(&tmA, p.a.ptr, g.N, g.To, g.Ho, g.Wo, g.Co, par_lo, par_hi, ones, BM, CU_TENSOR_MAP_SWIZZLE_128B))
          L.tma_a = 2;
        else { L.par = 0; continue; }   // not addressable: plan again for the cp.async gather path (any geometry)
      }
      if (AK == VLFB_OP_STEM_K && p.a.ld > 0) {
        // patch tiles need the lean epilogue's row mapping: whole 16-column blocks, 16-byte addressable rows, no mask
        const bool fast_ok = (p.N & 15) == 0 && (p.ldd & 3) == 0 && (p.d_batch_stride & 3) == 0 && (p.d_tap_stride & 3) == 0 &&
                             (reinterpret_cast<uintptr_t>(p.d) & 15) == 0 && !p.relu_mask && !MASK &&
                             (!p.residual || ((reinterpret_cast<uintptr_t>(p.residual) & 15) == 0 && !(p.flags & VLFB_EPI_ACCUM)));
        L.stem_patch = 0;
        if (fast_ok && (g.Ho & 7) == 0 && (g.Wo & 15) == 0 && !ev.no_patch &&
            make_tmap_stem(&tmA, p.a.ptr, g, p.a.ld, CU_TENSOR_MAP_SWIZZLE_128B, 8)) {
          L.tma_a = 3;
          L.stem_patch = 1;
          L.patch_wb = g.Wo / 16;
          L.patch_hb = g.Ho / 8;
        } else if (make_tmap_stem(&tmA, p.a.ptr, g, p.a.ld, CU_TENSOR_MAP_SWIZZLE_128B)) {
          L.tma_a = 3;
        }
      }
      if (BK == VLFB_OP_STEM_MN && p.b.ld > 0 && L.tma_a) {
        L.stem_patch = 0;
        CUtensorMap tmA2;
        memset(&tmA2, 0, sizeof(tmA2));
        // patch chunks: needs dY dense [N*To][Ho][Wo][Co] (ld == M), whole patches, all filter rows in one N tile, and the
        // sH + kH input-row slabs (2 KB each) inside the B stage
        if (!ev.no_patch && AK == VLFB_OP_DENSE_MN && p.a.ld == p.M && p.batch == 1 && (g.Ho & 1) == 0 && (g.Wo & 15) == 0 &&
            p.N <= L.bn && (g.sH + g.kH) * 2048 <= L.bn * KC * 4 && (p.K % KC) == 0 && g.sH <= 8 &&
            make_tmap_stem(&tmB, p.b.ptr, g, p.b.ld, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, -(g.sH + g.kH)) &&
            make_tmap_dy4(&tmA2, p.a.ptr, g)) {
          tmA = tmA2;
          L.tma_b = 3;
          L.stem_patch = 1;
          L.patch_wb = g.Wo / 16;
          L.patch_hb = g.Ho / 2;
        } else if (make_tmap_stem(&tmB, p.b.ptr, g, p.b.ld, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B)) {
          L.tma_b = 3;
        }
      }
      if (BK == VLFB_OP_CONV_MN && (g.C % KC) == 0 && L.tma_a &&
          make_tmap_im2col(&tmB, p.b.ptr, g.N, g.T, g.H, g.W, g.C, pad_lo, pad_hi, cstr, KC,
                           CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B))
        L.tma_b = 2;
      // ... and without spatial taps the whole B tile of a chunk is one dense box (make_tmap_conv_flat)
      if (BK == VLFB_OP_CONV_MN && L.tma_b == 2 && ev.fuse_atoms && !plan.pair &&
          make_tmap_conv_flat(&tmB, p.b.ptr, g, bnh / 32))
        L.tma_b = 5;
    }
    const bool fixup = plan.sk && (!(p.flags & VLFB_EPI_ATOMIC) || det_split);
    if (!(plan.pair || fixup) || (L.tma_a && L.tma_b)) break;
    pair_ok = false;                   // an operand fell back to cp.async: plan again without pairing / fix-ups
    sk_ws = false;
  }
  const int zbase = L.par ? L.par : (p.taps > 1 ? p.taps : p.batch);
  L.tile_rows = plan.pair ? 2 * BM : BM;
  L.tiles_m = ceil_div(L.par ? L.par_m : p.M, L.tile_rows);
  L.tiles_n = ceil_div(p.N, L.bn);
  L.total_tiles = (int)((int64_t)L.tiles_m * L.tiles_n * zbase * p.split_k);
  const int stage_bytes = A_TILE_BYTES + (plan.pair ? L.bn / 2 : L.bn) * KC * 4;
  L.stages = (227 * 1024 - EPI_STAGE_BYTES - 2048) / stage_bytes;
  if (L.stages > (plan.pair ? 7 : 6)) L.stages = plan.pair ? 7 : 6;
  if (ev.stages >= 2 && ev.stages <= L.stages) L.stages = ev.stages;
  L.lag = L.stages - 1 < 2 ? L.stages - 1 : 2;
  if (ev.lag >= 1 && ev.lag < L.stages && ev.lag <= 5) L.lag = ev.lag;
  const int cap = plan.pair ? max_pairs<AK, BK, MASK>() : num_sms;
  int units = L.total_tiles < cap ? L.total_tiles : cap;
#ifdef VLFB_TRACE
  L.trace = g_trace_buf;
#endif
  L.sk = 0;
  if (plan.sk) {
    L.sk = 1;
    L.nkt = ceil_div(p.K, KC);
    units = cap;
    make_bounds(L.bounds, units, (int64_t)L.total_tiles, L.nkt);
    if (!(p.flags & VLFB_EPI_ATOMIC) || det_split) {
      L.ws_cnt = reinterpret_cast<int*>(p.workspace);
      L.ws_tiles = reinterpret_cast<float*>(reinterpret_cast<char*>(p.workspace) + (size_t)SK_CNT_INTS * 4);
    }
  }
  const int smem = L.stages * stage_bytes + EPI_STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
  const bool cp = !(L.tma_a && L.tma_b);
  if (ev.debug)
    fprintf(stderr, "vlfb gemm_tc: kinds %d,%d M=%d N=%d K=%d z=%d | bn=%d pair=%d sk=%d split=%d tiles=%d units=%d stages=%d tma=%d,%d cap=%d patch=%d par=%d\n",
            AK, BK, p.M, p.N, p.K, zbase, L.bn, plan.pair, L.sk, p.split_k, L.total_tiles, units, L.stages, L.tma_a, L.tma_b, cap, L.stem_patch, L.par);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(plan.pair ? 2 * units : units));
  cfg.blockDim = dim3((unsigned)((cp ? NPROD : 32 * NTMAW) + 32 + NEPI));
  cfg.dynamicSmemBytes = (size_t)smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = plan.pair ? 1 : 0;
  // ReLU sign bits are emitted by the lean epilogue; any other path writes them in a second pass over the dense output
  const bool lean = !cp && (p.ldd & 3) == 0 && (p.N & 15) == 0 && span32_ok(p) && (reinterpret_cast<uintptr_t>(p.d) & 15) == 0 &&
                    (!p.residual || ((reinterpret_cast<uintptr_t>(p.residual) & 15) == 0 && !(p.flags & VLFB_EPI_ACCUM)));
  uint32_t* bits_after = nullptr;
  if (p.relu_bits_out && (!lean || MASK)) { bits_after = p.relu_bits_out; p.relu_bits_out = nullptr; }
  int rc = VLFB_OK;
  bool done = false;
  if constexpr (kind_pair_capable(AK) && kind_pair_capable(BK)) {
    if (plan.pair) { rc = launch_variant<AK, BK, MASK, true, false>(cfg, p, L, tmA, tmB); done = true; }
  }
  if (done) {}
  else if (!cp) rc = launch_variant<AK, BK, MASK, false, false>(cfg, p, L, tmA, tmB);
  else rc = launch_variant<AK, BK, MASK, false, true>(cfg, p, L, tmA, tmB);
  if (rc == VLFB_OK && bits_after) rc = relu_bits(p.d, bits_after, (int64_t)p.M * p.N, stream);
  return rc;
}

}  // namespace tc

void gemm_tc_plan(const vlfb_gemm_params_t& p, int num_sms, vlfb_gemm_plan_t* out) {
  // host-only view of the plan: pairing assumes both operands are TMA-addressable and one pair per two SMs
  const bool pair_ok = tc::kind_pair_capable(p.a.kind) && tc::kind_pair_capable(p.b.kind) && p.K >= tc::KC;
  bool sk_ws = p.workspace != nullptr && p.workspace_bytes >= tc::gemm_tc_workspace_bytes();
  const tc::Plan pl = tc::make_plan(p, num_sms, num_sms / 2, pair_ok, sk_ws);
  out->tile_n = pl.bn; out->split_k = pl.split_k; out->pair = pl.pair; out->stream_k = pl.sk;
  out->tiles = pl.tiles; out->units = pl.units;
}

size_t gemm_tc_workspace_bytes() { return tc::gemm_tc_workspace_bytes(); }
#ifdef VLFB_TRACE
void gemm_tc_set_trace(void* buf) { tc::g_trace_buf = reinterpret_cast<unsigned long long*>(buf); }
#endif

int gemm_tc(const vlfb_gemm_params_t& p, cudaStream_t stream) {
  const int ak = p.a.kind, bk = p.b.kind;
  if (p.relu_mask || p.relu_mask_bits) {
    // ReLU-backward mask: only the dgrad shapes need it (two more instantiations, not eighteen)
    if (ak == VLFB_OP_DGRAD_K && bk == VLFB_OP_DENSE_K) return tc::launch<VLFB_OP_DGRAD_K, VLFB_OP_DENSE_K, true>(p, stream);
    if (ak == VLFB_OP_DENSE_K && bk == VLFB_OP_DENSE_K) return tc::launch<VLFB_OP_DENSE_K, VLFB_OP_DENSE_K, true>(p, stream);
    set_error("vlfb_gemm: relu_mask is supported for DGRAD_K/DENSE_K x DENSE_K operands only (tensor-core engine)");
    return VLFB_E_BADARG;
  }
#define VLFB_TC_CASE(A, B) if (ak == A && bk == B) return tc::launch<A, B, false>(p, stream)
  VLFB_TC_CASE(VLFB_OP_CONV_K, VLFB_OP_DENSE_K);
  VLFB_TC_CASE(VLFB_OP_STEM_K, VLFB_OP_DENSE_K);
  VLFB_TC_CASE(VLFB_OP_DGRAD_K, VLFB_OP_DENSE_K);
  VLFB_TC_CASE(VLFB_OP_DENSE_MN, VLFB_OP_CONV_MN);
  VLFB_TC_CASE(VLFB_OP_DENSE_MN, VLFB_OP_STEM_MN);
  VLFB_TC_CASE(VLFB_OP_DENSE_K, VLFB_OP_DENSE_K);
  VLFB_TC_CASE(VLFB_OP_DENSE_K, VLFB_OP_DENSE_MN);
  VLFB_TC_CASE(VLFB_OP_DENSE_MN, VLFB_OP_DENSE_K);
  VLFB_TC_CASE(VLFB_OP_DENSE_MN, VLFB_OP_DENSE_MN);
#undef VLFB_TC_CASE
  set_error("gemm_tc: unsupported operand kinds (%d, %d)", ak, bk);
  return VLFB_E_UNSUPPORTED;
}

}  // namespace vlfb
