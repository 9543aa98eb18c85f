// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk[.tensor]), tcgen05 (alloc/mma/commit/ld).
// Written against the PTX ISA 8.7 forms; nothing here is a library call.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace csr {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
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
// Bounded wait: a protocol bug must surface as a launch failure, never as a hung GPU.
static __device__ __noinline__ void mbar_timeout(uint32_t bar, uint32_t parity) {
  printf("climsr_b200: mbarrier timeout block %d thread %d bar %u parity %u\n", blockIdx.x, threadIdx.x, bar, parity);
  __trap();
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 22)) mbar_timeout(bar, parity);
  }
}
// Unbounded wait, three instructions.  The conv kernel has ~20 wait sites and must stay below the ~32 KB the SM's
// instruction cache holds (growing past it cost 9 % of the whole forward), so only ONE site per kernel keeps the
// bounded form - the epilogue's accumulator wait, which every stalled pipeline ends up starving, so a protocol bug still
// surfaces there as a trap instead of a hang.
__device__ __forceinline__ void mbar_wait_spin(uint32_t bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ---------------------------------------------------------------- programmatic dependent launch
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// in-situ timeline of a launch sequence (debug): globaltimer stamps reduced over the CTAs of a launch
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void timeline_start(unsigned long long* tl, int id) {
  if (tl && threadIdx.x == 0) atomicMin(tl + 2 * id, globaltimer_ns());
}
__device__ __forceinline__ void timeline_end(unsigned long long* tl, int id) {
  if (tl && threadIdx.x == 0) atomicMax(tl + 2 * id + 1, globaltimer_ns());
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const void* tmap, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(bar)
               : "memory");
}


// bulk tensor store shared -> global (TMA clips coordinates outside the tensor), bulk async-group bookkeeping
__device__ __forceinline__ void tma_store_4d(const void* tmap, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void bulk_commit_group() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_group_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_group() { asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// fire-and-forget vector fp32 add into global memory (sm_90+): one L2 atomic per 16 bytes
__device__ __forceinline__ void red_add_v4_f32(float* ptr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(ptr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// One lane of a fully converged warp (the same lane every time, so tcgen05.commit tracks that lane's MMAs).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .b32 r;\n\t.reg .pred p;\n\t"
      "elect.sync r|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// Same MMA with the two 64-bit descriptors given as (lo, hi) 32-bit halves: between the MMAs of a tile only the
// 14-bit start-address field (lo word) changes, so the issue loop is two 32-bit adds per MMA.
__device__ __forceinline__ void umma_bf16_split(uint32_t d_tmem, uint32_t a_lo, uint32_t a_hi, uint32_t b_lo, uint32_t b_hi,
                                                uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %2};\n\t"
      "mov.b64 db, {%3, %4};\n\t"
      "setp.ne.b32 p, %6, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %5, p;\n\t}"
      ::"r"(d_tmem), "r"(a_lo), "r"(a_hi), "r"(b_lo), "r"(b_hi), "r"(idesc), "r"(accumulate)
      : "memory");
}

// D[tmem] (+)= A[smem desc] * B[smem desc], bf16 x bf16 -> fp32, single CTA.
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// All previously issued MMAs of this thread arrive on `bar` when they complete (implies fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// 32 lanes x 16 consecutive fp32 columns -> 16 registers per thread (lane i of the warp reads TMEM lane base+i).
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr)
      : "memory");
}
// 32 lanes x 8 consecutive fp32 columns -> 8 registers per thread.
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// ---------------------------------------------------------------- descriptors
// Instruction descriptor, kind::f16: D=f32 (bits 4-5 = 1), A=B=bf16 (bits 7-9, 10-12 = 1), K-major A and B,
// N>>3 at bit 17, M>>4 at bit 24.
__host__ __device__ constexpr uint32_t make_idesc_bf16(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
// Shared-memory matrix descriptor. addr/lbo/sbo in bytes (multiples of 16); version 1 (sm_100);
// layout: 0 = no swizzle (8x16B core matrices), 2 = 128-byte swizzle.
__device__ __forceinline__ uint64_t make_sdesc(uint32_t addr, uint32_t lbo, uint32_t sbo, uint32_t layout, uint32_t base_off) {
  return static_cast<uint64_t>((addr >> 4) & 0x3FFF) | (static_cast<uint64_t>((lbo >> 4) & 0x3FFF) << 16) |
         (static_cast<uint64_t>((sbo >> 4) & 0x3FFF) << 32) | (1ull << 46) | (static_cast<uint64_t>(base_off & 7) << 49) |
         (static_cast<uint64_t>(layout) << 61);
}

// ---------------------------------------------------------------- misc
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16hi(uint32_t v) { return __uint_as_float(v & 0xFFFF0000u); }
// hi/lo bf16 pair of two fp32 values: hi = bf16(v), lo = bf16(v - hi) (v - hi is exact in fp32; hi + lo is v to ~2^-16 relative)
__device__ __forceinline__ void split_bf16x2(float a, float b, uint32_t* hi, uint32_t* lo) {
  *hi = pack_bf16x2(a, b);
  *lo = pack_bf16x2(a - bf16lo(*hi), b - bf16hi(*hi));
}

// ---------------------------------------------------------------- whole-row tiles (conv_tc.cu / rdb_tc.cu, WR_T)
// The epilogue sums the folded 3x3 taps as out[m] = D[m-1][tap 0] + D[m][tap 1] + D[m+1][tap 2] with warp shuffles that wrap
// around the warp: lane 0 receives lane 31's tap-0 value, lane 31 lane 0's tap-2 value.  These two helpers put into those two
// source registers what the edge pixels need instead - +0 at an image edge (exactly what a zero-filled halo column contributed),
// or, where a 64-pixel row spans two warps (`left`: the TMEM lane quadrant with pixels 0..31 of the row), the other warp's
// boundary value - so the summation order, and with it every output bit, is that of a tiling with halo columns.
// 64 bytes per chunk and warp pair: the left warp's lane-31 tap 0, then the right warp's lane-0 tap 2.  row_edge_put: `dst` = this
// thread's half of the slot.  row_edge_get (after the pair's named barrier): lane 31 reloads tap 0, lane 0 tap 2 from `src` = the
// other warp's half of the slot, or 32 zero bytes (edge_addrs).
__device__ __forceinline__ void edge_addrs(uint32_t slot, uint32_t zeros, bool pair, bool left, int lane, uint32_t* dst, uint32_t* src) {
  *dst = left ? slot : slot + 32u;
  *src = !pair ? zeros : lane == 31 ? (left ? zeros : slot) : (left ? slot + 32u : zeros);
}
// predicated forms (one SETP, no branch): the exchange sits in the epilogue's unrolled chunk loop, inside the instruction-cache budget
__device__ __forceinline__ void st_shared_v8_if(bool pred, uint32_t addr, const uint32_t (&t)[8]) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %0, 0;\n\t"
               "@p st.shared.v4.b32 [%1], {%2, %3, %4, %5};\n\t@p st.shared.v4.b32 [%1+16], {%6, %7, %8, %9};\n\t}"
               ::"r"(static_cast<uint32_t>(pred)), "r"(addr), "r"(t[0]), "r"(t[1]), "r"(t[2]), "r"(t[3]), "r"(t[4]), "r"(t[5]), "r"(t[6]), "r"(t[7])
               : "memory");
}
__device__ __forceinline__ void ld_shared_v8_if(bool pred, uint32_t addr, uint32_t (&t)[8]) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %8, 0;\n\t"
               "@p ld.shared.v4.b32 {%0, %1, %2, %3}, [%9];\n\t@p ld.shared.v4.b32 {%4, %5, %6, %7}, [%9+16];\n\t}"
               : "+r"(t[0]), "+r"(t[1]), "+r"(t[2]), "+r"(t[3]), "+r"(t[4]), "+r"(t[5]), "+r"(t[6]), "+r"(t[7])
               : "r"(static_cast<uint32_t>(pred)), "r"(addr)
               : "memory");
}
__device__ __forceinline__ void row_edge_put(const uint32_t (&t0)[8], const uint32_t (&t2)[8], uint32_t dst, int lane, bool left) {
  st_shared_v8_if(left && lane == 31, dst, t0);
  st_shared_v8_if(!left && lane == 0, dst, t2);
}
__device__ __forceinline__ void row_edge_get(uint32_t (&t0)[8], uint32_t (&t2)[8], uint32_t src, int lane) {
  ld_shared_v8_if(lane == 31, src, t0);
  ld_shared_v8_if(lane == 0, src, t2);
}

}  // namespace csr
