// ptx.cuh -- the inline-PTX primitives of the sm_100a kernels, one wrapper per instruction form.  Every asm statement of the library
// lives here.  The qualifiers are part of each wrapper's contract: `volatile` keeps the statement in program order among the other
// volatile statements (decode_cluster.cu's mma_mtile and attn_tile rely on program order being issue order), a "memory" clobber
// orders it against ordinary loads and stores, and an "n" operand is an immediate of the instruction.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

// ---- addresses and cluster -----------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// the same shared address in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa(uint32_t addr, uint32_t rank) {
  uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank)); return r;
}
__device__ __forceinline__ uint32_t cluster_rank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n" : "=r"(pred));
  return pred != 0;
}
// 4 bytes into a peer CTA's shared memory, counted as transaction bytes on the peer's mbarrier
__device__ __forceinline__ void st_async_b32(uint32_t raddr, uint32_t v, uint32_t rbar) {
  asm volatile("st.async.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(raddr), "r"(v), "r"(rbar) : "memory");
}

// ---- mbarrier --------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbarrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_n(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t local_bar, uint32_t cta) {   // arrive on the same barrier in CTA `cta` of the cluster
  const uint32_t r = mapa(local_bar, cta);
  // default semantics (release at CTA scope): the arrival orders this warp's TMEM reads (tcgen05.fence::before_thread_sync) before the
  // leader's next MMAs; .release.cluster would add a cluster-scope memory fence per warp and tile (~1 us per tile measured)
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(r) : "memory");
}
// bounded wait: a protocol bug traps (reported as a launch failure) instead of hanging the GPU box.  try_wait carries a suspend-time
// hint: the waiting warp SLEEPS in hardware until the phase completes (or the hint expires) instead of spinning -- a spinning
// waiter (without the hint try_wait returns after a few hundred cycles: 1.2 G of the 6.5 G instructions of a 256-image launch were
// this loop, profiles/r2b) takes issue slots from the warps of the same SM sub-partition that have work, in particular from
// the second CTA that shares the SM in the two-CTAs-per-SM variant.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  while (true) {
    asm volatile("{\n\t.reg .pred P1;\n\tmbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2, %3;\n\tselp.u32 %0, 1, 0, P1;\n\t}\n"
                 : "=r"(done) : "r"(bar), "r"(parity), "r"(1000000u) : "memory");      // hint: 1 ms
    if (done) break;
    if (++spins > 2000u) __trap();          // ~2 s
  }
}
// bounded wait (the GEMM's spinning form): a protocol bug traps (reported as a launch failure) instead of hanging the GPU box
__device__ __forceinline__ void mbar_wait_spin(uint32_t bar, uint32_t parity) {
  uint32_t done = 0, spins = 0;
  long long t0 = 0;
  while (true) {
    asm volatile("{\n\t.reg .pred P1;\n\tmbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n\tselp.u32 %0, 1, 0, P1;\n\t}\n"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    if (done) break;
    if ((++spins & 1023u) == 0) {
      long long now = clock64();
      if (t0 == 0) t0 = now;
      else if (now - t0 > 4000000000LL) __trap();   // ~2 s
    }
  }
}

// ---- cp.async, bulk copies and TMA -----------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async8(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { cp_async_commit(); cp_async_wait<0>(); }
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
// TMA bulk copy (non-tensor): `bytes` contiguous bytes global -> shared, completion counted on an mbarrier.  The decode cluster kernel
// moves EVERYTHING it streams this way (16-32 KB weight stages, 2 KB key/value chunks): tensor-map boxes cost the TMA unit ~4.5 cycles
// per box ROW whatever its width (64-byte head slices: 14 B/clk/SM, 128-byte weight rows: 28 B/clk/SM -- profiles/r2d), which bounded
// the previous version of that kernel; contiguous copies of pre-arranged shared-memory images do not pay per row.
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}
// L2 prefetch of a contiguous block (no shared memory involved): the decode cluster kernel's producer warp pulls the cross-K/V chunks it
// will copy a few stages later from HBM into L2, so that the copies themselves meet L2 latency -- the ring holds at most three stages
// ahead, which at HBM latency is the per-SM streaming rate the cross-attention phase ran at (~40 B/clk)
__device__ __forceinline__ void bulk_prefetch_l2(const void* src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) { asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory"); }
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint32_t bar, uint32_t dst, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1) : "memory");
}
// cta_group::2: the load completes on the mbarrier of the pair's leader CTA (leader_bar is a cluster address)
__device__ __forceinline__ void tma_load_2d_2sm(const CUtensorMap* map, uint32_t leader_bar, uint32_t dst, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"(dst), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1) : "memory");
}
// shared -> global tile store / reduce-add through the TMA unit (coalesced, OOB rows and columns clipped)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map), "r"(src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
// order this thread's generic-proxy memory accesses before later async-proxy ones (TMA and bulk copies): every state space, or only
// this CTA's shared memory
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- ldmatrix and mma.sync -----------------------------------------------------------------------------------------------
__device__ __forceinline__ void ldsm_x4(uint32_t* r, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t* r, uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
// byte offset of 16-byte chunk `c` of row `r` in a [rows][HD 16-bit elements] panel, swizzled so that ldmatrix (eight consecutive
// rows, one chunk) is conflict-free: 64-byte rows: c ^ ((r >> 1) & 3); 128- and 256-byte rows: c ^ (r & 7)
template <int HD>
__device__ __forceinline__ uint32_t swz(int r, int c) {
  if constexpr (HD == 32) return (uint32_t)(r * 64 + ((c ^ ((r >> 1) & 3)) << 4));
  else return (uint32_t)(r * (HD * 2) + ((c ^ (r & 7)) << 4));
}
// c (16 x 8, f32) += a (16 x 16) . b (16 x 8), T = __nv_bfloat16 or __half operands
template <typename T> __device__ __forceinline__ void mma_m16n8k16(float* c, const uint32_t* a, uint32_t b0, uint32_t b1);
template <> __device__ __forceinline__ void mma_m16n8k16<__nv_bfloat16>(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
template <> __device__ __forceinline__ void mma_m16n8k16<__half>(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// ---- tcgen05 (5th-generation tensor cores, tensor memory) -----------------------------------------------------------------
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// D[tmem] (+)= A[smem desc] . B[smem desc]
__device__ __forceinline__ void umma_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
               ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// D[tmem] (+)= A[tmem] . B[smem desc]
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
               ::"r"(tmem_d), "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// umma_ss issued by the leader CTA of a pair for both (cta_group::2)
__device__ __forceinline__ void umma_ss_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
               ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint32_t bar) {     // arrives on the barrier at this offset in BOTH CTAs of the pair
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"((uint16_t)3) : "memory");
}
__device__ __forceinline__ void tmem_ld4(uint32_t addr, uint32_t* v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]) : "r"(addr));
}
__device__ __forceinline__ void tmem_ld16(uint32_t addr, uint32_t* v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                 "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]) : "r"(addr));
}
__device__ __forceinline__ void tmem_ld32(uint32_t addr, uint32_t* v) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
               "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
               "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                 "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                 "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
                 "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
               : "r"(addr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st2(uint32_t addr, uint32_t a, uint32_t b) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// tensor-memory allocation by one warp: `cols` columns, base address written to shared memory at `dst`; CG = CTA group (1 or 2)
template <int CG> __device__ __forceinline__ void tmem_alloc(uint32_t dst, uint32_t cols) {
  if constexpr (CG == 2) asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst), "r"(cols) : "memory");
  else asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst), "r"(cols) : "memory");
}
template <int CG> __device__ __forceinline__ void tmem_relinquish() {
  if constexpr (CG == 2) asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  else asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int CG> __device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t cols) {
  if constexpr (CG == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
  else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
}
// SWIZZLE_128B operand tile: rows of 128 B, 8-row groups 1024 B apart (SBO); LBO unused.  K-major use: the rows are the M / N index;
// MN-major use (selected by the instruction descriptor's transpose bit): the rows are the K index, the 64 elements of a row the N index.
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);          // start address        bits [0,14)
  d |= (uint64_t)(1024 >> 4) << 32;                // stride byte offset   bits [32,46)
  d |= (uint64_t)1 << 46;                          // descriptor version 1 (sm_100)
  d |= (uint64_t)2 << 61;                          // layout type SWIZZLE_128B
  return d;
}
// kind::f16 instruction descriptor: D = f32 (bits 4-5 = 1), A and B formats at bits 7-9 / 10-12 (0 = fp16, 1 = bf16), bit 16 = B is
// MN-major (else both operands K-major), N >> 3 at bit 17, M >> 4 at bit 24
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, bool f16 = false, bool b_mn_major = false) {
  return (1u << 4) | ((f16 ? 0u : 1u) << 7) | ((f16 ? 0u : 1u) << 10) | ((b_mn_major ? 1u : 0u) << 16) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

// ---- shared 128-bit load / store, named barriers --------------------------------------------------------------------------
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v; asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr)); return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// barrier ID over COUNT threads (a multiple of 32; ID 0 is __syncthreads' barrier)
template <int ID, int COUNT> __device__ __forceinline__ void bar_sync() { asm volatile("bar.sync %0, %1;" ::"n"(ID), "n"(COUNT) : "memory"); }
template <int COUNT> __device__ __forceinline__ void bar_sync(uint32_t id) { asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(COUNT) : "memory"); }

// ---- exp2 and packed f32x2 arithmetic --------------------------------------------------------------------------------------
// exp2f() adds denormal range handling the softmax does not need
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// packed fp32 pairs (sm_100 FFMA2 / FADD2): two values per instruction
__device__ __forceinline__ uint64_t pk2(float a, float b) { uint64_t r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void upk2(uint64_t v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ uint64_t fma2(uint64_t a, uint64_t b, uint64_t c) { uint64_t d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ uint64_t add2(uint64_t a, uint64_t b) { uint64_t d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

// ---- bf16x2 / f16x2 packing (round to nearest; a in the low half) ---------------------------------------------------------
__device__ __forceinline__ uint32_t pack_bf16x2(float a, float b) { __nv_bfloat162 h = __floats2bfloat162_rn(a, b); return *reinterpret_cast<uint32_t*>(&h); }
__device__ __forceinline__ uint32_t pack_f16x2(float a, float b) { __half2 h = __floats2half2_rn(a, b); return *reinterpret_cast<uint32_t*>(&h); }
