// Thin inline-PTX wrappers for sm_100a: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (MMA / TMEM),
// cp.async.  No CUTLASS/CuTe dependency: every encoding used here
// is written out so the SASS can be checked (UTCHMMA / UTMALDG / LDTM).
#pragma once
#include <cstdint>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

namespace jcb {

// Error codes a kernel can leave in the context's device-side status word.
enum : int {
  JCB_DEV_OK = 0,
  JCB_DEV_TIMEOUT_PRODUCER = 101,
  JCB_DEV_TIMEOUT_MMA = 102,
  JCB_DEV_TIMEOUT_EPILOGUE = 103,
  JCB_DEV_SMEM_ALIGN = 104,   // dynamic shared memory not 1024-byte aligned (swizzled TMA / UMMA tiles need it)
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a pipeline bug must never hang the GPU.  On timeout (or when another role already
// flagged an error) the caller's role loop is abandoned, the kernel drains and the host reports
// the status word.  Returns true when the barrier phase completed.
#ifndef JCB_MBAR_TIMEOUT_NS
#define JCB_MBAR_TIMEOUT_NS 2000000000ull
#endif
__device__ __forceinline__ bool mbar_wait(uint64_t* bar, uint32_t parity, int* status, int code) {
  if (mbar_try_wait(bar, parity)) return true;
  const uint64_t t0 = globaltimer_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (((++spins) & 255u) == 0u) {
      if (*reinterpret_cast<volatile int*>(status) != 0) return false;
      if (globaltimer_ns() - t0 > JCB_MBAR_TIMEOUT_NS) {
        atomicCAS(status, 0, code);
        return false;
      }
    }
  }
  return true;
}

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tm) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
}
// 2-D tiled load global -> shared, completion reported as tx bytes on `bar`.
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0,
                                            int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}


// ---------------------------------------------------------------- TMA stores (shared -> global, bulk groups)
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tm, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tm)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
// global[tile] += shared[tile], element-wise fp32 add performed by the memory system (no read into the SM)
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* tm, const void* smem_src, int c0, int c1) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tm)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// wait until at most N of this thread's bulk groups still READ their shared-memory source
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
// wait until at most N of this thread's bulk groups are incomplete (writes performed)
template <int N>
__device__ __forceinline__ void bulk_wait() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ float tanh_approx(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---------------------------------------------------------------- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// Arrive on `bar` once every tcgen05.mma issued so far by this thread has completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
// Shared-memory matrix descriptor: K-major operand tile written by TMA with 128-byte swizzle.
//   bits [0,14)  start address >> 4          bits [16,30) leading byte offset >> 4 (ignored for
//   bits [32,46) stride byte offset >> 4      swizzled K-major; 1 as CuTe sets it)
//   bits [46,48) descriptor version = 1 (sm_100)   bits [61,64) layout type 2 = SWIZZLE_128B
// Rows are 128 B apart, 8-row swizzle atoms are 1024 B apart (SBO).  Advancing K by 16 bf16 inside
// the 128-byte atom adds 32 B to the start address; tiles are 1024-B aligned so the hardware XOR
// pattern (address bits [4,7) ^ bits [7,10)) is preserved.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor for kind::f16: D=f32 (bits[4,6)=1), A=B=bf16 (bits[7,10)=1, [10,13)=1),
// both operands K-major (bits 15,16 = 0), N>>3 at [17,23), M>>4 at [24,29).
__host__ __device__ constexpr uint32_t umma_idesc_bf16_f32(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}
// The same with the 16-bit operand type chosen by the caller: kind::f16 multiplies fp16 (format 0) and bf16 (format 1)
// operands at the same rate, so the operand type is a property of the data, not of the kernel.
__host__ __device__ constexpr uint32_t umma_idesc_f32acc(bool f16, int m, int n, bool b_mn_major = false) {
  return (1u << 4) | (f16 ? 0u : ((1u << 7) | (1u << 10))) | (b_mn_major ? (1u << 16) : 0u) |
         (static_cast<uint32_t>(n >> 3) << 17) | (static_cast<uint32_t>(m >> 4) << 24);
}
// D[tmem] (+)= A[smem] * B[smem]^T ; issued by ONE thread for the whole CTA.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (thread = lane = row).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]),
        "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]),
        "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// registers -> TMEM: this warp's 32 lanes x 32 consecutive 32-bit columns (thread = lane = row)
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
        "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
        "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
        "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// Shared-memory matrix descriptor of an MN-major operand tile (the MN dimension is the contiguous one) written
// by TMA with 128-byte swizzle: rows = K index, 128 B (64 bf16 of MN) per row, 8-row groups 1024 B apart (SBO).
// One 64-element MN atom only, so the leading byte offset (stride between MN atoms) is never used.
// Advancing K by 16 = two 8-row groups adds 2048 B to the start address.
__device__ __forceinline__ uint64_t umma_desc_sw128_mn(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(1024 >> 4) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// kind::f16 instruction descriptor with B MN-major (bit 16): D = f32, A = B = bf16, A K-major
__host__ __device__ constexpr uint32_t umma_idesc_bf16_f32_bmn(int m, int n) {
  return (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | (static_cast<uint32_t>(n >> 3) << 17) |
         (static_cast<uint32_t>(m >> 4) << 24);
}
// D[tmem] (+)= A[tmem] * B[smem]: the A operand (bf16 pairs packed in 32-bit columns, row = lane) comes from TMEM
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// 4-D tiled TMA load / store (attention: [view][head block][token][64] boxes)
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0, int c1,
                                            int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2),
      "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* tm, const void* smem_src, int c0, int c1, int c2,
                                             int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(tm)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
// Packed fp32 pairs (FADD2 / FMUL2 / FFMA2 on sm_100): one instruction, two IEEE fp32 results -- the epilogues'
// elementwise math costs half the issue slots and instruction energy, with bit-identical results per element.
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// ---------------------------------------------------------------- programmatic dependent launch
// A kernel launched with cudaLaunchAttributeProgrammaticStreamSerialization (kernels.h launch_pdl) may become resident
// while the kernel in front of it in the stream is still running: everything up to griddep_wait() -- barrier
// initialisation, TMEM allocation, tensor-map prefetch, the cluster's first synchronisation -- overlaps that kernel's
// tail, and the launch latency itself disappears from the chain (~70 dependent kernels per pipeline call).
// griddep_wait() returns once ALL prerequisite grids have completed and their memory is visible; nothing that another
// kernel wrote may be read, and nothing it may still read may be written, before it.  It is a no-op in a kernel launched
// without the attribute.  The attribute is opt-in (JCB_PDL=1, api.cu pdl_enabled).
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// No kernel issues griddepcontrol.launch_dependents: with that early trigger right after the wait, two full-size pipeline
// calls adjacent in a stream hang (tools/pdl_first_calls_probe.py, profiles/r02_pdl_hang_probes.log).  The dependents are
// released by the exit of the primary's CTAs instead -- the same probe finishes (0.55 s) -- and still overlap their
// prologue with its last wave.

__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}


// ---------------------------------------------------------------- clusters / CTA pairs (cta_group::2)
// In the shared::cluster window the two CTAs of a pair differ in bit 24 of the address; clearing it
// turns "my barrier" into "the same barrier in the even (leader) CTA" (CuTe's Sm100MmaPeerBitMask).
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Arrive on an mbarrier that may live in the peer CTA (address in the shared::cluster window).  Default semantics
// (release at CTA scope = one SYNCS.ARRIVE): the `.release.cluster` form compiles to MEMBAR.ALL.GPU + ERRBAR +
// CGAERRBAR in front of the arrive, which cost an epilogue warp ~20 % of its time (profiles/r01e: 14 % of all stall
// samples of the c_fc GEMM).  The TMEM reads this arrive publishes are ordered by tcgen05.wait::ld +
// tcgen05.fence::before_thread_sync, not by the memory model.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// 2-D tiled load issued by either CTA of a pair into ITS OWN shared memory; the bytes are reported
// on the LEADER CTA's mbarrier (which the single MMA-issuing thread waits on).
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* tm, uint64_t* bar, int c0,
                                                 int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tm)), "r"(smem_u32(bar) & PEER_BIT_MASK), "r"(c0),
      "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// Arrive on the barrier at this offset in BOTH CTAs of the pair once all MMAs issued so far completed.
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  const uint16_t mask = 0x3;
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
          smem_u32(bar)),
      "h"(mask)
      : "memory");
}
// D[tmem, both CTAs] (+)= A[smem, 128 rows per CTA] * B[smem, N/2 rows per CTA]^T: UMMA M = 256 across the
// pair, issued by ONE thread of the leader CTA.
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  const uint32_t z = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(z)
      : "memory");
}

// ---------------------------------------------------------------- cp.async (MTA probabilities)
__device__ __forceinline__ void cp_async_16(uint32_t saddr, const void* gptr) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(gptr) : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
// ---------------------------------------------------------------- 16-bit operand type (bf16 | fp16)
// Every 16-bit tensor of a tower (weights, the raw residual copy, q|k|v, P, attention output, MLP hidden) has ONE
// element type, fixed when the tower is packed: bf16 (the north star's wording) or fp16 (3 more mantissa bits at the
// same tensor-core rate: 8x less operand rounding, which is what puts the x100 logits within 1e-2 of the fp32
// reference; DESIGN.md section 3).  fp16 conversions SATURATE (+-65504) instead of producing inf.
template <bool F16>
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  if (F16) {
    uint32_t r;
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
  }
  return pack_bf16x2(lo, hi);
}
template <bool F16>
__device__ __forceinline__ float2 unpack_h2(uint32_t v) {
  if (F16) return __half22float2(*reinterpret_cast<const __half2*>(&v));
  return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&v));
}
template <bool F16>
__device__ __forceinline__ uint16_t to_h(float x) {
  return static_cast<uint16_t>(pack_h2<F16>(x, 0.f) & 0xFFFFu);
}
template <bool F16>
__device__ __forceinline__ float from_h(uint16_t v) {
  return unpack_h2<F16>(static_cast<uint32_t>(v)).x;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

}  // namespace jcb
