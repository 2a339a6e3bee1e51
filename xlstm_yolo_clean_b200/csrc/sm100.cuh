// Inline-PTX wrappers for the Blackwell (sm_100a) primitives the tensor-core kernels use:
// mbarrier, TMA (cp.async.bulk.tensor), tcgen05.mma / commit / ld, TMEM alloc, proxy fences, cluster / DSMEM.
// Descriptor bit layouts follow the PTX ISA "tcgen05 matrix / instruction descriptor" tables.
#pragma once

#include <cuda.h>  // CUtensorMap
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

namespace sm100 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\tmbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\tselp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a lost arrival traps (the error surfaces to the host) instead of hanging the GPU.
// The bound is ~2^31 SM cycles (about one second); `tag` is stored to *g_dbg (if set) first.
#ifndef SM100_WAIT_CYCLES
#define SM100_WAIT_CYCLES (1ll << 31)
#endif
static __device__ volatile int* g_dbg = nullptr;
// slow path kept out of line: the kernels are instruction-cache sensitive
__device__ __noinline__ void mbar_wait_slow(uint64_t* bar, uint32_t parity, int tag) {
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > SM100_WAIT_CYCLES) {
      if (g_dbg) {
        g_dbg[0] = tag;
        g_dbg[1] = (int)(blockIdx.x * 1000 + threadIdx.x);
        __threadfence_system();
      }
      __trap();
    }
  }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int tag = 0) {
  if (mbar_try_wait(bar, parity)) return;
  if (mbar_try_wait(bar, parity)) return;  // try_wait suspends for a while by itself; retry once inline
  mbar_wait_slow(bar, parity, tag);
}

// ---------------------------------------------------------------- thread-block clusters / distributed shared memory
// shared::cluster address of the variable at `p` (own shared memory) in the CTA of cluster rank `rank`
__device__ __forceinline__ uint32_t cluster_map(const void* p, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
__device__ __forceinline__ void st_cluster_f2(uint32_t caddr, float a, float b) {
  asm volatile("st.shared::cluster.v2.f32 [%0], {%1, %2};" ::"r"(caddr), "f"(a), "f"(b) : "memory");
}
// arrive on an mbarrier of another CTA of the cluster; release: this thread's earlier writes (and those it has observed,
// e.g. through __syncwarp) are visible to whoever acquires the completed phase
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t caddr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(caddr) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait_cluster(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\tmbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P, [%1], %2;\n\tselp.u32 %0, 1, 0, P;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// bounded like mbar_wait: a lost remote arrival traps instead of hanging the GPU
__device__ __noinline__ void mbar_wait_cluster_slow(uint64_t* bar, uint32_t parity) {
  const long long t0 = clock64();
  while (!mbar_try_wait_cluster(bar, parity))
    if (clock64() - t0 > SM100_WAIT_CYCLES) __trap();
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait_cluster(bar, parity)) return;
  mbar_wait_cluster_slow(bar, parity);
}
// every thread of every CTA of the cluster; release / acquire order the shared-memory accesses around it cluster-wide
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// ---------------------------------------------------------------- programmatic dependent launch
// wait: blocks until the grid this one was made dependent on (launch attribute programmaticStreamSerialization)
// has completed and its memory is visible; a no-op for a normal launch.  launch_dependents: lets the NEXT
// dependent grid's CTAs take an SM as soon as resources free up; they must not touch global memory before their
// own wait.
__device__ __forceinline__ void grid_dep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void grid_dep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// ---------------------------------------------------------------- named barriers (sub-CTA handoff)
// arrive: non-blocking (producer side); sync: blocking.  `count` = total participating threads.
__device__ __forceinline__ void named_arrive(int id, int count) {
  asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(count) : "memory");
}
__device__ __forceinline__ void named_sync(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---------------------------------------------------------------- fences
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// ---------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"((uint64_t)m) : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2,
                                            int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"((uint64_t)m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_4d(const CUtensorMap* m, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global [%0, {%1, %2, %3, %4}];" ::"l"((uint64_t)m), "r"(c0), "r"(c1),
               "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"((uint64_t)m),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
// global[tile] += shared[tile] (element type of the tensor map: f16 / bf16 add, rounded once per element), bulk-group tracked
__device__ __forceinline__ void tma_reduce_add_4d(const CUtensorMap* m, const void* smem_src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.reduce.async.bulk.tensor.4d.global.shared::cta.add.tile.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"((uint64_t)m),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait_all() {
  asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}

// ---------------------------------------------------------------- TMEM
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(NCOLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {  // same warp that allocated
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}

__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive fp32 columns: thread i of warp w gets TMEM lane 32*(w%4)+i.
// _nowait: the caller issues several loads and then one tmem_ld_wait().
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
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
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
// one 32-bit column of this thread's lane (no wait)
__device__ __forceinline__ void tmem_ld1_nowait(uint32_t taddr, uint32_t& r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld16_nowait(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}

// registers -> TMEM: thread i of warp w writes TMEM lane 32*(w%4)+i, N consecutive 32-bit columns
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
      "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr), "r"(r[0]),
               "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- UMMA descriptors
// Shared-memory matrix descriptor for a 128B-swizzled tile whose rows are 128 bytes
// (64 x 16-bit) and whose 8-row swizzle atoms are 1024 B apart (dense [rows][64] tile):
//   bits  0-13 start address >> 4        bits 16-29 leading byte offset >> 4
//   bits 32-45 stride byte offset >> 4   bits 46-47 version = 1 (sm_100)
//   bits 61-63 layout type (2 = SWIZZLE_128B)
// K-major  (rows = M/N index, 128B row = 64 K elements): SBO = 1024 (next 8 rows), LBO unused.
// MN-major (rows = K index,  128B row = 64 M/N elements): SBO = 1024 (next 8 K rows),
//           LBO = byte distance to the next 64-wide M/N block.
// general form: layout type 2 = SWIZZLE_128B, 4 = SWIZZLE_64B (rows of 64 bytes, 512-byte swizzle atoms)
__device__ __forceinline__ uint64_t umma_smem_desc_lt(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                                      uint32_t layout_type) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout_type << 61;
  return d;
}
__device__ __forceinline__ uint64_t umma_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Advance the start address of a descriptor by `bytes` (multiple of 16; no carry out of the field
// as long as the tile stays inside the 256 KB shared window).
__device__ __forceinline__ uint64_t umma_desc_advance(uint64_t desc, uint32_t bytes) { return desc + (uint64_t)(bytes >> 4); }

// Instruction descriptor for kind::f16 (bf16 or fp16 inputs, fp32 accumulate).
//   bits 4-5 D format (1 = f32), 7-9 A format, 10-12 B format (0 = f16, 1 = bf16),
//   bit 15 A major, bit 16 B major (0 = K, 1 = MN), bits 17-22 N>>3, bits 24-28 M>>4.
//   A and B formats are independent: one operand may be fp16 and the other bf16 (tests/cuda/umma_probe.cu `mixed`).
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N, bool a_mn, bool b_mn, bool a_bf16, bool b_bf16) {
  return (1u << 4) | ((a_bf16 ? 1u : 0u) << 7) | ((b_bf16 ? 1u : 0u) << 10) | ((a_mn ? 1u : 0u) << 15) |
         ((b_mn ? 1u : 0u) << 16) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N, bool a_mn, bool b_mn, bool bf16) {
  return umma_idesc(M, N, a_mn, b_mn, bf16, bf16);
}
// D[tmem] (+)= A[smem] * B[smem]; issued by ONE thread.
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, bool accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accum)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]: A is a [128 lanes][K] 16-bit tile held in TMEM, two elements per 32-bit
// column (element 2j in the low half of column j), K = 16 per instruction = 8 columns.
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, bool accum) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"((uint32_t)accum)
      : "memory");
}
// Arrive on an mbarrier when all previously issued MMAs of this thread have completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}

// Byte offset of element (row, col) inside a dense 128B-swizzled [rows][64] 16-bit tile
// (the layout TMA SWIZZLE_128B writes and the descriptors above read): the 16-byte chunk
// index is XORed with (row mod 8).
__device__ __forceinline__ uint32_t swz128(int row, int col) {
  return (uint32_t)(row * 128 + ((((col >> 3) ^ row) & 7) << 4) + ((col & 7) << 1));
}

// Same for a dense 64B-swizzled [rows][32] 16-bit tile (TMA SWIZZLE_64B): chunk index XOR ((row >> 1) & 3).
__device__ __forceinline__ uint32_t swz64(int row, int col) {
  return (uint32_t)(row * 64 + ((((col >> 3) ^ (row >> 1)) & 3) << 4) + ((col & 7) << 1));
}

}  // namespace sm100

// ------------------------------------------------------------------- host: tensor maps
namespace sm100_host {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline EncodeTiledFn get_encode_fn() {
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

// true if a CUDA context is current on the calling thread (driver-level query: the runtime never says)
inline bool context_is_current() {
  typedef CUresult (*CtxGetCurrentFn)(CUcontext*);
  static CtxGetCurrentFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuCtxGetCurrent", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (CtxGetCurrentFn)p;
  }
  if (!fn) return false;
  CUcontext ctx = nullptr;
  return fn(&ctx) == CUDA_SUCCESS && ctx != nullptr;
}

// 4-D map over a (B, NH, S, D) 16-bit tensor with element strides (sb, sh, ss, 1);
// box = (64 cols, box_rows, 1, 1), 128B swizzle, out-of-bounds rows read as zero / are not written.
// box_cols = 64 -> 128B swizzle (default); box_cols = 32 -> 64B swizzle (head dim 32).
//
// cuTensorMapEncodeTiled costs about a microsecond and a forward + backward call pair needs 13 maps; a training step
// re-issues the same (pointer, shape, strides) signatures step after step (the caching allocator hands the same blocks
// back), so encoded maps are kept in a small per-thread direct-mapped cache: no lock, re-entrant, nothing shared
// between the caller's thread and the autograd threads (SURVEY.md section 8b "Threading").
struct MapKey {
  const void* ptr;
  int64_t sb, sh, ss;
  int32_t B, NH, S, D, box_rows, box_cols, bf16, pad;
};
inline int make_map_bhsd(CUtensorMap* map, const void* ptr, bool bf16, int B, int NH, int S, int D, int64_t sb,
                         int64_t sh, int64_t ss, int box_rows, int box_cols = 64) {
  constexpr int kSlots = 128;
  struct Slot {
    MapKey key;
    CUtensorMap map;
    bool valid;
  };
  static thread_local Slot cache[kSlots];
  MapKey key{ptr, sb, sh, ss, B, NH, S, D, box_rows, box_cols, bf16 ? 1 : 0, 0};
  uint64_t h = (uint64_t)(uintptr_t)ptr * 0x9E3779B97F4A7C15ull;
  h ^= ((uint64_t)(uint32_t)S << 32 | (uint32_t)D) * 0xC2B2AE3D27D4EB4Full + (uint64_t)ss * 31 + (uint64_t)box_rows;
  Slot& slot = cache[(h >> 32) % kSlots];
  if (slot.valid && memcmp(&slot.key, &key, sizeof(MapKey)) == 0) {
    *map = slot.map;
    return 0;
  }
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return -1;
  cuuint64_t dims[4] = {(cuuint64_t)D, (cuuint64_t)S, (cuuint64_t)NH, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)ss * 2, (cuuint64_t)sh * 2, (cuuint64_t)sb * 2};
  cuuint32_t box[4] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows, 1, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  if (((uintptr_t)ptr & 15) || (strides[0] & 15) || (strides[1] & 15) || (strides[2] & 15)) return -2;
  CUresult r = fn(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, (void*)ptr, dims,
                  strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  box_cols == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return (int)r;
  slot.key = key;
  slot.map = *map;
  slot.valid = true;
  return 0;
}

}  // namespace sm100_host
