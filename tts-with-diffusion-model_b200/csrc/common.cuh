// Shared device/host helpers for libvalle_b200.so (sm_100a only).
// Hand-written PTX wrappers for mbarrier, TMA (cp.async.bulk.tensor) and tcgen05/TMEM.
#pragma once
#include <atomic>
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/vb200.h"

namespace vb200 {

// ---------------------------------------------------------------- error plumbing (host)
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);
#define VB_CHECK_CUDA(expr)                                              \
  do {                                                                   \
    cudaError_t _e = (expr);                                             \
    if (_e != cudaSuccess) return ::vb200::cuda_fail(_e, #expr);         \
  } while (0)
#define VB_REQUIRE(cond, ...)                                            \
  do {                                                                   \
    if (!(cond)) {                                                       \
      ::vb200::set_error(__VA_ARGS__);                                   \
      return VB200_ERR_INVALID;                                          \
    }                                                                    \
  } while (0)

int num_sms();

// classifier GEMM with the reverse step as its epilogue (head_sample_tcgen05.cu)
int head_sample_fused(int32_t* x_out, const void* head_in, const void* W, const float* bias, const int32_t* x_t,
                      const int32_t* row_utt, const int32_t* t_utt, const int32_t* utt, const float* table,
                      int n_rows, int d, int n_levels, int K, int S, int tr, int noise, uint64_t seed,
                      int in_f16, const int32_t* known, cudaStream_t st);
int head_ce_fused(float* loss_out, const void* head_in, const void* W, const float* bias, const int32_t* targets,
                  int n_rows, int d, int n_levels, int K, int in_f16, cudaStream_t st);

// Programmatic dependent launch (PDL).  Every kernel of the denoise step goes through launch_pdl() and
// brackets its first access to memory that an earlier kernel produced (or still reads) with pdl_wait(), so
// that with the "programmatic stream serialization" attribute its CTAs may become resident and run their
// prologue (barrier init, TMEM allocation, tensor-map prefetch, TMA loads of STATIC data: the first ring of
// weight tiles) while the previous kernel drains.  Valid under stream capture too.
// Which launches carry the attribute is a bit mask (VB200_PDL, default 2 | 4 | 8 | 16 | 32), measured per class on
// the batch-1 denoise step (88 kernels, one graph replay; tools/latency_ab.py, same box):
//   4 | 8  GEMMs (QKV / FFN1 behind an AdaLN, the residual GEMMs behind attention / FFN1)   765 -> 735 us,
//          -> 722 us once the weight halves of the first ring are requested before the wait
//   32     fused classifier + reverse step                                                   -1.5 us
//   AdaLN as it is (eight small blocks per SM)                                               +17 us
//   attention as it is (two CTAs per SM)                                                     +46 us
//   1      every launch (what rounds 1 and 2 first measured: 832 against 797 us, "PDL is slower")
// The difference is CTA placement: an early-launched grid takes SM slots as they free up.  The tensor-core
// GEMMs fit one CTA per SM, so nothing changes for them but the start time; attention (two CTAs per SM) and
// AdaLN (eight blocks) get PACKED onto the first SMs that drain instead of being spread breadth-first over
// idle SMs, and a one-wave launch then runs at half speed.  Hence, for grids that fit the SMs once, those two
// kernels ask for 116 KB of dynamic shared memory they do not use — one CTA per SM — and then gain from the
// early launch like the GEMMs:
//   2      AdaLN, padded                                                                     721 -> 717 us
//   16     attention, padded                                                                 721 -> 712 us (both: 708)
// Larger grids (more than one utterance) keep stream order for these two (measured neutral to slightly
// negative at 32 utterances); the GEMM mask gives 12.56 -> 12.50 ms per step there, 97.2 -> 96.8 ms at 256.
// cudaFuncSetAttribute is per DEVICE: each launch site remembers which devices it has configured (a
// process that drives several GPUs would otherwise launch with the 48 KB default on the second one).
#define VB_CONFIGURE_SMEM(kern, bytes)                                                                   \
  do {                                                                                                   \
    static std::atomic<uint64_t> vb_cfg_done{0};                                                         \
    int vb_cfg_dev = 0;                                                                                  \
    VB_CHECK_CUDA(cudaGetDevice(&vb_cfg_dev));                                                           \
    const uint64_t vb_cfg_bit = 1ull << (vb_cfg_dev & 63);                                               \
    if (!(vb_cfg_done.load(std::memory_order_acquire) & vb_cfg_bit)) {                                   \
      VB_CHECK_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));     \
      vb_cfg_done.fetch_or(vb_cfg_bit, std::memory_order_release);                                       \
    }                                                                                                    \
  } while (0)
bool pdl_enabled();
// VB200_PDL is a bit mask: 1 = every launch; 2 = AdaLN padded to one block per SM; 4 = GEMMs behind an AdaLN (QKV,
// FFN1); 8 = residual GEMMs; 16 = attention padded to one CTA per SM; 32 = fused classifier + reverse step;
// 64 / 128 = attention / AdaLN grids larger than the SM count.  A launch site names its class through PdlTag
// before calling launch_pdl().
int pdl_mask();
extern thread_local int g_pdl_tag;
struct PdlTag {
  int prev;
  explicit PdlTag(int t) : prev(g_pdl_tag) { g_pdl_tag = t; }
  ~PdlTag() { g_pdl_tag = prev; }
};
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              int cluster_x, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster_x;
    attr[n].val.clusterDim.y = 1;
    attr[n].val.clusterDim.z = 1;
    ++n;
  }
  if (pdl_mask() & (1 | g_pdl_tag)) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  cfg.attrs = attr;
  cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// Encodes a 2D row-major tensor map: dims {inner, outer}, box {box_inner, box_outer},
// SWIZZLE_128B (box_inner * element size must be 128 bytes), zero fill / clipping out of bounds.
int make_tmap_2d(CUtensorMap* out, vb200_dtype dtype, const void* gptr, uint64_t inner,
                 uint64_t outer, uint64_t row_stride_bytes, uint32_t box_inner, uint32_t box_outer);
// Same, memoised on (pointer, dtype, shape, box): tensor maps are pure functions of their inputs.
int cached_tmap(CUtensorMap* out, vb200_dtype dtype, const void* ptr, uint64_t inner,
                uint64_t outer, uint64_t stride_bytes, uint32_t box_inner, uint32_t box_outer);

// ---------------------------------------------------------------- device PTX wrappers
// PDL, device side: launch_dependents lets the next kernel's CTAs be scheduled as soon as this grid
// leaves room; wait blocks until every kernel this one depends on has completed and flushed.  Both
// are no-ops for a kernel launched without the attribute.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

#ifdef __CUDACC__

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}

// ---- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Non-blocking poll (try_wait may suspend the warp for a while; this never does).
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (launch failure reported to the host) instead of hanging
// the GPU box.  try_wait suspends in hardware, so the bound is generous in wall time.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > (1u << 24)) __trap();
  }
}

// ---- TMA
__device__ __forceinline__ void prefetch_l1(const void* p) {
  asm volatile("prefetch.global.L1 [%0];" ::"l"(p));
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                            int32_t c_inner, int32_t c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)),
      "r"(c_inner), "r"(c_outer)
      : "memory");
}

// smem tile -> global (bulk async group); out-of-bounds parts of the box are clipped
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* m, const void* smem_src,
                                             int32_t c_inner, int32_t c_outer) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c_inner),
               "r"(c_outer)
               : "memory");
}
// global += smem tile (element-wise add performed at L2)
__device__ __forceinline__ void tma_reduce_add_2d(const CUtensorMap* m, const void* smem_src,
                                                  int32_t c_inner, int32_t c_outer) {
  asm volatile("cp.reduce.async.bulk.tensor.2d.global.shared::cta.add.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(smem_src)), "r"(c_inner),
               "r"(c_outer)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_read() {   // smem source reusable
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void tma_store_wait_all() {    // writes complete
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}

// ---- tcgen05 / TMEM
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
// D[tmem] (+)= A[smem] * B[smem]; kind::f16 (bf16/fp16 in, fp32 accumulate)
__device__ __forceinline__ void umma_ss(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void umma_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b,
                                        uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread completed.
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_st_wait() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp gets lane (base_lane + i).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
      "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]),
        "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]),
        "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
      "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]),
      "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]),
      "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]),
      "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
      "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}

// ---- CTA-pair (cta_group::2) forms: two CTAs of a cluster drive one 256-row MMA
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// TMA load into this CTA's smem whose bytes are counted on the barrier of the pair's leader CTA
// (bit 24 of a shared::cluster address selects the peer; clearing it addresses CTA 0 of the pair).
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const CUtensorMap* m, uint64_t* bar,
                                                 int32_t c_inner, int32_t c_outer) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & 0xFEFFFFFFu),
      "r"(c_inner), "r"(c_outer)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_slot, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                   smem_u32(smem_slot)),
               "r"(ncols)
               : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// D[tmem of both CTAs] (+)= A[smem, 128 rows per CTA] * B[smem, N/2 rows per CTA]; issued by the leader
__device__ __forceinline__ void umma_ss_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                             uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on the barrier at this smem offset in BOTH CTAs once the leader's prior MMAs retired
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
  const uint16_t mask = 3;
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
      ::"r"(smem_u32(bar)), "h"(mask)
      : "memory");
}
// arrive on the barrier at the same smem offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t rank) {
  uint32_t remote;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(rank));
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}

// ---- UMMA descriptors (cute/arch/mma_sm100_desc.hpp bit layout, re-derived by hand)
// K-major operand tile, rows of 64 bf16 (=128 B) stored with the TMA SWIZZLE_128B pattern:
// 8-row groups are 1024 B apart (SBO), LBO is ignored for swizzled K-major (canonical value 1).
__device__ __forceinline__ uint64_t umma_desc_kmajor_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);   // start address  [0,14)
  d |= static_cast<uint64_t>(1) << 16;                      // LBO >> 4       [16,30)
  d |= static_cast<uint64_t>(1024 >> 4) << 32;              // SBO >> 4       [32,46)
  d |= static_cast<uint64_t>(1) << 46;                      // descriptor version (sm_100)
  d |= static_cast<uint64_t>(2) << 61;                      // SWIZZLE_128B
  return d;
}
// MN-major operand tile: rows (one per k) of 64 contiguous bf16 along MN (=128 B) with
// SWIZZLE_128B; 8-k groups 1024 B apart (SBO); LBO = stride between 64-element MN chunks.
__device__ __forceinline__ uint64_t umma_desc_mnmajor_sw128(uint32_t smem_addr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
  d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}
// Instruction descriptor for kind::f16 with bf16 A/B and fp32 D.  A and B carry separate format
// fields (0 = F16, 1 = BF16), but the hardware only takes them EQUAL: fp16 rows against bf16 weights
// raises an illegal-instruction fault on B200 (measured).  Clearing kIdescBf16 makes both operands
// fp16 — used where the activation range is safe (11 significand bits against 8), see DESIGN.md §4.
constexpr uint32_t kIdescBf16 = (1u << 7) | (1u << 10);
__host__ __device__ constexpr uint32_t umma_idesc_bf16(uint32_t M, uint32_t N, bool a_mn_major,
                                                       bool b_mn_major) {
  return (1u << 4)                         // D format: F32
         | kIdescBf16                      // A and B format: BF16
         | ((a_mn_major ? 1u : 0u) << 15)  // A major
         | ((b_mn_major ? 1u : 0u) << 16)  // B major
         | ((N >> 3) << 17)                // N >> 3
         | ((M >> 4) << 24);               // M >> 4
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t v;                              // saturating: an outlier becomes +-65504, never inf
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(v) : "f"(hi), "f"(lo));
  return v;
}
// 16-bit activations: fp16 or bf16 chosen at run time (warp-uniform flag)
__device__ __forceinline__ uint32_t pack_act16x2(float lo, float hi, bool f16) {
  return f16 ? pack_f16x2(lo, hi) : pack_bf16x2(lo, hi);
}

// Packed fp32 pairs (sm_100 FFMA2 / FADD2): one issue slot per two lanes' worth of fp32 work
// (tools/fma2_bench.cu: same flops per clock as FFMA, half the instructions).
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t ffma2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t fadd2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
constexpr float kEps = 1.0e-6f;          // ar_discrete.py:276

// ---------------------------------------------------------------- Philox4x32-10
struct Philox {
  uint32_t k0, k1;
  __device__ __forceinline__ uint4 operator()(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3) const {
    uint32_t a = k0, b = k1;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
      const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
      c0 = hi1 ^ c1 ^ a;
      c1 = lo1;
      c2 = hi0 ^ c3 ^ b;
      c3 = lo0;
      a += 0x9E3779B9u;
      b += 0xBB67AE85u;
    }
    return make_uint4(c0, c1, c2, c3);
  }
};
__device__ __forceinline__ float u01(uint32_t x) { return (x >> 8) * 5.9604644775390625e-8f; }
__device__ __forceinline__ float exp2f_fast(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
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

#endif  // __CUDACC__

// AdaLN of one row (base.py:145-158) for d = 256 * NV, one warp per row: lane owns elements
// [i*256 + lane*8, +8) of the row in v[i][*]; g / bt are the matching slices of exp(log gamma) and
// beta.
template <int NV>
__device__ __forceinline__ void adaln_row_finish(const float (&v)[NV][8], const float (&g)[NV][8],
                                                 const float (&bt)[NV][8], __nv_bfloat16* orow, int lane,
                                                 float eps, float k, float c, bool f16 = false) {
  constexpr int d = NV * 256;
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i)
#pragma unroll
    for (int e = 0; e < 8; ++e) s += v[i][e];
  const float mean = warp_sum(s) * (1.0f / d);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i)
#pragma unroll
    for (int e = 0; e < 8; ++e) { const float dv = v[i][e] - mean; q += dv * dv; }
  const float rstd = rsqrtf(warp_sum(q) * (1.0f / d) + eps);
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    float y[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) {
      float h = (v[i][e] - mean) * rstd;
      h = c * (1.f - k * h) * h;
      y[e] = fmaf(g[i][e], h, bt[i][e]);
    }
    uint4 o;
    o.x = pack_act16x2(y[0], y[1], f16); o.y = pack_act16x2(y[2], y[3], f16);
    o.z = pack_act16x2(y[4], y[5], f16); o.w = pack_act16x2(y[6], y[7], f16);
    *reinterpret_cast<uint4*>(orow + i * 256 + lane * 8) = o;
  }
}
// loads the [gamma | beta] slices of table row `lvl` (2d floats per row) for this lane
template <int NV>
__device__ __forceinline__ void adaln_load_params(const float* __restrict__ table, int lvl, int lane,
                                                  float (&g)[NV][8], float (&bt)[NV][8]) {
  constexpr int d = NV * 256;
  const float* gp = table + static_cast<size_t>(lvl) * 2 * d;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const float4 g0 = __ldg(reinterpret_cast<const float4*>(gp + i * 256 + lane * 8));
    const float4 g1 = __ldg(reinterpret_cast<const float4*>(gp + i * 256 + lane * 8 + 4));
    const float4 b0 = __ldg(reinterpret_cast<const float4*>(gp + d + i * 256 + lane * 8));
    const float4 b1 = __ldg(reinterpret_cast<const float4*>(gp + d + i * 256 + lane * 8 + 4));
    g[i][0] = g0.x; g[i][1] = g0.y; g[i][2] = g0.z; g[i][3] = g0.w;
    g[i][4] = g1.x; g[i][5] = g1.y; g[i][6] = g1.z; g[i][7] = g1.w;
    bt[i][0] = b0.x; bt[i][1] = b0.y; bt[i][2] = b0.z; bt[i][3] = b0.w;
    bt[i][4] = b1.x; bt[i][5] = b1.y; bt[i][6] = b1.z; bt[i][7] = b1.w;
  }
}

}  // namespace vb200
