// Shared helpers for the roomslam_b200 sm_100a kernels: error plumbing for the C-ABI, and thin
// inline-PTX wrappers for mbarrier, TMA (cp.async.bulk.tensor) and tcgen05 / TMEM.
#pragma once

#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

namespace rs {

// ---- C-ABI error plumbing -------------------------------------------------------------------
void set_error(const char* fmt, ...);
int check_device_sm100();  // 0 when the current device is sm_100; sets the error otherwise
void count_launch(int n = 1);  // bookkeeping for rs_launch_count(): kernels launched by this library

#define RS_CUDA_OK(expr)                                                                    \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            rs::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return 2;                                                                       \
        }                                                                                   \
    } while (0)

#define RS_REQUIRE(cond, ...)                                                               \
    do {                                                                                    \
        if (!(cond)) {                                                                      \
            rs::set_error(__VA_ARGS__);                                                     \
            return 1;                                                                       \
        }                                                                                   \
    } while (0)

// Encodes a 2-D row-major tensor map (driver entry point fetched at run time; no -lcuda needed).
// dims/box are {inner, outer}; row_stride_bytes is the outer stride.  Returns 0 on success.
int make_tmap_2d(CUtensorMap* out, const void* base, CUtensorMapDataType dtype, uint32_t elem_bytes,
                 uint64_t inner, uint64_t outer, uint64_t row_stride_bytes, uint32_t box_inner,
                 uint32_t box_outer, CUtensorMapSwizzle swizzle);

// ---- deterministic mode (rs_set_deterministic) ----------------------------------------------
// A reduction split over CTAs then stores one partial per split into a workspace instead of adding it to the output with
// atomics, and slot_sum adds the partials in ascending split order.  The split of a reduction may depend on the shape
// only: kDetSplitSms stands in for the SM count wherever the default path sizes a split by num_sms().
bool deterministic();
constexpr int kDetSplitSms = 148;

// out[r * ldo + c] = (accumulate ? out[r * ldo + c] : 0) + parts[0][r * cols + c] + parts[1][...] + ..., slot s at
// parts + s * part_stride.  Up to kMaxSlotSums outputs of different shapes in one launch.
template <typename T>
struct SlotSum {
    const T* parts;
    T* out;
    long long ldo;
    int rows, cols;
};
constexpr int kMaxSlotSums = 64;
template <typename T>
int slot_sum(const SlotSum<T>* jobs, int n_jobs, int n_parts, long long part_stride, bool accumulate, cudaStream_t stream);

// Workspace allocated in stream order on the call's stream and freed in stream order when it goes out of scope.
struct StreamScratch {
    void* p = nullptr;
    cudaStream_t stream;
    explicit StreamScratch(cudaStream_t s) : stream(s) {}
    ~StreamScratch() { if (p) cudaFreeAsync(p, stream); }
    cudaError_t alloc(size_t bytes) { return cudaMallocAsync(&p, bytes, stream); }
    template <typename T> T* as() const { return static_cast<T*>(p); }
};

// ---- device-side PTX ------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
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
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}

// TMA: 2-D tiled load global -> shared, completion on an mbarrier (SASS: UTMALDG).
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c_inner,
                                            int c_outer) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c_inner),
        "r"(c_outer)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d_hint(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar,
                                                 int c_inner, int c_outer, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint "
        "[%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar)), "r"(c_inner),
        "r"(c_outer), "l"(policy)
        : "memory");
}
// TMA: 2-D tiled store shared -> global (SASS: UTMASTG).
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* tmap, const void* smem_src, int c_inner, int c_outer) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(smem_src)), "r"(c_inner), "r"(c_outer)
                 : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() {
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
template <int N>
__device__ __forceinline__ void tma_store_wait() {
    asm volatile("cp.async.bulk.wait_group %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b32 r;\n\t"
        "elect.sync r|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// ---- tcgen05 / TMEM ---------------------------------------------------------------------------
// Allocation is done by ONE full warp; the base address lands in shared memory.
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot) {
    static_assert(kCols >= 32 && kCols <= 512 && (kCols & (kCols - 1)) == 0, "TMEM columns: power of two in [32,512]");
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)),
                 "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
// tcgen05.commit: the mbarrier gets one arrival once every previously issued MMA of this thread retired.
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], bf16 x bf16 -> fp32, issued by ONE thread (SASS: UTCHMMA).
__device__ __forceinline__ void tc_mma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// TMEM -> registers: this warp's 32 lanes x 32 consecutive fp32 columns (SASS: LDTM).
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
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
__device__ __forceinline__ void tmem_ld_32x32b_x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// registers -> TMEM: this warp's 32 lanes x 16 consecutive 32-bit columns (SASS: STTM).
__device__ __forceinline__ void tmem_st_32x32b_x16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// Bulk prefetch of a contiguous global range into L2 (no registers, no completion tracking).  bytes % 16 == 0.
__device__ __forceinline__ void l2_prefetch(const void* gptr, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(reinterpret_cast<uint64_t>(gptr)), "r"(bytes) : "memory");
}

// Shared-memory matrix descriptor, K-major operand stored as rows of exactly 128 bytes (64 bf16) with
// the 128-byte swizzle (what TMA SWIZZLE_128B writes): 8-row groups are 1024 B apart (SBO), LBO unused.
// Bit layout follows the sm_100 descriptor format (version field = 1, layout type 2 = SWIZZLE_128B).
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);       // start address, bits [0,14)
    d |= static_cast<uint64_t>(0) << 16;                           // leading byte offset (unused for SW128 K-major)
    d |= static_cast<uint64_t>(1024 >> 4) << 32;                   // stride byte offset, bits [32,46)
    d |= static_cast<uint64_t>(1) << 46;                           // descriptor version (Blackwell)
    d |= static_cast<uint64_t>(2) << 61;                           // SWIZZLE_128B
    return d;
}
// Same for an MN-major operand: 64 MN-elements (128 B) contiguous per K row, 8 K-rows per 1024-B atom.
// lbo_bytes = distance between atoms along MN, sbo_bytes = distance between 8-row groups along K.
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    d |= static_cast<uint64_t>(2) << 61;
    return d;
}
// No-swizzle ("interleaved") descriptors: the operand is stored as 8-row x 16-byte core matrices (128 contiguous
// bytes each).  K-major: lbo = bytes between the two 16-byte K chunks of one K=16 step, sbo = bytes between
// 8-row groups along M/N.  MN-major: lbo = bytes between 8-row groups along K, sbo = bytes between 16-byte chunks
// along M/N.  This is the layout of the library's tile-major activations: [chunk][128 rows][8 bf16].
__device__ __forceinline__ uint64_t umma_desc_noswz(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr & 0x3FFFF) >> 4);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= static_cast<uint64_t>(1) << 46;
    return d;
}
// 1-D bulk copy global -> shared with mbarrier completion (SASS: UBLKCP).  bytes % 16 == 0, 16-byte aligned.
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// Instruction descriptor for kind::f16 with bf16 A/B, fp32 accumulate.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(uint32_t M, uint32_t N, uint32_t a_mn_major, uint32_t b_mn_major) {
    return (1u << 4)                 // D format: F32
           | (1u << 7)               // A format: BF16
           | (1u << 10)              // B format: BF16
           | (a_mn_major << 15)      // A major: 0 = K, 1 = MN
           | (b_mn_major << 16)      // B major
           | ((N >> 3) << 17)        // N / 8
           | ((M >> 4) << 24);       // M / 16
}

// ---- CTA pair (thread-block cluster of 2 on one TPC, tcgen05 cta_group::2) ---------------------------------------
// One thread of the even CTA issues an MMA that spans both SMs: each CTA supplies its own rows of A and its half
// of the N rows of B from the SAME shared-memory offsets; each CTA's TMEM receives its own rows of D.
//   M = 256: 128 rows per CTA, lane = row, all N columns ("4x1");
//   M = 128:  64 rows per CTA, lane = row + 64 * (n >= N/2), column = n mod N/2 ("2x2": all 128 lanes busy).
// (layouts verified on hardware by tools/pair_probe.cu)
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `smem_addr` (a shared::cta address of this CTA) in the CTA of rank `rank`
__device__ __forceinline__ uint32_t mapa_cluster(uint32_t smem_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
    return r;
}
// Arrival on a barrier of another CTA of the cluster.  Default semantics (release at CTA scope), as CUTLASS's 2-SM
// kernels use: what the arrival publishes here are this CTA's OWN shared-memory writes, already fenced into the async
// proxy, for this SM's own tensor core.  A cluster-scope release compiles to MEMBAR.ALL.GPU + CCTL.IVALL, which waits
// for every global store of the step (~1000 cycles on the per-step critical path, ncu: stall_membar).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) { mbar_wait(bar, parity); }
template <uint32_t kCols>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_slot) {      // the same warp of BOTH CTAs executes this
    static_assert(kCols >= 32 && kCols <= 512 && (kCols & (kCols - 1)) == 0, "TMEM columns: power of two in [32,512]");
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <uint32_t kCols>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                                 uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// one arrival on the mbarrier at this shared-memory offset in BOTH CTAs once every MMA issued so far has retired
__device__ __forceinline__ void tc_commit_pair(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(static_cast<uint16_t>(3))
                 : "memory");
}

// cta_group::1 commit that arrives on the mbarrier at this shared-memory offset in every CTA of `cta_mask` (cluster ranks)
__device__ __forceinline__ void tc_commit_mc(uint64_t* bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(cta_mask)
                 : "memory");
}
// 1-D bulk copy global -> the same shared-memory offset of every CTA in `cta_mask`; each destination CTA's mbarrier (same
// offset) receives the complete_tx of the bytes written there
__device__ __forceinline__ void bulk_load_mc(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar, uint16_t cta_mask) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1], %2, [%3], %4;"
                 ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar)), "h"(cta_mask)
                 : "memory");
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

#endif  // __CUDACC__

}  // namespace rs
