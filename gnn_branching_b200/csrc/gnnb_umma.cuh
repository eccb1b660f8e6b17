// tcgen05 / TMEM / TMA building blocks shared by the tensor-core kernels (gnnb_tc.cu, gnnb_prop_tc.cu).
#pragma once

#include <cuda_fp16.h>
#include <stdio.h>
#include <string.h>

#include "gnnb_common.cuh"

namespace gnnb {
namespace tcx {

constexpr int TILE = 128;                        // nodes per tile = UMMA M
constexpr uint32_t WPLANE = 64 * 64 * 2;         // one 64(n) x 64(k) fp16 weight plane: 8 KB
constexpr uint32_t APLANE = TILE * 64 * 2;       // one A plane: 16 KB
constexpr uint32_t ABUF = 2 * APLANE;            // hi + lo

// byte offset of 16-byte chunk `chunk` (8 fp16 along K) of row `row` inside a K-major SWIZZLE_128B tile whose rows
// are 128 bytes (64 fp16): 8-row groups are 1024 bytes apart (SBO), chunks are XOR-swizzled with the row
__host__ __device__ inline uint32_t swz(uint32_t row, uint32_t chunk) {
    return (row >> 3) * 1024u + (row & 7u) * 128u + ((chunk ^ (row & 7u)) << 4);
}

// ---- operand precision ----------------------------------------------------------------------------
// Operands are split into two fp16 planes, x ~= hi + lo with hi = fp16(x), lo = fp16(x - hi): 22 significant bits,
// so the three products hi*hi + lo*hi + hi*lo carry ~2^-22 relative error (a bf16 split gives 2^-17, which left the
// scores only ~1.5x inside the 1e-4 parity bound).  fp16's narrow exponent is handled by keeping every activation
// operand scaled by ASCALE: ReLU and the linears are positively homogeneous, so the whole chain runs in the scaled
// domain with pre-scaled biases, and results are multiplied by AINV when they leave for global memory.
// |activation| >= 65504 / ASCALE = 524 288 overflows to inf -> NaN -> GNNB_ERR_NAN (never silent), or, with option "rescore",
// the subdomain is scored again in exact fp32 (gnnb_api.cu rescore_flagged).
constexpr float ASCALE = 0.125f;
constexpr float AINV = 8.0f;

inline void split_host(float x, uint16_t& hi, uint16_t& lo) {
    const __half h = __float2half_rn(x);
    const float rem = x - __half2float(h);
    const __half l = (rem == rem && rem - rem == 0.f) ? __float2half_rn(rem) : __float2half_rn(0.f);
    memcpy(&hi, &h, 2);
    memcpy(&lo, &l, 2);
}

// ---- PTX wrappers ---------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t a, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t a, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t a, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(a), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(mbar) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void named_bar(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void named_bar_arrive(int id, int nthreads) {
    asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(slot), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T, fp16 x fp16 -> fp32
__device__ __forceinline__ void umma(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]^T: the A operand is read from tensor memory (lane = row, 32-bit column j holds
// k = 2j in its low half and k = 2j + 1 in its high half; one K = 16 instruction reads 8 columns)
__device__ __forceinline__ void umma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
        "}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t mbar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
}
// 16 consecutive fp32 columns of this thread's TMEM lane (lane = accumulator row).  The load is asynchronous:
// tmem_wait16 must run on the same array before its values are read (the "+r" operands pin that order for the compiler)
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait16(uint32_t (&r)[16], float (&v)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;\n"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                   "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
                 :: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld16_sync(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    tmem_ld16(taddr, r);
    tmem_wait16(r, v);
}

// 16 consecutive 32-bit columns of this thread's TMEM lane <- registers (asynchronous: tmem_st_wait before the data is used)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};\n"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
          "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]) : "memory");
}
// one 32-bit column of this thread's TMEM lane
__device__ __forceinline__ void tmem_st1(uint32_t taddr, uint32_t v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t tmem_ld1_sync(uint32_t taddr) {
    uint32_t v;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];\ntcgen05.wait::ld.sync.aligned;" : "=r"(v) : "r"(taddr) : "memory");
    return v;
}
// register budget of the calling warpgroup (all 4 warps execute it): producers give registers back, the chain warpgroups take them
template <int N> __device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// L2 prefetch of a contiguous global range (one thread issues it; bytes is a multiple of 16)
__device__ __forceinline__ void prefetch_l2(const void* p, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}

// UMMA shared-memory descriptor: K-major, SWIZZLE_128B, 8-row groups 1024 B apart (cute::UMMA::SmemDescriptor)
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);          // start address, bits [0,14)
    d |= (uint64_t)1 << 16;                                 // leading byte offset (unused for swizzled K-major), [16,30)
    d |= (uint64_t)(1024u >> 4) << 32;                      // stride byte offset, bits [32,46)
    d |= (uint64_t)1 << 46;                                 // descriptor version (Blackwell), bits [46,48)
    d |= (uint64_t)2 << 61;                                 // layout type SWIZZLE_128B, bits [61,64)
    return d;
}
// K-major operand without swizzle ("piece-major" tile image): 16-byte pieces (8 fp16 along K) of consecutive rows are
// contiguous, so a core matrix (8 rows x 16 B) is 128 contiguous bytes; 8-row groups are `sbo` bytes apart and the
// pieces (K direction) `lbo` bytes apart (cute::UMMA::make_umma_desc<Major::K>, LayoutType::INTERLEAVE)
__device__ __forceinline__ uint64_t make_desc_nosw(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(lbo_bytes >> 4) << 16;
    d |= (uint64_t)(sbo_bytes >> 4) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}
// MN-major SWIZZLE_128B operand: 64-element (128 B) rows along N, 8 K-rows per 1024 B group (SBO), further 64-wide N
// blocks `lbo_bytes` apart (cute::UMMA::make_umma_desc<Major::MN>)
__device__ __forceinline__ uint64_t make_desc_mn(uint32_t smem_addr, uint32_t lbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)(lbo_bytes >> 4) << 16;
    d |= (uint64_t)(1024u >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// ---- tile images in global memory (private workspace formats of the tensor-core kernels) ------------------------------
// Every per-node tensor of the tensor-core path lives in tiles of 128 consecutive global rows (row = subdomain * n + node),
// 32 KB per tile = [fp16 hi plane 16 KB][fp16 lo plane 16 KB], values in the scaled domain (x ASCALE):
//   mu image  each plane is the K-major SWIZZLE_128B image (byte offset swz(row, chunk)): a row's 64 channels are 128
//             contiguous bytes (16-byte chunks XOR-permuted), written with one bulk store per tile, gathered row-wise;
//   nb image  each plane is piece-major (byte offset piece * 2048 + row * 16): rows of one piece are contiguous, so the
//             propagation epilogue (thread = row) stores coalesced and the update kernels read it as a no-swizzle A operand.
constexpr uint32_t NB_PIECE = TILE * 16;          // 2 KB: one 16-byte piece of all 128 rows

// shared -> global bulk copy (async proxy reads shared memory: generic-proxy writes need fence.proxy.async first)
__device__ __forceinline__ void bulk_s2g(void* dst, uint32_t src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// several bulk stores in one group: issue them with bulk_s2g_nocommit, then bulk_commit once
__device__ __forceinline__ void bulk_s2g_nocommit(void* dst, uint32_t src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// 16-byte asynchronous copy global -> shared (L2 only), zero-filled when !valid; completion is tracked by an mbarrier
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src, bool valid) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(valid ? 16u : 0u) : "memory");
}
__device__ __forceinline__ void cp_async16_sz(uint32_t dst, const void* src, uint32_t src_bytes) {      // src_bytes 16, or 0 = zero fill
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_arrive(uint32_t mbar) {      // arrives when this thread's earlier cp.async have landed
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(mbar) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
// wait until at most n (0 .. 7) of this thread's committed cp.async groups are pending (the instruction takes an immediate)
__device__ __forceinline__ void cp_async_wait_dyn(int n) {
    switch (n) {
        case 0: asm volatile("cp.async.wait_group 0;" ::: "memory"); break;
        case 1: asm volatile("cp.async.wait_group 1;" ::: "memory"); break;
        case 2: asm volatile("cp.async.wait_group 2;" ::: "memory"); break;
        case 3: asm volatile("cp.async.wait_group 3;" ::: "memory"); break;
        case 4: asm volatile("cp.async.wait_group 4;" ::: "memory"); break;
        case 5: asm volatile("cp.async.wait_group 5;" ::: "memory"); break;
        case 6: asm volatile("cp.async.wait_group 6;" ::: "memory"); break;
        default: asm volatile("cp.async.wait_group 7;" ::: "memory"); break;
    }
}
__device__ __forceinline__ void mbar_arrive(uint32_t mbar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(mbar) : "memory");
}

// Issuing tcgen05.mma / tcgen05.commit from warp-uniform code: every lane of the warp walks the (uniform) loop and one
// elected lane executes the instruction.  With operands that are uniform by data flow the compiler keeps descriptors in
// uniform registers and emits one UTCHMMA per MMA; a `if (lane == 0)` region instead makes every MMA a ~30-instruction
// sequence (per-thread 64-bit descriptor arithmetic, 5 R2UR, an ELECT / BRA.U.ANY loop), i.e. 150-220 cycles of issue per
// MMA against 32-128 cycles of tensor time (scripts/micro/mma_rate.cu).
__device__ __forceinline__ bool elect_one() {
    uint32_t p;
    asm volatile("{\n.reg .pred q;\nelect.sync _|q, 0xffffffff;\nselp.u32 %0, 1, 0, q;\n}" : "=r"(p));
    return p != 0;
}
// a value every lane holds identically, in a form the compiler can prove uniform (loaded data, threadIdx-derived warp ids)
__device__ __forceinline__ int uniform(int v) { return __shfl_sync(0xffffffffu, v, 0); }

// ---- programmatic dependent launch -----------------------------------------------------------------------------------
// The big kernels are launched with cudaLaunchAttributeProgrammaticStreamSerialization (launch_pdl below): a kernel may be
// scheduled while its predecessor in the stream is still draining, so its prologue (barrier init, tensor-memory allocation,
// the bulk loads of the constant weight planes) overlaps the predecessor's tail.  pdl_wait() blocks until the predecessor
// grid has completed and its writes are visible: NOTHING but constant parameters may be touched before it.  pdl_trigger()
// lets the successor be scheduled as soon as every CTA of this (single-wave) grid has started.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3((unsigned)block);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// instruction descriptor (cute::UMMA::InstrDescriptor): D fp32 (bits [4,6) = 1), A/B fp16 (format 0), both K-major, M = 128
__device__ __forceinline__ uint32_t make_idesc(uint32_t N) {
    return (1u << 4) | ((N >> 3) << 17) | ((uint32_t)(TILE >> 4) << 24);
}

__device__ __forceinline__ float relu_nan(float x) {      // F.relu keeps NaN: max.NaN propagates it (fmaxf would not)
    float y;
    asm("max.NaN.f32 %0, %1, 0f00000000;" : "=f"(y) : "f"(x));
    return y;
}

// (a, b) -> packed fp16x2 hi and lo words; element a sits at the lower address
__device__ __forceinline__ void split2(float a, float b, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(a, b);
    const __half2 l = __floats2half2_rn(a - __low2float(h), b - __high2float(h));
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

// ---- phase tracing (debug builds with -DGNNB_TRACE only; scripts/trace_build.sh) ---------------------------------
// One thread of one warpgroup records clock64() at fixed points of its first tiles and prints the deltas at kernel end.
#ifdef GNNB_TRACE
#define GNNB_TR_DECL long long tr_[16 * 12]; int tr_n_ = 0; const bool tr_on_ = (blockIdx.x == 1 && (threadIdx.x & 127) == 0 && (threadIdx.x >> 7) == 1)
#define GNNB_TR(i) do { if (tr_on_ && tr_n_ < 16) tr_[tr_n_ * 12 + (i)] = clock64(); } while (0)
#define GNNB_TR_NEXT() do { if (tr_on_ && tr_n_ < 16) ++tr_n_; } while (0)
#define GNNB_TR_PRINT(name, npts) do { if (tr_on_) { for (int a_ = 0; a_ < tr_n_; ++a_) { printf("TRACE %s it %d:", name, a_); \
    for (int b_ = 1; b_ < (npts); ++b_) printf(" %lld", tr_[a_ * 12 + b_] - tr_[a_ * 12 + b_ - 1]); \
    if (a_ + 1 < tr_n_) printf(" | next %lld", tr_[(a_ + 1) * 12] - tr_[a_ * 12 + (npts) - 1]); printf("\n"); } } } while (0)
#else
#define GNNB_TR_DECL
#define GNNB_TR(i) do {} while (0)
#define GNNB_TR_NEXT() do {} while (0)
#define GNNB_TR_PRINT(name, npts) do {} while (0)
#endif

}  // namespace tcx
}  // namespace gnnb
