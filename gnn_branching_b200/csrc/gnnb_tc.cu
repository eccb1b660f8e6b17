// Per-node MLP kernels on the 5th-generation tensor cores (GNNB_MATH_TC_FP16X3) — the product path.
//
// Every dense layer of the GNN with K >= 64 is a [128 nodes x K] x [K x N] GEMM per tile, issued as
// tcgen05.mma (cta_group::1, kind::f16, M = 128, N = 64 / 128 / 192, K = 16 per instruction) with fp32
// accumulators in tensor memory.  fp32 accuracy (scores within 1e-4, BASELINE.json) comes from an fp16 hi/lo
// split of BOTH operands and three MMAs per K step:  x*w ~= xh*wh + xl*wh + xh*wl  (error ~2^-22 per product;
// see gnnb_umma.cuh for the scaled operand domain that keeps fp16 in range).
//
// Algebra that shortens the per-tile chain (exact up to fp32 rounding; composed on the host in double):
//   * two linears with nothing but a bias between them are one linear.  The reference computes
//       mu = W4_2 relu(W4 [relax, e] + b4),  e = W3_2 relu(W3 [nb r0, nb r1] + b3) + b3_2,
//       relax = amb (W1_1 h1 + b1_1)                                              (graph_conv.py:153-181, 273-347)
//     so with W4 = [W4a | W4b]:  W4 [relax, e] + b4 = amb (Wr h1 + br) + Wc h3 + bc,  Wr = W4a W1_1, br = W4a b1_1,
//     Wc = W4b W3_2, bc = b4 + W4b b3_2.  The relax kernel therefore emits relax' = amb (Wr h1 + br) directly (the
//     round-independent part of the fc4 / bc4 pre-activation), and the update kernel is three GEMMs per tile:
//       D = nb [W3a; W3b]^T (N = 128) -> h3 = relu(r0 Da + r1 Db + b3) -> D = h3 Wc^T -> g = relu(D + relax' + bc)
//       -> D = g W4_2^T -> mu = (D + b4_2) (r0 != 0)   [-> score head on the last backward sweep];
//   * row scalings of GEMM *inputs* move to the epilogue by linearity (SURVEY §8a fact 3): [nb r0, nb r1] W3^T is one
//     N = 128 MMA, bc2's [s1, -d2 s1, d1 s1] input three N = 64 MMAs that share one A operand (summed in registers).
//
// Rows are in slot order (gnnb_common.cuh RowMap): a tile is 128 slots of one subdomain = one tile of the propagation
// plans; the caller's node-order arrays (bounds, duals, primals, scores) are reached through node_of_slot.
//
// Launch: programmatic dependent launch (gnnb_umma.cuh launch_pdl): the prologue (barriers, tensor memory, weight planes) of a
// kernel overlaps the tail of its predecessor; pdl_wait() precedes the first access to anything a predecessor wrote.
//
// Structure of a CTA (1 per SM, persistent over work items = 4 subdomains x tile, one tile per warpgroup): 4 warpgroups
// of 128 threads; the stage's weights sit in shared memory for the CTA's lifetime as fp16 hi/lo planes in the UMMA
// K-major SWIZZLE_128B image (repacked once on the host, landed with one cp.async.bulk per linear); each warpgroup
// owns one 128-slot tile at a time with 128 tensor-memory columns, a 32 KB shared-memory buffer and two mbarriers, and
// walks the chain of its tile sequentially:
//   GEMM (the warpgroup's first warp walks the issue code uniformly, one elected lane issues 3 x 4 tcgen05.mma +
//   tcgen05.commit: 12 back-to-back UTCHMMA, gnnb_umma.cuh elect_one) -> everyone waits on the mbarrier -> tcgen05.ld ->
//   bias / ReLU / row scaling in registers (thread = row = TMEM lane) -> fp16 hi/lo split -> tcgen05.st of the next
//   A operand straight back into tensor memory -> tcgen05.wait::st + fence + warpgroup barrier -> next GEMM ...
// Only the first GEMM of the update chain reads its A operand from shared memory (the nb tile image, one 32 KB
// cp.async.bulk, used as a no-swizzle K-major operand); every chained GEMM takes A from tensor memory (the ".ts" form
// of tcgen05.mma), so intermediate activations never touch shared memory.  The same 32 KB buffer then stages the
// tile's result as the mu image (conflict-free swizzled 16-byte stores) and leaves with one bulk store; the next
// tile's nb image is requested once the store has read the buffer (it was prefetched to L2 a tile earlier, as are the
// row's relax' pieces and bounds).  The warpgroups are independent, so one tile's epilogue overlaps the others' MMAs.
//
// Private workspace layouts (produced and consumed only by the tensor-core kernels; gnnb_umma.cuh):
//   nb       per tile the A-operand image itself, [hi plane 16 KB][lo plane 16 KB] piece-major, scaled by ASCALE —
//            written by the propagation kernel, loaded with one 32 KB cp.async.bulk;
//   mu       per tile [hi plane][lo plane] K-major SWIZZLE_128B (a row's 64 channels = 128 contiguous bytes), bulk-stored;
//   relax'   ambiguous rows only, compacted in row order: [tile][16 channel quads][128 slots][4] fp32 (scaled domain).
#include "gnnb_prop_body.cuh"
#include "gnnb_umma.cuh"

namespace gnnb {
namespace {

using namespace tcx;

// ---- warpgroup context ------------------------------------------------------------------------------
// Tensor-memory map of a warpgroup (128 columns): [0, 64) the A operand of the chained GEMMs — fp16 hi/lo pairs written by
// the epilogues with tcgen05.st, K step ks at columns [16 ks, 16 ks + 8) (hi) and [16 ks + 8, 16 ks + 16) (lo) — and
// [64, 128) the fp32 accumulator of a 64-wide GEMM.  The first GEMM of the update chain (N = 128, A = nb from shared
// memory) accumulates into [0, 128); its epilogue overwrites the columns it has consumed with the next A operand in place.
constexpr uint32_t ACOL = 0, DCOL = 64, WG_COLS = 128;

struct WG {
    uint32_t land;              // shared address of this warpgroup's 32 KB landing buffer (TMA'd nb tile image: hi, lo plane)
    uint32_t mbar_mma, mbar_tma;
    uint32_t ph_mma, ph_tma;
    uint32_t tmem;              // TMEM address: lane base of this warp, first column of this warpgroup
    uint32_t tmem0;             // lane 0, first column of this warpgroup (MMA operand / accumulator addresses)
    uint32_t acol;              // first column of the A operand of the chained GEMMs, relative to tmem / tmem0
    int t;                      // thread index within the warpgroup = row of the tile this thread owns
    int bar_threads;            // threads that walk the chain of one tile together: 128 (one warpgroup) or 256 (k_tc_fused: two, half the columns each)
    int wg;
    bool lead_warp;             // first warp of the warpgroup (warp-uniform): it issues the warpgroup's MMAs, one elected lane
};

__device__ __forceinline__ void wg_barrier(const WG& c) { named_bar(1 + c.wg, c.bar_threads); }

// 3 passes x 4 K steps with the A operand in tensor memory (issued by one thread)
__device__ __forceinline__ void issue_ts(const WG& c, uint32_t b_hi, uint32_t b_lo, uint32_t N, uint32_t dcol, bool accumulate) {
    const uint32_t idesc = make_idesc(N);
    const uint32_t d = c.tmem0 + dcol, a = c.tmem0 + c.acol;
#pragma unroll
    for (int pass = 0; pass < 3; ++pass) {
        const uint64_t bd = make_desc(pass == 2 ? b_lo : b_hi);
#pragma unroll
        for (int k = 0; k < 4; ++k)          // 16 fp16 along K per instruction: 32 bytes of B, 8 columns of A
            umma_ts(d, a + 16 * k + (pass == 1 ? 8 : 0), bd + 2 * k, idesc, (accumulate || pass > 0 || k > 0) ? 1u : 0u);
    }
}
// the same with the A operand in the landing buffer: the nb tile image, piece-major without swizzle (gnnb_umma.cuh)
__device__ __forceinline__ void issue_ss(const WG& c, uint32_t b_hi, uint32_t b_lo, uint32_t N, uint32_t dcol, bool accumulate) {
    const uint32_t idesc = make_idesc(N);
    const uint32_t d = c.tmem0 + dcol;
#pragma unroll
    for (int pass = 0; pass < 3; ++pass) {
        const uint64_t ad = make_desc_nosw(pass == 1 ? c.land + APLANE : c.land, NB_PIECE, 128u);
        const uint64_t bd = make_desc(pass == 2 ? b_lo : b_hi);
#pragma unroll
        for (int k = 0; k < 4; ++k)          // one K step = two pieces = 2 * NB_PIECE bytes of A
            umma(d, ad + (uint64_t)(k * ((2 * NB_PIECE) >> 4)), bd + 2 * k, idesc, (accumulate || pass > 0 || k > 0) ? 1u : 0u);
    }
}

// every thread: its tensor-memory accesses (A stores, accumulator loads) are complete and ordered before the MMAs
__device__ __forceinline__ void gemm_sync(const WG& c) {
    tmem_st_wait();
    tc_fence_before();
    wg_barrier(c);
}
__device__ __forceinline__ void gemm_finish(WG& c) {
    mbar_wait(c.mbar_mma, c.ph_mma);
    c.ph_mma ^= 1u;
    tc_fence_after();
}
// D[dcol, dcol + N) = A(tmem) W^T
__device__ __forceinline__ void gemm_ts_start(WG& c, uint32_t b_hi, uint32_t b_lo, uint32_t N, uint32_t dcol, bool accumulate = false) {
    gemm_sync(c);
    if (c.lead_warp) {          // uniform operands + one elected lane: 12 back-to-back UTCHMMA (gnnb_umma.cuh, elect_one)
        tc_fence_after();
        if (elect_one()) {
            issue_ts(c, b_hi, b_lo, N, dcol, accumulate);
            umma_commit(c.mbar_mma);
        }
        __syncwarp();
    }
}
__device__ __forceinline__ void gemm_ts(WG& c, uint32_t b_hi, uint32_t b_lo, uint32_t N, uint32_t dcol, bool accumulate = false) {
    gemm_ts_start(c, b_hi, b_lo, N, dcol, accumulate);
    gemm_finish(c);
}
// D[dcol, dcol + N) = A(landing buffer, after its TMA has completed) W^T
__device__ __forceinline__ void gemm_ss(WG& c, uint32_t b_hi, uint32_t b_lo, uint32_t N, uint32_t dcol, bool accumulate = false) {
    gemm_sync(c);
    if (c.lead_warp) {
        tc_fence_after();
        mbar_wait(c.mbar_tma, c.ph_tma);
        if (elect_one()) {
            issue_ss(c, b_hi, b_lo, N, dcol, accumulate);
            umma_commit(c.mbar_mma);
        }
        __syncwarp();
    }
    c.ph_tma ^= 1u;
    gemm_finish(c);
}

// 16 consecutive features [16 ks, 16 ks + 16) of this thread's row -> A operand columns of K step ks
__device__ __forceinline__ void a_store16(const WG& c, int ks, const float (&v)[16]) {
    uint32_t w[16];
#pragma unroll
    for (int i = 0; i < 8; ++i) split2(v[2 * i], v[2 * i + 1], w[i], w[8 + i]);
    tmem_st16(c.tmem + c.acol + 16 * ks, w);
}

__device__ __forceinline__ float4 lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ void lds16(const float* p, float (&b)[16]) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float4 x = lds4(p + 4 * i);
        b[4 * i] = x.x; b[4 * i + 1] = x.y; b[4 * i + 2] = x.z; b[4 * i + 3] = x.w;
    }
}

// read-only global loads the compiler must not sink past the MMA waits (they are issued early to hide DRAM latency)
__device__ __forceinline__ float4 ldg4_now(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
__device__ __forceinline__ float ldg1_now(const float* p) {
    float v;
    asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ int ldgi_now(const int32_t* p) {
    int v;
    asm volatile("ld.global.nc.s32 %0, [%1];" : "=r"(v) : "l"(p));
    return v;
}

// accumulator columns [dcol, dcol+64) + bias (optionally ReLU) -> A operand
template <bool RELU>
__device__ __forceinline__ void epilogue_to_a(const WG& c, uint32_t dcol, const float* __restrict__ bias_s) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        float v[16], bb[16];
        tmem_ld16_sync(c.tmem + dcol + q * 16, v);
        lds16(bias_s + q * 16, bb);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const float x = v[j] + bb[j];
            v[j] = RELU ? relu_nan(x) : x;
        }
        a_store16(c, q, v);
    }
}

// K < 64 first layer on CUDA cores: relu(bias + sum_k feat[k] * wt[k][:]) -> A operand.  wt_s: fp32 [K][64] in smem
template <int K>
__device__ __forceinline__ void first_layer_to_a(const WG& c, const float (&feat)[K], const float* __restrict__ wt_s,
                                                 const float* __restrict__ bias_s) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        float o[16];
        lds16(bias_s + q * 16, o);
#pragma unroll
        for (int k = 0; k < K; ++k) {
            float w[16];
            lds16(wt_s + k * P + q * 16, w);
#pragma unroll
            for (int j = 0; j < 16; ++j) o[j] = fmaf(feat[k], w[j], o[j]);
        }
#pragma unroll
        for (int j = 0; j < 16; ++j) o[j] = relu_nan(o[j]);
        a_store16(c, q, o);
    }
}

// (accumulator columns [dcol, dcol+64) + bias) * rowscale -> this thread's row of the mu tile image, staged in the
// warpgroup's landing buffer (free at this point: the tile's first GEMM has completed and the next tile's nb image has
// not been requested yet): fp16 hi / lo planes, K-major SWIZZLE_128B, scaled domain — conflict-free 16-byte stores.
// TO_A: the same values also become the next A operand (score head).  Returns true on NaN in a valid row.
template <bool TO_A>
__device__ __forceinline__ bool epilogue_to_mu(const WG& c, uint32_t dcol, const float* __restrict__ bias_s, float rowscale,
                                               bool valid, bool stage = true) {
    bool bad = false;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        float v[16], bb[16];
        tmem_ld16_sync(c.tmem + dcol + q * 16, v);
        lds16(bias_s + q * 16, bb);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            v[j] = (v[j] + bb[j]) * rowscale;
            bad |= (v[j] != v[j]);
        }
        uint32_t w[16];
#pragma unroll
        for (int i = 0; i < 8; ++i) split2(v[2 * i], v[2 * i + 1], w[i], w[8 + i]);
#pragma unroll
        for (int h = 0; h < 2 && stage; ++h) {
            const uint32_t off = swz((uint32_t)c.t, (uint32_t)(q * 2 + h));
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(c.land + off), "r"(w[4 * h]), "r"(w[4 * h + 1]),
                         "r"(w[4 * h + 2]), "r"(w[4 * h + 3]) : "memory");
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(c.land + APLANE + off), "r"(w[8 + 4 * h]),
                         "r"(w[8 + 4 * h + 1]), "r"(w[8 + 4 * h + 2]), "r"(w[8 + 4 * h + 3]) : "memory");
        }
        if (TO_A) tmem_st16(c.tmem + c.acol + 16 * q, w);
    }
    return bad && valid;
}
// the staged tile image -> global with one bulk store (the landing buffer is busy until bulk_wait_read)
__device__ __forceinline__ void commit_tile(const WG& c, void* dst_tile) {
    fence_proxy_async();                 // the staging stores are generic-proxy writes, the bulk store reads through the async proxy
    wg_barrier(c);
    if (c.t == 0) bulk_s2g(dst_tile, c.land, ABUF);
}
// request a tile's nb image into the landing buffer (one thread), after the previous tile's bulk store has read the buffer
__device__ __forceinline__ void request_nb(const WG& c, const void* src) {
    if (c.t == 0) {
        bulk_wait_read();
        mbar_expect_tx(c.mbar_tma, ABUF);
        bulk_g2s(c.land, src, ABUF, c.mbar_tma);
    }
}

// (accumulator columns [dcol, dcol+64) + bias) * rowscale -> relax' layout [tile][16][128][4] (scaled domain, coalesced)
__device__ __forceinline__ void epilogue_to_rlx(const WG& c, uint32_t dcol, const float* __restrict__ bias_s, float rowscale,
                                                float* __restrict__ dst_tile) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        float v[16], bb[16];
        tmem_ld16_sync(c.tmem + dcol + q * 16, v);
        lds16(bias_s + q * 16, bb);
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            const float4 o = make_float4((v[h * 4 + 0] + bb[h * 4 + 0]) * rowscale, (v[h * 4 + 1] + bb[h * 4 + 1]) * rowscale,
                                         (v[h * 4 + 2] + bb[h * 4 + 2]) * rowscale, (v[h * 4 + 3] + bb[h * 4 + 3]) * rowscale);
            *reinterpret_cast<float4*>(dst_tile + ((size_t)(q * 4 + h) * TILE + c.t) * 4) = o;
        }
    }
}

// ---- shared-memory layout -----------------------------------------------------------------------------
constexpr int NWG = 4;          // warpgroups (tiles in flight) per CTA: 4 x 128 tensor-memory columns
struct Tail {                   // small fp32 data after the weight planes and landing buffers
    float bias[6][P];           // pre-scaled by ASCALE
    float w_small[2][8 * P];    // first-layer weights (K <= 7), transposed [K][64], pre-scaled
    float vec[P];
    uint64_t mbar[1 + 2 * NWG];
    uint32_t tmem_slot;
    int32_t wcnt[NWG][4];       // ambiguous rows per warp of the warpgroup's current tile
};

struct CtaSetup {
    unsigned char* base;        // 1024-aligned dynamic shared memory
    uint32_t w;                 // shared address of the weight planes
    Tail* tail;
    uint32_t tmem_base;
};

__device__ __forceinline__ unsigned char* smem_dyn() {
    extern __shared__ unsigned char smem_raw_[];
    return smem_raw_;
}

// common prologue: carve shared memory, allocate TMEM, init mbarriers, TMA the weight planes in.
// LAND: the kernel has a 32 KB landing buffer per warpgroup after the weights.
template <bool LAND, int NW>
__device__ __forceinline__ CtaSetup cta_setup(unsigned char* smem_raw, uint32_t wbytes, const uint16_t* const (&wsrc)[NW],
                                              const uint32_t (&woff)[NW], const uint32_t (&wlen)[NW]) {
    CtaSetup s;
    s.base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);     // pointer arithmetic keeps the shared address space
    s.w = smem_u32(s.base);
    s.tail = reinterpret_cast<Tail*>(s.base + wbytes + (LAND ? NWG * ABUF : 0));
    if (threadIdx.x == 0) {
        for (int i = 0; i < 1 + 2 * NWG; ++i) mbar_init(smem_u32(&s.tail->mbar[i]), 1);
        fence_mbar_init();
    }
    __syncwarp();
    if (threadIdx.x < 32) tmem_alloc(smem_u32(&s.tail->tmem_slot), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    s.tmem_base = s.tail->tmem_slot;
    if (threadIdx.x == 0) {
        const uint32_t mb = smem_u32(&s.tail->mbar[0]);
        uint32_t total = 0;
        for (int i = 0; i < NW; ++i) total += wlen[i];
        mbar_expect_tx(mb, total);
        for (int i = 0; i < NW; ++i) bulk_g2s(s.w + woff[i], wsrc[i], wlen[i], mb);
    }
    return s;
}
__device__ __forceinline__ WG make_wg(const CtaSetup& s, uint32_t wbytes) {
    WG c;
    c.wg = uniform((int)(threadIdx.x >> 7));
    c.lead_warp = (uniform((int)(threadIdx.x >> 5)) & 3) == 0;
    c.t = threadIdx.x & 127;
    c.land = s.w + wbytes + (uint32_t)c.wg * ABUF;
    c.mbar_mma = smem_u32(&s.tail->mbar[1 + 2 * c.wg]);
    c.mbar_tma = smem_u32(&s.tail->mbar[2 + 2 * c.wg]);
    c.ph_mma = 0;
    c.ph_tma = 0;
    c.acol = ACOL;
    c.bar_threads = 128;
    c.tmem0 = ((uint32_t)uniform((int)s.tmem_base) & 0x0000FFFFu) + (uint32_t)c.wg * WG_COLS;
    c.tmem = s.tmem_base + ((uint32_t)((c.t >> 5) * 32) << 16) + (uint32_t)c.wg * WG_COLS;
    return c;
}
__device__ __forceinline__ void cta_teardown(const CtaSetup& s) {
    tc_fence_before();
    __syncthreads();
    if (threadIdx.x < 32) tmem_dealloc(s.tmem_base, 512);
}
__device__ __forceinline__ void copy_vec(float* dst, const float* __restrict__ src, int n, float scale = ASCALE) {
    for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i] * scale;     // biases live in the scaled domain
}

// ---- update: 3 GEMMs per tile (see the header) [+ score head] ---------------------------------------------
constexpr uint32_t UPD_W3 = 0, UPD_WC = 4 * WPLANE, UPD_W42 = 6 * WPLANE, UPD_FN = 8 * WPLANE, UPD_WBYTES = 10 * WPLANE;   // 80 KB

struct UpdArgs {
    GnnParams g;
    int backward;
    const float *lb, *ub;
    const uint16_t* nb_img;
    const float* rlx;
    const int32_t* amb_base;
    uint16_t* mu_out;
    float* scores;
    RowMap map;
    int64_t score_stride, score_off;
    int Bc;
    unsigned long long* nan_count;
    NanDoms nan_doms;
};

// NaN watch of a row of subdomain `dom` (of the wave): with option "rescore" the subdomain's first NaN puts it on the call's
// list of subdomains that are scored again in exact fp32.  Rows of a tile all belong to one subdomain.
__device__ __forceinline__ bool nan_watch(const NanDoms& nd, int dom, bool nan_row) {
    if (nan_row && nd.flag != nullptr && atomicExch(nd.flag + nd.dom0 + dom, 1) == 0) nd.list[atomicAdd(nd.count, 1)] = nd.dom0 + dom;
    return nan_row;
}

// One CTA's share of a node-update launch.  Work items are the propagation's: item = group of 4 subdomains x tile, taken
// rank, rank + nranks, ...; warpgroup w updates the tile of subdomain 4 * group + w.
__device__ __forceinline__ void update_body(const UpdArgs& a, unsigned char* smem_raw, int rank, int nranks, bool pdl = false) {
    const GnnParams& g = a.g;
    const int backward = a.backward;
    const float* __restrict__ lb = a.lb;
    const float* __restrict__ ub = a.ub;
    const uint16_t* __restrict__ nb_img = a.nb_img;
    const float* __restrict__ rlx = a.rlx;
    const int32_t* __restrict__ amb_base = a.amb_base;
    uint16_t* __restrict__ mu_out = a.mu_out;
    float* __restrict__ scores = a.scores;
    const RowMap map = a.map;
    const int64_t score_stride = a.score_stride, score_off = a.score_off;
    const int l3 = backward ? BC3 : FC3, l4b = backward ? BC4_1 : FC4_2, lc = backward ? T_BWD_C : T_FWD_C;
    const uint16_t* const wsrc[4] = {g.tc[l3], g.tcx_w[lc], g.tc[l4b], g.tc[FNODE]};
    const uint32_t woff[4] = {UPD_W3, UPD_WC, UPD_W42, UPD_FN};
    const uint32_t wlen[4] = {4 * WPLANE, 2 * WPLANE, 2 * WPLANE, 2 * WPLANE};
    CtaSetup s = cta_setup<true, 4>(smem_raw, UPD_WBYTES, wsrc, woff, wlen);
    Tail& tl = *s.tail;
    copy_vec(tl.bias[0], g.bias[l3], P); copy_vec(tl.bias[1], g.tcx_b[lc], P); copy_vec(tl.bias[2], g.bias[l4b], P);
    copy_vec(tl.bias[3], g.bias[FNODE], P); copy_vec(tl.vec, g.wt[FSCORE], P, 1.0f);
    const float bscore = g.bias[FSCORE][0];
    __syncthreads();
    mbar_wait(smem_u32(&tl.mbar[0]), 0);                      // weight planes have landed
    if (pdl) { pdl_trigger(); pdl_wait(); }                   // everything above read constant parameters only
    WG c = make_wg(s, UPD_WBYTES);
    const uint32_t W = s.w;
    const int tiles_per_dom = map.nslots / TILE;
    const int64_t nitems = (int64_t)tiles_per_dom * ((a.Bc + NWG - 1) / NWG);
    bool bad = false;
    GNNB_TR_DECL;
    // this row's bounds are fetched one item ahead (two dependent 4-byte gathers from HBM would otherwise stall the
    // warpgroup at the top of every tile)
    int64_t nrow_n = -1;
    float l_n = 0.f, u_n = 1.f;
    int slot0_n = 0;
    auto fetch_row = [&](int64_t it) {
        nrow_n = -1; l_n = 0.f; u_n = 1.f; slot0_n = 0;
        if (it >= nitems) return;
        const int d = (int)(it / tiles_per_dom) * NWG + c.wg;
        if (d >= a.Bc) return;
        const int64_t tl_ = (int64_t)d * tiles_per_dom + it % tiles_per_dom;
        nrow_n = natural_row(map, tl_ * TILE + c.t);           // index into the caller's [B, n] arrays, -1 = padding slot
        if (nrow_n >= 0) { l_n = ldg1_now(lb + nrow_n); u_n = ldg1_now(ub + nrow_n); }
        slot0_n = __ldg(amb_base + tl_);
    };
    fetch_row(rank);
    for (int64_t item = rank; item < nitems; item += nranks) {
        const int dom = (int)(item / tiles_per_dom) * NWG + c.wg;
        const int64_t nrow = nrow_n;
        const float l = l_n, u = u_n;
        const int slot0 = slot0_n;
        if (dom >= a.Bc) {
            fetch_row(item + nranks);
            continue;
        }
        const int64_t tile = (int64_t)dom * tiles_per_dom + item % tiles_per_dom;
        const int64_t row0 = tile * TILE, grow = row0 + c.t;
        request_nb(c, nb_img + (size_t)tile * (ABUF / 2));
        fetch_row(item + nranks);
        const Ratio q = compute_ratio(l, u);
        const float gate = (q.r0 != 0.0f) ? 1.0f : 0.0f;
        // slot of this row's relax' = first slot of the tile + number of ambiguous rows before it (amb_compact keeps row order)
        const bool amb = (q.amb != 0.0f) && nrow >= 0;
        const unsigned bal = __ballot_sync(0xffffffffu, amb);
        if ((c.t & 31) == 0) tl.wcnt[c.wg][c.t >> 5] = __popc(bal);
        GNNB_TR(0);
        // D[0:128) = nb [W3a; W3b]^T
        gemm_ss(c, W + UPD_W3, W + UPD_W3 + 2 * WPLANE, 128, 0);
        GNNB_TR(1);
        // towards L2 while this tile runs its chain: the next tile's nb image and this row's relax' pieces
        if (c.t == 0 && item + nranks < nitems) {
            const int64_t nitem = item + nranks;
            const int ndom = (int)(nitem / tiles_per_dom) * NWG + c.wg;
            if (ndom < a.Bc) prefetch_l2(nb_img + (size_t)((int64_t)ndom * tiles_per_dom + nitem % tiles_per_dom) * (ABUF / 2), ABUF);
        }
        int slot = slot0 + __popc(bal & ((1u << (c.t & 31)) - 1u));
#pragma unroll
        for (int w = 0; w < 3; ++w) slot += (w < (c.t >> 5)) ? tl.wcnt[c.wg][w] : 0;
        const float* rt = rlx + (size_t)(slot >> 7) * (TILE * P) + (size_t)(slot & (TILE - 1)) * 4;
        if (amb) {
#pragma unroll
            for (int i = 0; i < 16; ++i) asm volatile("prefetch.global.L2 [%0];" ::"l"(rt + (size_t)i * (TILE * 4)));
        }
        // h3 = relu(r0 * D[0:64) + r1 * D[64:128) + b3) -> A, in place over the consumed columns (graph_conv.py:169-170 / 331-336)
#pragma unroll
        for (int qd = 0; qd < 4; ++qd) {
            float a[16], b[16], bb[16];
            {
                uint32_t ra[16], rb[16];
                tmem_ld16(c.tmem + qd * 16, ra);
                tmem_ld16(c.tmem + 64 + qd * 16, rb);
                tmem_wait16(ra, a);
                tmem_wait16(rb, b);
            }
            lds16(tl.bias[0] + qd * 16, bb);
#pragma unroll
            for (int j = 0; j < 16; ++j) a[j] = relu_nan(fmaf(q.r0, a[j], fmaf(q.r1, b[j], bb[j])));
            a_store16(c, qd, a);
        }
        GNNB_TR(2);
        // D[64:128) = h3 Wc^T; meanwhile fetch this row's relax' (coalesced by layout, L2-resident by prefetch)
        gemm_ts_start(c, W + UPD_WC, W + UPD_WC + WPLANE, 64, DCOL);
        float4 rx[16];
        {
#pragma unroll
            for (int i = 0; i < 16; ++i) rx[i] = amb ? ldg4_now(rt + (size_t)i * (TILE * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        gemm_finish(c);
        GNNB_TR(3);
        // g = relu(D + relax' + bc) -> A
#pragma unroll
        for (int qd = 0; qd < 4; ++qd) {
            float v[16], bb[16];
            tmem_ld16_sync(c.tmem + DCOL + qd * 16, v);
            lds16(tl.bias[1] + qd * 16, bb);
#pragma unroll
            for (int h = 0; h < 4; ++h) {
                const float4 x = rx[qd * 4 + h];
                v[h * 4 + 0] = relu_nan(v[h * 4 + 0] + x.x + bb[h * 4 + 0]);
                v[h * 4 + 1] = relu_nan(v[h * 4 + 1] + x.y + bb[h * 4 + 1]);
                v[h * 4 + 2] = relu_nan(v[h * 4 + 2] + x.z + bb[h * 4 + 2]);
                v[h * 4 + 3] = relu_nan(v[h * 4 + 3] + x.w + bb[h * 4 + 3]);
            }
            a_store16(c, qd, v);
        }
        GNNB_TR(4);
        // D[64:128) = g W4_2^T;  mu = (D + b) * (r0 != 0) -> global
        gemm_ts(c, W + UPD_W42, W + UPD_W42 + WPLANE, 64, DCOL);
        GNNB_TR(5);
        if (scores == nullptr) {
            bad |= nan_watch(a.nan_doms, dom, epilogue_to_mu<false>(c, DCOL, tl.bias[2], gate, nrow >= 0));
            commit_tile(c, mu_out + (size_t)tile * (ABUF / 2));
        } else {      // score head on the new embeddings (graph_conv.py:448-449)
            bad |= nan_watch(a.nan_doms, dom, epilogue_to_mu<true>(c, DCOL, tl.bias[2], gate, nrow >= 0, mu_out != nullptr));
            // mu_out == null: nothing reads these embeddings (first hidden layer on the last backward sweep: its only
            // consumer would be the input-layer update, which is dead on the last round) — the scores are all that is kept
            if (mu_out != nullptr) commit_tile(c, mu_out + (size_t)tile * (ABUF / 2));
            gemm_ts(c, W + UPD_FN, W + UPD_FN + WPLANE, 64, DCOL);
            float sc = 0.f;
#pragma unroll
            for (int qd = 0; qd < 4; ++qd) {
                float v[16], bb[16], ww[16];
                tmem_ld16_sync(c.tmem + DCOL + qd * 16, v);
                lds16(tl.bias[3] + qd * 16, bb);
                lds16(tl.vec + qd * 16, ww);
#pragma unroll
                for (int j = 0; j < 16; ++j) sc = fmaf(relu_nan(v[j] + bb[j]), ww[j], sc);
            }
            if (nrow >= 0) scores[(nrow / map.n) * score_stride + score_off + (nrow % map.n)] = fmaf(sc, AINV, bscore);
        }
        GNNB_TR(6);
        GNNB_TR_NEXT();
    }
    GNNB_TR_PRINT("update[top gemm1 epi1 gemm2 epi2 gemm3 epi3]", 7);
    if (bad) atomicAdd(a.nan_count, 1ULL);
    if (c.t == 0) bulk_wait_all();       // the last tile's bulk store still reads this CTA's shared memory
    cta_teardown(s);
}

__global__ void __launch_bounds__(128 * NWG, 1) k_tc_update(UpdArgs a) {
    update_body(a, smem_dyn(), (int)blockIdx.x, (int)gridDim.x, true);
}

// ---- fused layer: propagation gather-GEMM -> tensor memory -> node-update chain ------------------------------------------
// One launch per (layer, sweep): the neighbour embeddings nb = A(mu) of a tile never leave the SM.  A persistent CTA (1 per
// SM, 24 warps) walks items = (tile of 128 nodes) x (pair of subdomains); the propagation of item i + 1 runs while the two
// chains of item i run (the propagation accumulator is double-buffered in tensor memory).  One ring of 6 - 8 stages, one K
// step (16 input nodes) each: [8 KB weight block | 8 KB gathered rows] = everything the step's three MMAs read.
//   warp 0      one bulk copy per K step: the step's weight block (plan.ks_w: 128 x 16 fp16 hi + lo, K-major without swizzle)
//   warps 2-7   gather: warp g owns the steps g, g + 6, ... and copies the step's 16 input-node rows of both subdomains with
//               16-byte cp.async from the mu images into the MN-major SWIZZLE_128B B operand (16 instructions per lane = 8 KB,
//               which is what one warp can keep in flight: scripts/micro/gather_bw2.cu)
//   warp 1      tcgen05.mma M = 128, N = 128 (2 subdomains x 64 channels), K = 16, three fp16 hi / lo passes, into accumulator
//               it & 1 (tensor-memory columns [128 (it & 1), +128)); tcgen05.commit frees the stage and publishes the accumulator
//   warps 8-23  four chain warpgroups: subdomain j of every item is walked by two of them, h = 0 / 1 owning channels [32 h, +32)
//               of every epilogue (thread = row of the tile = TMEM lane): tcgen05.ld of the accumulator columns -> fp16 hi / lo
//               split -> tcgen05.st back IN PLACE as the A operand of the chain (the same split the stand-alone propagation
//               kernel writes to its nb image); then the update chain of k_tc_update with every GEMM in the TS form (A from
//               tensor memory) and the chain's 128 accumulator columns at [256 + 128 j, +128).  The new embeddings are staged
//               per pair of warps (32 rows x 128 B of one plane = 4 KB, contiguous in the swizzled mu image) and leave with one
//               bulk store per plane.
// Registers: 768 threads x 80; with half a row's channels per thread the chain fits (no setmaxnreg needed).
// Tensor memory: 2 x 128 (propagation accumulators = the chains' A operands) + 2 x 128 (chain accumulators) = 512 columns.
// Shared memory: chain weights 64 KB (80 KB with the score head) + staging 64 KB (32 KB) + ring 96 KB (112 KB) — all of it.
// Accumulator b is free for item i + 2 when both chains of item i have completed their FIRST GEMM, the only one that reads its
// A columns (acc_empty[b], 2 arrivals): the later A operands live in columns [64, 128) of the chain's own window, which the
// first epilogue has just consumed.  The chains are software-pipelined by one stage (start_item below): a tile's accumulator
// wait, conversion and first GEMM issue run inside the last epilogue of the tile before it.
namespace fz {
constexpr int PD = 2;                               // subdomains per item = accumulator columns / 64
constexpr int CW = 2;                               // chain warpgroups = PD
constexpr int NS_MAX = 8;                           // ring stages (one K step each)
constexpr uint32_t W_KS = 8192;                     // weight block of one K step: [hi 128 x 16][lo 128 x 16] fp16, no swizzle
constexpr uint32_t B_ROWS = 16;                     // input nodes per stage = one K step
constexpr uint32_t B_DOM = B_ROWS * 128;            // 2 KB: one plane of one subdomain
constexpr uint32_t B_PLANE = PD * B_DOM;            // 4 KB
constexpr uint32_t B_STAGE = 2 * B_PLANE;           // 8 KB
constexpr uint32_t STAGE = W_KS + B_STAGE;          // 16 KB: everything the three MMAs of a K step read
constexpr uint32_t STG_PLANE = 32 * 128;            // 4 KB: a warp's 32 rows of one plane of a mu tile image
constexpr uint32_t STG_WARP = 2 * STG_PLANE;        // 8 KB: hi + lo
constexpr uint32_t STG_BYTES = CW * 4 * STG_WARP;   // 64 KB, only in launches that store embeddings
constexpr uint32_t INF_WN = 0, INF_WI = 2 * WPLANE, INF_B22 = 4 * WPLANE;      // chain weights of the input-layer variant
constexpr int THREADS = 768;                        // 8 producer warps + 4 chain warpgroups
constexpr int GATHER_WARP0 = 2, GATHER_WARPS = 6, CHAIN_WARP0 = 8;
constexpr uint32_t ACC_COL = 0, ACC_WIN = PD * 64, D_COL = 256, D_WIN = 128;

struct Tail {
    float bias[4][P];           // pre-scaled by ASCALE
    float vec[P];
    uint64_t wts, full[NS_MAX], empty[NS_MAX], acc_full[2], acc_empty[2], mma[CW];
    uint32_t tmem_slot;
    int32_t wcnt[2 * CW][4];
};
// staging: 0 = none (nothing stored), 1 = one plane per warp (score-head launches), 2 = both planes
constexpr size_t smem_for(uint32_t wbytes, int staging, int n_stages) {
    return 1024 + wbytes + (size_t)staging * (STG_BYTES / 2) + (size_t)n_stages * STAGE + sizeof(Tail);
}
constexpr size_t SMEM_MAX = 232448;                 // 227 KB: the per-block opt-in limit of sm_100
}  // namespace fz

struct FusedArgs {
    UpdArgs u;                  // u.nb_img is unused
    PropPlanDev plan;
    const uint16_t* mu_in;      // mu images of the layer the propagation reads
    uint16_t* nb_dbg;           // snapshots only: the nb tile images the two-launch path would have written, or null
    int n_stages;               // ring stages that fit beside the chain weights and the staging buffers (6 .. 8)
    int mma_group;              // K steps the propagation issues per pass of its loop (1 .. 4)
    int input_layer;            // 1: the chain is the input-layer update (graph_conv.py:360-385; u.lb / u.ub are the input bounds, no
                                // relaxation term, no gate), 0: a hidden layer's forward / backward update
};

// two 16-column tensor-memory loads in flight, then both -> fp32
__device__ __forceinline__ void tmem_ld32_sync(uint32_t taddr, float (&v0)[16], float (&v1)[16]) {
    uint32_t r0[16], r1[16];
    tmem_ld16(taddr, r0);
    tmem_ld16(taddr + 16, r1);
    tmem_wait16(r0, v0);
    tmem_wait16(r1, v1);
}

// 16 fp32 -> 8 hi + 8 lo packed fp16x2 words (element 2i at the lower half of word i)
__device__ __forceinline__ void split16(const float (&v)[16], uint32_t (&w)[16]) {
#pragma unroll
    for (int i = 0; i < 8; ++i) split2(v[2 * i], v[2 * i + 1], w[i], w[8 + i]);
}
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// (accumulator columns [dcol + 32 h, +32) + bias) * rowscale -> channels [32 h, 32 h + 32) of this thread's row of the mu tile
// image (fp16 hi / lo planes, K-major SWIZZLE_128B, scaled domain).  The two warps that hold the same 32 rows (one per column
// half) share an 8 KB staging buffer: a warp's 32 rows of one plane are 4 KB contiguous in the image, both planes are staged
// (conflict-free swizzled 16-byte stores) and leave with one bulk store per plane issued by the h = 0 warp — no warpgroup
// barrier, only the 64-thread barrier `pair_bar` of the two warps; the stores drain while the warps run their next tile (a
// synchronous store of any kind — 32-byte direct stores, coalesced 16-byte stores, a bulk store waited for — costs the chain
// 2 500 - 4 000 cycles per tile [measured, profiles/r02*_fused_phase_trace.log]).  TO_A (score-head launches, which need
// 16 KB more weights): the values also become the next A operand, and the buffer is 4 KB — the hi plane leaves first, the lo
// plane (kept in registers) follows once the first bulk store has read the buffer.  img: the tile image in global memory or
// null (nothing is stored).  Returns true on NaN in a valid row.  Both warps of the pair call it.
#ifdef GNNB_TRACE
__device__ long long g_e3_trace[4];          // e3 sub-phases of the tracing thread: wait for the previous stores, compute + stage, fence + issue
#define E3TR(i) do { if (blockIdx.x == 1 && threadIdx.x == fz::CHAIN_WARP0 * 32) { const long long n_ = clock64(); g_e3_trace[i] += n_ - e3t_; e3t_ = n_; } } while (0)
#else
#define E3TR(i) do {} while (0)
#endif
struct NoOp { __device__ __forceinline__ void operator()() const {} };
// `between` runs after the accumulator columns have been read and the values staged, before the stores are issued (!TO_A only):
// k_tc_fused starts its next tile there (the tile's first GEMM then runs under the fence, barrier and store issue below)
template <bool TO_A, class Between = NoOp>
__device__ __forceinline__ bool epilogue_to_mu_pair(const WG& c, int h, int pair_bar, uint32_t dcol, const float* __restrict__ bias_s,
                                                    float rowscale, bool valid, unsigned char* img, uint32_t stage, Between between = Between()) {
    bool bad = false;
#ifdef GNNB_TRACE
    long long e3t_ = clock64();
#endif
    const uint32_t rl = (uint32_t)c.t & 31u;                       // row within the warp's 32 rows = lane
    const bool issuer = h == 0 && rl == 0;
    unsigned char* dst = img + ((uint32_t)c.t >> 5) * fz::STG_PLANE;
    uint32_t lo[TO_A ? 16 : 1];
    if (img != nullptr) {
        if (issuer) bulk_wait_read();                               // the previous tile's bulk stores have read the buffer
        named_bar(pair_bar, 64);
    }
    E3TR(0);
    {
        float v0[16], v1[16];
        tmem_ld32_sync(c.tmem + dcol + h * 32, v0, v1);
        E3TR(1);
#pragma unroll
        for (int qq = 0; qq < 2; ++qq) {
            float (&v)[16] = qq ? v1 : v0;
            const int q = 2 * h + qq;
            float bb[16];
            lds16(bias_s + q * 16, bb);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                v[j] = (v[j] + bb[j]) * rowscale;
                bad |= (v[j] != v[j]);
            }
            uint32_t w[16];
            split16(v, w);
            if (img != nullptr) {
                const uint32_t o0 = stage + swz(rl, (uint32_t)(2 * q)), o1 = stage + swz(rl, (uint32_t)(2 * q + 1));
                sts128(o0, w[0], w[1], w[2], w[3]);
                sts128(o1, w[4], w[5], w[6], w[7]);
                if (!TO_A) {
                    sts128(o0 + fz::STG_PLANE, w[8], w[9], w[10], w[11]);
                    sts128(o1 + fz::STG_PLANE, w[12], w[13], w[14], w[15]);
                }
            }
            if (TO_A) {
#pragma unroll
                for (int i = 0; i < 8; ++i) lo[qq * 8 + i] = w[8 + i];
                tmem_st16(c.tmem + c.acol + 16 * q, w);
            }
        }
    }
    E3TR(2);
    if (!TO_A) between();
    if (img != nullptr) {
        fence_proxy_async();             // the staging stores are generic-proxy writes, the bulk stores read through the async proxy
        named_bar(pair_bar, 64);
        if (!TO_A) {
            if (issuer) {
                bulk_s2g_nocommit(dst, stage, fz::STG_PLANE);
                bulk_s2g_nocommit(dst + APLANE, stage + fz::STG_PLANE, fz::STG_PLANE);
                bulk_commit();
            }
        } else {
            if (issuer) { bulk_s2g(dst, stage, fz::STG_PLANE); bulk_wait_read(); }
            named_bar(pair_bar, 64);
#pragma unroll
            for (int qq = 0; qq < 2; ++qq) {
                const int q = 2 * h + qq;
                sts128(stage + swz(rl, (uint32_t)(2 * q)), lo[qq * 8], lo[qq * 8 + 1], lo[qq * 8 + 2], lo[qq * 8 + 3]);
                sts128(stage + swz(rl, (uint32_t)(2 * q + 1)), lo[qq * 8 + 4], lo[qq * 8 + 5], lo[qq * 8 + 6], lo[qq * 8 + 7]);
            }
            fence_proxy_async();
            named_bar(pair_bar, 64);
            if (issuer) bulk_s2g(dst + APLANE, stage, fz::STG_PLANE);
        }
    }
    E3TR(3);
    return bad && valid;
}

// The CTA's item sequence rank, rank + nranks, ... as (pair of subdomains, tile) with item = pair * ntiles + tile, advanced
// without divisions (a 64-bit division by a run-time value is ~100 instructions; the roles walk the sequence once per item).
struct ItemCursor {
    int pair, tile, dq, dr, ntiles, npairs;
    __device__ __forceinline__ ItemCursor(int rank, int nranks, int ntiles_, int npairs_)
        : pair(rank / ntiles_), tile(rank % ntiles_), dq(nranks / ntiles_), dr(nranks % ntiles_), ntiles(ntiles_), npairs(npairs_) {}
    __device__ __forceinline__ bool valid() const { return pair < npairs; }
    __device__ __forceinline__ void next() {
        tile += dr; pair += dq;
        if (tile >= ntiles) { tile -= ntiles; ++pair; }
    }
};

template <bool INPUT_LAYER>
__device__ __forceinline__ void fused_body(const FusedArgs& fa) {
    using namespace fz;
    const UpdArgs& a = fa.u;
    const GnnParams& g = a.g;
    const PropPlanDev& plan = fa.plan;
    const bool with_score = a.scores != nullptr;
    const uint32_t wbytes = with_score ? UPD_WBYTES : UPD_FN;          // the fnode planes are only needed by the score head
    const int NS = fa.n_stages;
    unsigned char* base = smem_dyn();
    base += (1024u - (smem_u32(base) & 1023u)) & 1023u;
    const uint32_t stg_warp = a.mu_out == nullptr ? 0u : (with_score ? STG_PLANE : STG_WARP), stg_bytes = CW * 4 * stg_warp;
    const uint32_t W = smem_u32(base), stg = W + wbytes, ring = stg + stg_bytes;
    fz::Tail* tl = reinterpret_cast<fz::Tail*>(base + wbytes + stg_bytes + (size_t)NS * STAGE);
    const int warp = uniform((int)(threadIdx.x >> 5)), lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        mbar_init(smem_u32(&tl->wts), 1);
        // a stage is full when its weight block has landed (1 arrival + its bytes) and the 32 lanes of the gather warp that owns
        // it have seen their copies land; it is empty again when the step's MMAs have completed (tcgen05.commit)
        for (int i = 0; i < NS; ++i) { mbar_init(smem_u32(&tl->full[i]), 1 + 32); mbar_init(smem_u32(&tl->empty[i]), 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(smem_u32(&tl->acc_full[i]), 1); mbar_init(smem_u32(&tl->acc_empty[i]), PD); }
        for (int i = 0; i < CW; ++i) mbar_init(smem_u32(&tl->mma[i]), 1);
        fence_mbar_init();
    }
    __syncwarp();
    if (warp == 0) tmem_alloc(smem_u32(&tl->tmem_slot), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tl->tmem_slot;
    const int l3 = a.backward ? BC3 : FC3, l4b = a.backward ? BC4_1 : FC4_2, lc = a.backward ? T_BWD_C : T_FWD_C;
    constexpr bool inp = INPUT_LAYER;
    if (threadIdx.x == 0) {
        const uint32_t mb = smem_u32(&tl->wts);
        if (!inp) {
            mbar_expect_tx(mb, wbytes);
            bulk_g2s(W + UPD_W3, g.tc[l3], 4 * WPLANE, mb);
            bulk_g2s(W + UPD_WC, g.tcx_w[lc], 2 * WPLANE, mb);
            bulk_g2s(W + UPD_W42, g.tc[l4b], 2 * WPLANE, mb);
            if (with_score) bulk_g2s(W + UPD_FN, g.tc[FNODE], 2 * WPLANE, mb);
        } else {      // mu0 = inp_b2_2(relu(Wi relu(inp_b([l0, u0])) + Wn nb + bi)),  Wi = W_b2[:, :64] W_b1,  Wn = W_b2[:, 64:]
            mbar_expect_tx(mb, 6 * WPLANE);
            bulk_g2s(W + INF_WN, g.tcx_w[T_INP_NB], 2 * WPLANE, mb);
            bulk_g2s(W + INF_WI, g.tcx_w[T_INP_C], 2 * WPLANE, mb);
            bulk_g2s(W + INF_B22, g.tc[INP_B2_2], 2 * WPLANE, mb);
        }
    }
    if (!inp) {
        copy_vec(tl->bias[0], g.bias[l3], P); copy_vec(tl->bias[1], g.tcx_b[lc], P); copy_vec(tl->bias[2], g.bias[l4b], P);
        copy_vec(tl->bias[3], g.bias[FNODE], P); copy_vec(tl->vec, g.wt[FSCORE], P, 1.0f);
    } else {
        copy_vec(tl->bias[0], g.tcx_b[T_INP_C], P); copy_vec(tl->bias[1], g.bias[INP_B2_2], P); copy_vec(tl->bias[2], g.bias[INP_B], P);
        copy_vec(tl->bias[3], g.wt[INP_B], 2 * P);          // [2][64] transposed first-layer weight: fills bias[3] and vec (adjacent)
    }
    __syncthreads();
    pdl_trigger(); pdl_wait();                    // everything above read constant parameters only

    const int ntiles = plan.ntiles, npairs = (a.Bc + PD - 1) / PD;       // item = pair * ntiles + tile
    const int rank = (int)blockIdx.x, nranks = (int)gridDim.x;

    if (warp == 0) {
        // ---- propagation weight blocks: 8 KB per K step into the W half of the step's ring stage ----
        if (lane == 0) {
            uint32_t slot = 0, ph = 0;
            for (ItemCursor cur(rank, nranks, ntiles, npairs); cur.valid(); cur.next()) {
                const int ks0 = plan.tile_ks0[cur.tile], ks1 = plan.tile_ks0[cur.tile + 1];
                for (int ks = ks0; ks < ks1; ++ks) {
                    mbar_wait(smem_u32(&tl->empty[slot]), ph ^ 1u);
                    const uint32_t full = smem_u32(&tl->full[slot]);
                    mbar_expect_tx(full, W_KS);
                    bulk_g2s(ring + slot * STAGE, plan.ks_w + (size_t)ks * (W_KS / 2), W_KS, full);
                    if (++slot == (uint32_t)NS) { slot = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ---- propagation MMAs: the whole warp walks the loop (uniform control and operands), one elected lane issues ----
        // D fp32, A fp16 K-major (no swizzle), B fp16 MN-major SWIZZLE_128B (bit 16), M = 128, N = 128
        const uint32_t idesc = (1u << 4) | (1u << 16) | ((uint32_t)(PD * 64 >> 3) << 17) | ((uint32_t)(TILE >> 4) << 24);
        uint32_t t = 0, it = 0, slot = 0, ph = 0;
        const int group = fa.mma_group;
        // operand descriptors of ring stage 0; stage s adds s * STAGE / 16 to the 14-bit address field (the whole ring lies below
        // 256 KB, so the field never carries): one add per descriptor and K step instead of rebuilding four descriptors
        const uint64_t d_a_hi = make_desc_nosw(ring, NB_PIECE, 128u), d_a_lo = make_desc_nosw(ring + W_KS / 2, NB_PIECE, 128u);
        const uint64_t d_b_hi = make_desc_mn(ring + W_KS, B_DOM), d_b_lo = make_desc_mn(ring + W_KS + B_PLANE, B_DOM);
        uint32_t lag_slot0 = 0, lag_slot1 = 0, lag_ph0 = 0, lag_ph1 = 0;       // last step of the group before the previous one / of the previous one
        bool have_lag = false, have_prev = false;
#ifdef GNNB_TRACE
        long long t_acc = 0, t_b = 0, t_lag = 0, t_all = clock64(), t0_;
#define FTR_BEGIN() t0_ = clock64()
#define FTR_END(x) x += clock64() - t0_
#else
#define FTR_BEGIN()
#define FTR_END(x)
#endif
        for (ItemCursor cur(rank, nranks, ntiles, npairs); cur.valid(); cur.next(), ++it) {
            const int ks0 = uniform(plan.tile_ks0[cur.tile]), ks1 = uniform(plan.tile_ks0[cur.tile + 1]);
            const uint32_t buf = it & 1u, bufph = (it >> 1) & 1u;
            FTR_BEGIN();
            mbar_wait(smem_u32(&tl->acc_empty[buf]), bufph ^ 1u);     // the chains of item it - 2 no longer read these A columns
            FTR_END(t_acc);
            tc_fence_after();
            const uint32_t d = (tmem_base & 0x0000FFFFu) + ACC_COL + buf * ACC_WIN;
            uint32_t accum = 0;
            // K steps are issued in groups of up to GROUP: one pass through the loop costs ~350 cycles of waits, fences and
            // descriptor arithmetic whatever it issues, a K step's three N = 128 MMAs 192 cycles of tensor time.  The tensor pipe
            // executes MMAs in issue order, so a group is only issued when the group before the previous one has completed: a
            // chain GEMM issued meanwhile waits for at most two groups.
            for (int ks = ks0; ks < ks1;) {
                const int n = ks1 - ks < group ? ks1 - ks : group;
                FTR_BEGIN();
                if (have_lag) mbar_wait(smem_u32(&tl->empty[lag_slot0]), lag_ph0);
                FTR_END(t_lag);
                lag_slot0 = lag_slot1; lag_ph0 = lag_ph1; have_lag = have_prev;
                for (int i = 0; i < n; ++i, ++t) {
                    FTR_BEGIN();
                    mbar_wait(smem_u32(&tl->full[slot]), ph);
                    FTR_END(t_b);
                    tc_fence_after();
                    const uint64_t soff = (uint64_t)(slot * (STAGE >> 4));
                    const uint64_t a_hi = d_a_hi + soff, a_lo = d_a_lo + soff, b_hi = d_b_hi + soff, b_lo = d_b_lo + soff;
                    if (elect_one()) {
                        umma(d, a_hi, b_hi, idesc, accum);               // Wh Mh
                        umma(d, a_lo, b_hi, idesc, 1u);                  // Wl Mh
                        umma(d, a_hi, b_lo, idesc, 1u);                  // Wh Ml
                        umma_commit(smem_u32(&tl->empty[slot]));
                    }
                    __syncwarp();
                    accum = 1u;
                    lag_slot1 = slot; lag_ph1 = ph;                      // the group's last step completes last
                    if (++slot == (uint32_t)NS) { slot = 0; ph ^= 1u; }
                }
                have_prev = true;
                ks += n;
            }
            if (elect_one()) umma_commit(smem_u32(&tl->acc_full[buf]));
            __syncwarp();
        }
#ifdef GNNB_TRACE
        if (rank == 1 && lane == 0) printf("TRACE fused-mma: items %u ksteps %u total %lld | wait acc_empty %lld, lag %lld, stage full %lld\n", it, t,
                                           clock64() - t_all, t_acc, t_lag, t_b);
#endif
    } else if (warp >= GATHER_WARP0 && warp < GATHER_WARP0 + GATHER_WARPS) {
        // ---- gather: warp gw owns the K steps t = gw, gw + 6, ... of the CTA's sequence and copies the step's 16 input-node rows
        //      of both subdomains (hi + lo plane: 8 KB, 16 x 16-byte cp.async per lane) from the mu images into the MN-major
        //      SWIZZLE_128B B half of the step's stage.  A warp keeps ~8 KB of cp.async misses in flight whatever it does
        //      (scripts/micro/gather_bw2.cu: 5 B / cycle / warp from DRAM with 2, 4 or 8 stages per warp, arrive- or
        //      commit-group-tracked; L2 prefetches share the budget; the rate scales with the number of warps), so the six warps
        //      work on six different stages: 48 KB in flight ----
        const int gw = warp - GATHER_WARP0;
        // A gather warp may run at most one revolution of the ring ahead of the others: it waits for "the previous use of my stage
        // has been consumed" by the PARITY of that use, and a warp that skipped a whole revolution would read the parity of the use
        // before as its own (measured the hard way: seven warps on a six-stage ring arrive twice on one `full` barrier and fault).
        // So never more owners than stages.
        const int GW = GATHER_WARPS < NS ? GATHER_WARPS : NS;
        const unsigned char* mu_bytes = reinterpret_cast<const unsigned char*>(fa.mu_in);
#ifdef GNNB_TRACE
        long long g_wait = 0, g_all = clock64();
#endif
        uint32_t slot = 0, ph = 0;
        int turn = 0;                                   // stage counter modulo the number of gather warps
        for (ItemCursor cur(rank, nranks, ntiles, npairs); cur.valid(); cur.next()) {
            const int ks0 = __ldg(plan.tile_ks0 + cur.tile), ks1 = __ldg(plan.tile_ks0 + cur.tile + 1);
            const int dm0 = cur.pair * PD;
            // per item: this lane's 16-byte column of the two subdomains' mu images, and what a copy from them reads (0 = zero fill:
            // the second subdomain of an odd batch).  Per row only its byte offset inside a subdomain's image is left to add: slot s
            // sits in tile s >> 7 (32 KB: hi plane, lo plane) at row s & 127 of 128 bytes
            const uint32_t jp = (uint32_t)(lane & 7);               // physical 16-byte chunk of the row in the mu image
            const unsigned char* base0 = mu_bytes + (int64_t)dm0 * (plan.nslots_in >> 7) * (int64_t)ABUF + jp * 16u;
            const uint32_t sz0 = dm0 < a.Bc ? 16u : 0u, sz1 = dm0 + 1 < a.Bc ? 16u : 0u;
            const unsigned char* base1 = sz1 ? base0 + (int64_t)(plan.nslots_in >> 7) * (int64_t)ABUF : base0;      // (a zero-fill copy still names an address)
            for (int ks = ks0; ks < ks1; ++ks) {
                const uint32_t slot_ = slot, ph_ = ph;
                const bool mine = turn == gw;
                if (++slot == (uint32_t)NS) { slot = 0; ph ^= 1u; }
                if (++turn == GW) turn = 0;
                if (!mine) continue;
                const int idx = __ldg(plan.ks_rows + (size_t)ks * 16 + (lane & 15));      // issued before the wait below
                const int off = idx < 0 ? -1 : (idx << 7) + ((idx >> 7) << 14);           // (s >> 7) * 32 KB + (s & 127) * 128
#ifdef GNNB_TRACE
                const long long g0_ = clock64();
#endif
                mbar_wait(smem_u32(&tl->empty[slot_]), ph_ ^ 1u);
#ifdef GNNB_TRACE
                g_wait += clock64() - g0_;
#endif
                const uint32_t dst0 = ring + slot_ * STAGE + W_KS;
#pragma unroll
                for (int q = 0; q < 4; ++q) {                            // 4 rows x 8 chunks per instruction, both subdomains, both planes
                    const int k = q * 4 + (lane >> 3);                   // row of the stage
                    const int o = __shfl_sync(0xffffffffu, off, k);
                    const bool ok = o >= 0;
                    const uint32_t oo = ok ? (uint32_t)o : 0u, r7 = (oo >> 7) & 7u;       // logical chunk = physical ^ (row & 7)
                    const uint32_t dst = dst0 + swz((uint32_t)k, jp ^ r7);
                    const uint32_t z0 = ok ? sz0 : 0u, z1 = ok ? sz1 : 0u;
                    cp_async16_sz(dst, base0 + oo, z0);
                    cp_async16_sz(dst + B_PLANE, base0 + oo + APLANE, z0);
                    cp_async16_sz(dst + B_DOM, base1 + oo, z1);
                    cp_async16_sz(dst + B_DOM + B_PLANE, base1 + oo + APLANE, z1);
                }
                cp_async_arrive(smem_u32(&tl->full[slot_]));
            }
        }
#ifdef GNNB_TRACE
        if (rank == 1 && gw == 0 && lane == 0) printf("TRACE fused-gather: total %lld, wait stage empty %lld\n", clock64() - g_all, g_wait);
#endif
    } else if (warp >= CHAIN_WARP0) {
        // ---- node-update chains: subdomain j of every item is walked by TWO warpgroups, h = 0 / 1 owning channels [32 h, +32)
        //      of every epilogue (thread = row of the tile = TMEM lane in both); the chain is a latency chain of three GEMMs and
        //      four epilogues, and halving each epilogue's per-thread work shortens it more than anything else did ----
        const float* __restrict__ lb = a.lb;
        const float* __restrict__ ub = a.ub;
        const float* __restrict__ rlx = a.rlx;
        const int32_t* __restrict__ amb_base = a.amb_base;
        float* __restrict__ scores = a.scores;
        const RowMap map = a.map;
        const float bscore = g.bias[FSCORE][0];
        const int cw = warp - CHAIN_WARP0;                        // 0 .. 15
        const int j = uniform(cw >> 3), h = uniform((cw >> 2) & 1);
        WG c;
        c.wg = j;                                                // named barrier 1 + j, 256 threads
        c.bar_threads = 256;
        c.lead_warp = (cw & 7) == 0;
        c.t = threadIdx.x & 127;
        c.land = 0;
        c.mbar_mma = smem_u32(&tl->mma[j]);
        c.mbar_tma = 0;
        c.ph_mma = 0;
        c.ph_tma = 0;
        c.acol = ACC_COL;
        c.tmem0 = (uint32_t)uniform((int)tmem_base) & 0x0000FFFFu;
        c.tmem = tmem_base + ((uint32_t)((c.t >> 5) * 32) << 16);
        const uint32_t D = D_COL + D_WIN * (uint32_t)j;          // this chain's accumulator window [D, D + 128)
        const int pw = j * 4 + (cw & 3);                          // the pair of warps (one per half) that holds rows 32 (cw & 3) .. + 31
        const uint32_t stage = stg + (uint32_t)pw * stg_warp;     // the pair's 8 KB (4 KB with the score head) staging buffer
        const int pair_bar = 3 + pw;                              // named barriers 3 .. 10, 64 threads
        const int Q0 = 2 * h;                                     // this half's K steps / 16-channel groups: Q0, Q0 + 1
        mbar_wait(smem_u32(&tl->wts), 0);                        // chain weights have landed
        bool bad = false;
        // the node of a slot does not depend on the subdomain: node_of_slot[tile * 128 + t]; index into the caller's [B, n] arrays =
        // dom * n + node.  Two dependent 4-byte gathers (slot -> node, node -> bounds): the node is fetched two items ahead and
        // the bounds one item ahead, so neither latency is on the chain's path
        int node_n = -1, node_nn = -1;
        float l_n = 0.f, u_n = 1.f;
        int slot0_n = 0;
        auto fetch_node = [&](const ItemCursor& cu) -> int {     // -1 = padding slot / no item / no such subdomain
            if (!cu.valid() || cu.pair * PD + j >= a.Bc) return -1;
            return ldgi_now(map.node_of_slot + cu.tile * TILE + c.t);      // issued here, not sunk to its first use an item later
        };
        auto fetch_bounds = [&](const ItemCursor& cu, int node_) {
            node_n = node_; l_n = 0.f; u_n = 1.f; slot0_n = 0;
            if (!cu.valid()) return;
            const int d_ = cu.pair * PD + j;
            if (d_ >= a.Bc) return;
            if (node_ >= 0) { l_n = ldg1_now(lb + (int64_t)d_ * map.n + node_); u_n = ldg1_now(ub + (int64_t)d_ * map.n + node_); }
            if (amb_base != nullptr) slot0_n = ldgi_now(amb_base + (int64_t)d_ * ntiles + cu.tile);
        };
        ItemCursor cur(rank, nranks, ntiles, npairs), cur1 = cur, cur2 = cur;
        cur1.next();
        cur2.next(); cur2.next();
        fetch_bounds(cur, fetch_node(cur));
        node_nn = fetch_node(cur1);
        uint32_t it = 0;
#ifdef GNNB_TRACE
        long long c_wait = 0, c_ph[8] = {0, 0, 0, 0, 0, 0, 0, 0}, c_all = clock64(), c0_;
        int c_tiles = 0;
#define CTR(i) do { const long long n_ = clock64(); c_ph[i] += n_ - c0_; c0_ = n_; } while (0)
#else
#define CTR(i) do {} while (0)
#endif
        // The chain of a tile is software-pipelined by one stage: its first section — wait for the item's accumulator, nb -> A operand
        // in place, first GEMM issued — runs inside the LAST epilogue of the tile before it, right after that epilogue has read its
        // accumulator columns, so the GEMM executes under the store of the previous tile and the bookkeeping between two tiles
        // (~1 500 cycles of a ~10 800-cycle chain otherwise spent with nothing of this pair in the tensor pipe).
        // start_item: item `it_` at cursor `cu`, row inputs node_ / l_ / u_ (input-layer variant only).  Returns false when this
        // pair has no subdomain in the item (odd batch).
        auto start_item = [&](const ItemCursor& cu, uint32_t it_, int node_, float l_, float u_) -> bool {
            const uint32_t buf = it_ & 1u, bufph = (it_ >> 1) & 1u;
            const int dom_ = cu.pair * PD + j;
#ifdef GNNB_TRACE
            const long long w0_ = clock64();
#endif
            mbar_wait(smem_u32(&tl->acc_full[buf]), bufph);       // the item's nb = A(mu) is complete in tensor memory
#ifdef GNNB_TRACE
            c_wait += clock64() - w0_;
#endif
            tc_fence_after();
            if (dom_ >= a.Bc) {                                   // odd batch: the last pair has one subdomain
                if (h == 0 && c.t == 0) mbar_arrive(smem_u32(&tl->acc_empty[buf]));
                return false;
            }
            const int64_t tile = (int64_t)dom_ * ntiles + cu.tile;
            c.acol = ACC_COL + buf * ACC_WIN + 64u * (uint32_t)j;
            // nb: accumulator columns -> fp16 hi / lo A operand, in place (K step qd = channels [16 qd, 16 qd + 16))
            {
                unsigned char* dbg = fa.nb_dbg ? reinterpret_cast<unsigned char*>(fa.nb_dbg) + tile * (int64_t)ABUF + (uint32_t)c.t * 16u : nullptr;
                float v0[16], v1[16];
                tmem_ld32_sync(c.tmem + c.acol + h * 32, v0, v1);
#pragma unroll
                for (int qq = 0; qq < 2; ++qq) {
                    const int qd = Q0 + qq;
                    uint32_t w[16];
                    split16(qq ? v1 : v0, w);
                    tmem_st16(c.tmem + c.acol + 16 * qd, w);
                    if (dbg != nullptr) {      // piece-major nb image of the two-launch path (snapshots)
#pragma unroll
                        for (int hh = 0; hh < 2; ++hh) {
                            const uint32_t off = (uint32_t)(qd * 2 + hh) * NB_PIECE;
                            *reinterpret_cast<uint4*>(dbg + off) = make_uint4(w[4 * hh], w[4 * hh + 1], w[4 * hh + 2], w[4 * hh + 3]);
                            *reinterpret_cast<uint4*>(dbg + APLANE + off) = make_uint4(w[8 + 4 * hh], w[8 + 4 * hh + 1], w[8 + 4 * hh + 2], w[8 + 4 * hh + 3]);
                        }
                    }
                }
            }
            if (inp) {
                // ---- input-layer update (graph_conv.py:380-385): a second A operand relu(inp_b([l0, u0])) of this half's 32 channels
                //      (K < 64 first layer on CUDA cores) goes to D[64:128); D[0:64) = nb Wn^T + that Wi^T, one commit ----
                {
                    const float* w0 = &tl->bias[3][0];
#pragma unroll
                    for (int qq = 0; qq < 2; ++qq) {
                        const int qd = Q0 + qq;
                        float o[16], wl[16], wu[16];
                        lds16(tl->bias[2] + qd * 16, o);
                        lds16(w0 + qd * 16, wl);
                        lds16(w0 + P + qd * 16, wu);
#pragma unroll
                        for (int i = 0; i < 16; ++i) o[i] = relu_nan(fmaf(node_ >= 0 ? l_ : 0.f, wl[i], fmaf(node_ >= 0 ? u_ : 0.f, wu[i], o[i])));
                        uint32_t w[16];
                        split16(o, w);
                        tmem_st16(c.tmem + D + 64 + 16 * qd, w);
                    }
                }
                gemm_sync(c);
                if (c.lead_warp) {
                    tc_fence_after();
                    if (elect_one()) {
                        WG c2 = c;
                        c2.acol = D + 64;
                        issue_ts(c, W + INF_WN, W + INF_WN + WPLANE, 64, D, false);
                        issue_ts(c2, W + INF_WI, W + INF_WI + WPLANE, 64, D, true);
                        umma_commit(c.mbar_mma);
                    }
                    __syncwarp();
                }
            } else {
                gemm_ts_start(c, W + UPD_W3, W + UPD_W3 + 2 * WPLANE, 128, D);      // D[0:128) = nb [W3a; W3b]^T
            }
            return true;
        };
        bool have = cur.valid() ? start_item(cur, 0, node_n, l_n, u_n) : false;
        for (; cur.valid(); cur.next(), cur1.next(), cur2.next(), ++it) {
            const uint32_t buf = it & 1u;
            const uint32_t acc_empty = smem_u32(&tl->acc_empty[buf]);
            const int dom = cur.pair * PD + j;
            const int node = node_n;
            const float l = l_n, u = u_n;
            const int slot0 = slot0_n;
            fetch_bounds(cur1, node_nn);               // from here on node_n / l_n / u_n / slot0_n belong to item it + 1
            node_nn = fetch_node(cur2);
            // the next tile's first section, run from inside this tile's last epilogue (or directly, when this pair has no tile here)
            auto advance = [&]() { have = cur1.valid() ? start_item(cur1, it + 1, node_n, l_n, u_n) : false; };
            if (!have) {
                advance();
                continue;
            }
            const int64_t tile = (int64_t)dom * ntiles + cur.tile;
#ifdef GNNB_TRACE
            c0_ = clock64(); ++c_tiles;
#endif
            const Ratio q = compute_ratio(l, u);
            const float gate = (q.r0 != 0.0f) ? 1.0f : 0.0f;
            const bool amb = (q.amb != 0.0f) && node >= 0;
            const unsigned bal = __ballot_sync(0xffffffffu, amb);
            if ((c.t & 31) == 0) tl->wcnt[j * 2 + h][c.t >> 5] = __popc(bal);
            unsigned char* img = a.mu_out ? reinterpret_cast<unsigned char*>(a.mu_out) + tile * (int64_t)ABUF : nullptr;
            if (inp) {
                gemm_finish(c);
                if (h == 0 && c.t == 0) mbar_arrive(acc_empty);    // nb has been read: the propagation may refill this accumulator
                c.acol = D + 64;                                  // the remaining A operands live in the consumed half of the window
                CTR(1);
                {
                    float v0[16], v1[16];
                    tmem_ld32_sync(c.tmem + D + h * 32, v0, v1);
#pragma unroll
                    for (int qq = 0; qq < 2; ++qq) {
                        float (&v)[16] = qq ? v1 : v0;
                        const int qd = Q0 + qq;
                        float bb[16];
                        lds16(tl->bias[0] + qd * 16, bb);
#pragma unroll
                        for (int i = 0; i < 16; ++i) v[i] = relu_nan(v[i] + bb[i]);
                        a_store16(c, qd, v);
                    }
                }
                CTR(2);
                gemm_ts_start(c, W + INF_B22, W + INF_B22 + WPLANE, 64, D);
                gemm_finish(c);
                CTR(3);
                bad |= nan_watch(a.nan_doms, dom, epilogue_to_mu_pair<false>(c, h, pair_bar, D, tl->bias[1], 1.0f, node >= 0, img, stage, advance));
                CTR(6);
                continue;
            }
            gemm_finish(c);                                       // D[0:128) = nb [W3a; W3b]^T (issued by start_item)
            // nb has been read: the propagation may refill this accumulator while the chain goes on.  The remaining A operands
            // (h3, g, and the embeddings of the score head) live in D[64:128), each 16-column piece written by the thread that has
            // just consumed it in the first epilogue
            if (h == 0 && c.t == 0) mbar_arrive(acc_empty);
            c.acol = D + 64;
            CTR(1);
            // h3 = relu(r0 * D[0:64) + r1 * D[64:128) + b3) -> A (graph_conv.py:169-170 / 331-336)
#pragma unroll
            for (int qq = 0; qq < 2; ++qq) {
                const int qd = Q0 + qq;
                float x[16], y[16], bb[16];
                {
                    uint32_t ra[16], rb[16];
                    tmem_ld16(c.tmem + D + qd * 16, ra);
                    tmem_ld16(c.tmem + D + 64 + qd * 16, rb);
                    tmem_wait16(ra, x);
                    tmem_wait16(rb, y);
                }
                lds16(tl->bias[0] + qd * 16, bb);
#pragma unroll
                for (int i = 0; i < 16; ++i) x[i] = relu_nan(fmaf(q.r0, x[i], fmaf(q.r1, y[i], bb[i])));
                a_store16(c, qd, x);
            }
            CTR(2);
            // D[0:64) = h3 Wc^T; meanwhile fetch this row's relax'
            gemm_ts_start(c, W + UPD_WC, W + UPD_WC + WPLANE, 64, D);
            // slot of this row's relax' = first slot of the tile + number of ambiguous rows before it (the warps' counts were written
            // at the top of the iteration; the barrier of the GEMM above orders them)
            int slot = slot0 + __popc(bal & ((1u << (c.t & 31)) - 1u));
#pragma unroll
            for (int w = 0; w < 3; ++w) slot += (w < (c.t >> 5)) ? tl->wcnt[j * 2 + h][w] : 0;
            const float* rt = rlx + (size_t)(slot >> 7) * (TILE * P) + (size_t)(slot & (TILE - 1)) * 4 + (size_t)(8 * h) * (TILE * 4);
            float4 rx[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) rx[i] = amb ? ldg4_now(rt + (size_t)i * (TILE * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
            gemm_finish(c);
            CTR(3);
            // g = relu(D + relax' + bc) -> A
            {
                float v0[16], v1[16];
                tmem_ld32_sync(c.tmem + D + h * 32, v0, v1);
#pragma unroll
                for (int qq = 0; qq < 2; ++qq) {
                    float (&v)[16] = qq ? v1 : v0;
                    const int qd = Q0 + qq;
                    float bb[16];
                    lds16(tl->bias[1] + qd * 16, bb);
#pragma unroll
                    for (int hh = 0; hh < 4; ++hh) {
                        const float4 x = rx[qq * 4 + hh];
                        v[hh * 4 + 0] = relu_nan(v[hh * 4 + 0] + x.x + bb[hh * 4 + 0]);
                        v[hh * 4 + 1] = relu_nan(v[hh * 4 + 1] + x.y + bb[hh * 4 + 1]);
                        v[hh * 4 + 2] = relu_nan(v[hh * 4 + 2] + x.z + bb[hh * 4 + 2]);
                        v[hh * 4 + 3] = relu_nan(v[hh * 4 + 3] + x.w + bb[hh * 4 + 3]);
                    }
                    a_store16(c, qd, v);
                }
            }
            CTR(4);
            // D[0:64) = g W4_2^T;  mu = (D + b) * (r0 != 0) -> global
            gemm_ts_start(c, W + UPD_W42, W + UPD_W42 + WPLANE, 64, D);
            gemm_finish(c);
            CTR(5);
            if (!with_score) {
                bad |= nan_watch(a.nan_doms, dom, epilogue_to_mu_pair<false>(c, h, pair_bar, D, tl->bias[2], gate, node >= 0, img, stage, advance));
            } else {      // score head on the new embeddings (graph_conv.py:448-449)
                bad |= nan_watch(a.nan_doms, dom, epilogue_to_mu_pair<true>(c, h, pair_bar, D, tl->bias[2], gate, node >= 0, img, stage));
                gemm_ts_start(c, W + UPD_FN, W + UPD_FN + WPLANE, 64, D);
                gemm_finish(c);
                float sc = 0.f;
                {
                    float v0[16], v1[16];
                    tmem_ld32_sync(c.tmem + D + h * 32, v0, v1);
#pragma unroll
                    for (int qq = 0; qq < 2; ++qq) {
                        const int qd = Q0 + qq;
                        float bb[16], ww[16];
                        lds16(tl->bias[3] + qd * 16, bb);
                        lds16(tl->vec + qd * 16, ww);
#pragma unroll
                        for (int i = 0; i < 16; ++i) sc = fmaf(relu_nan((qq ? v1 : v0)[i] + bb[i]), ww[i], sc);
                    }
                }
                // the two halves of the dot product meet in a free tensor-memory column of the row's lane (D[64:128) is unused here)
                if (h == 1) {
                    tmem_st1(c.tmem + D + 64, __float_as_uint(sc));
                    tmem_st_wait();
                }
                tc_fence_before();
                wg_barrier(c);
                tc_fence_after();
                if (h == 0) {
                    sc += __uint_as_float(tmem_ld1_sync(c.tmem + D + 64));
                    if (node >= 0) scores[(int64_t)dom * a.score_stride + a.score_off + node] = fmaf(sc, AINV, bscore);
                }
                advance();                                        // (its GEMM is issued behind a barrier of the pair: both halves have read D)
            }
            CTR(6);
        }
#ifdef GNNB_TRACE
        if (rank == 1 && threadIdx.x == CHAIN_WARP0 * 32)
            printf("TRACE fused-chain wg0: tiles %d total %lld | wait acc_full %lld | per tile: convert %lld gemm1 %lld epi1 %lld gemm2 %lld epi2 %lld gemm3 %lld epi3 %lld\n",
                   c_tiles, clock64() - c_all, c_wait, c_ph[0] / max(c_tiles, 1), c_ph[1] / max(c_tiles, 1), c_ph[2] / max(c_tiles, 1), c_ph[3] / max(c_tiles, 1),
                   c_ph[4] / max(c_tiles, 1), c_ph[5] / max(c_tiles, 1), c_ph[6] / max(c_tiles, 1));
        if (rank == 1 && threadIdx.x == CHAIN_WARP0 * 32) {
            printf("TRACE fused-e3 (cumulative over launches): wait prev store %lld, tmem load %lld, compute + stage %lld, fence + issue %lld\n",
                   g_e3_trace[0], g_e3_trace[1], g_e3_trace[2], g_e3_trace[3]);
        }
#endif
        if (bad) atomicAdd(a.nan_count, 1ULL);
        if (h == 0 && (c.t & 31) == 0) bulk_wait_all();        // this pair's last bulk stores still read its staging buffer
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
}

// hidden layers (forward / backward sweep, + score head) and the input-layer update: the same body under two kernel names, so that
// profiles tell them apart
__global__ void __launch_bounds__(fz::THREADS, 1) k_tc_fused(FusedArgs fa) { fused_body<false>(fa); }
__global__ void __launch_bounds__(fz::THREADS, 1) k_tc_fused_input(FusedArgs fa) { fused_body<true>(fa); }

// ---- relax: round-independent part of the fc4 / bc4 pre-activation of a hidden layer --------------------------
constexpr uint32_t RLX_FR = 0, RLX_BC11 = 2 * WPLANE, RLX_BC12 = 4 * WPLANE, RLX_BC2 = 6 * WPLANE, RLX_BR = 12 * WPLANE;
constexpr uint32_t RLX_WBYTES = 14 * WPLANE;

// every hidden layer of a wave in one launch: the warpgroups walk the concatenation of the layers' compacted ambiguous tiles
struct RelaxLayers {
    NodeInputs in[AMB_MAX_LAYERS];
    float* rlx_f[AMB_MAX_LAYERS];
    float* rlx_b[AMB_MAX_LAYERS];
    int n;
};

__global__ void __launch_bounds__(128 * NWG, 1) k_tc_relax(GnnParams g, const __grid_constant__ RelaxLayers rl) {
    const uint16_t* const wsrc[5] = {g.tcx_w[T_FWD_R], g.tc[BC1_1], g.tc[BC1_2], g.tc[BC2], g.tcx_w[T_BWD_R]};
    const uint32_t woff[5] = {RLX_FR, RLX_BC11, RLX_BC12, RLX_BC2, RLX_BR};
    const uint32_t wlen[5] = {2 * WPLANE, 2 * WPLANE, 2 * WPLANE, 6 * WPLANE, 2 * WPLANE};
    CtaSetup s = cta_setup<false, 5>(smem_dyn(), RLX_WBYTES, wsrc, woff, wlen);
    Tail& tl = *s.tail;
    copy_vec(tl.bias[0], g.tcx_b[T_FWD_R], P); copy_vec(tl.bias[1], g.bias[BC1_1], P); copy_vec(tl.bias[2], g.bias[BC1_2], P);
    copy_vec(tl.bias[3], g.bias[BC2], P); copy_vec(tl.bias[4], g.tcx_b[T_BWD_R], P);
    copy_vec(tl.w_small[0], g.wt[FC1], 7 * P); copy_vec(tl.w_small[1], g.wt[BC1], 7 * P);
    copy_vec(tl.bias[5], g.bias[FC1], P); copy_vec(tl.vec, g.bias[BC1], P);
    __syncthreads();
    mbar_wait(smem_u32(&tl.mbar[0]), 0);
    pdl_trigger(); pdl_wait();
    WG c = make_wg(s, RLX_WBYTES);
    const uint32_t W = s.w;
    // only the ambiguous rows have non-zero relaxation features: walk them in compacted order (slot = tile * 128 + t), layer
    // after layer (tile0[k] = first global tile of layer k)
    int tile0[AMB_MAX_LAYERS + 1];
    tile0[0] = 0;
#pragma unroll 1
    for (int k = 0; k < rl.n; ++k) {
        const int namb_k = __ldg(rl.in[k].amb_base + (rl.in[k].rows + TILE - 1) / TILE);
        tile0[k + 1] = tile0[k] + (namb_k + TILE - 1) / TILE;
    }
    const int total_tiles = tile0[rl.n];
    int k = 0;
    for (int gt = (int)blockIdx.x * NWG + c.wg; gt < total_tiles; gt += (int)gridDim.x * NWG) {
        while (gt >= tile0[k + 1]) ++k;
        const NodeInputs& in = rl.in[k];
        float* __restrict__ rlx_f = rl.rlx_f[k];
        float* __restrict__ rlx_b = rl.rlx_b[k];
        const int64_t tile = gt - tile0[k];
        const int64_t namb = __ldg(in.amb_base + (in.rows + TILE - 1) / TILE);
        const int64_t slot = tile * TILE + c.t;
        float l = 0.f, u = 1.f, d1 = 0.f, d2 = 0.f, pp = 0.f, po = 0.f, bs = 0.f;
        if (slot < namb) {
            const int64_t grow = natural_row(in.map, __ldg(in.amb_rows + slot));      // ambiguous rows are never padding
            l = in.lb[grow]; u = in.ub[grow];
            d1 = in.dual[grow * 3 + 1]; d2 = in.dual[grow * 3 + 2];
            pp = in.prim_pre[grow]; po = in.prim_post[grow];
            bs = in.bias_node[grow % in.map.n];
        }
        const Ratio q = compute_ratio(l, u);
        // forward: relax' = amb * (Wr relu(fc1([beta, l, u, d1-d2, x_pre, x_post, bias])) + br)   (graph_conv.py:153-161, :176)
        {
            const float feat[7] = {q.beta, l, u, d1 - d2, pp, po, bs};
            first_layer_to_a<7>(c, feat, tl.w_small[0], tl.bias[5]);
        }
        gemm_ts(c, W + RLX_FR, W + RLX_FR + WPLANE, 64, DCOL);
        epilogue_to_rlx(c, DCOL, tl.bias[0], q.amb, rlx_f + (size_t)tile * (TILE * P));
        // backward (graph_conv.py:273-293, :344)
        {
            const float feat[7] = {l, u, q.beta, -d2 + d1, po, pp, bs};
            first_layer_to_a<7>(c, feat, tl.w_small[1], tl.vec);
        }
        gemm_ts(c, W + RLX_BC11, W + RLX_BC11 + WPLANE, 64, DCOL);
        epilogue_to_a<true>(c, DCOL, tl.bias[1]);
        gemm_ts(c, W + RLX_BC12, W + RLX_BC12 + WPLANE, 64, DCOL);
        epilogue_to_a<false>(c, DCOL, tl.bias[2]);                                  // s1
        // relu(s1 W2a^T - d2 s1 W2b^T + d1 s1 W2c^T + b2): the three 64-wide products share the A operand and the one
        // accumulator, so they run one after the other with the running sum in registers
        float acc[64];
        gemm_ts(c, W + RLX_BC2, W + RLX_BC2 + 3 * WPLANE, 64, DCOL);
#pragma unroll
        for (int qd = 0; qd < 4; ++qd) {
            float v[16], bb[16];
            tmem_ld16_sync(c.tmem + DCOL + qd * 16, v);
            lds16(tl.bias[3] + qd * 16, bb);
#pragma unroll
            for (int j = 0; j < 16; ++j) acc[qd * 16 + j] = v[j] + bb[j];
        }
        gemm_ts(c, W + RLX_BC2 + WPLANE, W + RLX_BC2 + 4 * WPLANE, 64, DCOL);
        {
            const float nd2 = -d2;
#pragma unroll
            for (int qd = 0; qd < 4; ++qd) {
                float v[16];
                tmem_ld16_sync(c.tmem + DCOL + qd * 16, v);
#pragma unroll
                for (int j = 0; j < 16; ++j) acc[qd * 16 + j] = fmaf(nd2, v[j], acc[qd * 16 + j]);
            }
        }
        gemm_ts(c, W + RLX_BC2 + 2 * WPLANE, W + RLX_BC2 + 5 * WPLANE, 64, DCOL);
#pragma unroll
        for (int qd = 0; qd < 4; ++qd) {
            float v[16];
            tmem_ld16_sync(c.tmem + DCOL + qd * 16, v);
#pragma unroll
            for (int j = 0; j < 16; ++j) v[j] = relu_nan(fmaf(d1, v[j], acc[qd * 16 + j]));
            a_store16(c, qd, v);
        }
        gemm_ts(c, W + RLX_BR, W + RLX_BR + WPLANE, 64, DCOL);
        epilogue_to_rlx(c, DCOL, tl.bias[4], q.amb, rlx_b + (size_t)tile * (TILE * P));
    }
    cta_teardown(s);
}

// ---- input embedding: mu0 = inp_f_1(relu(inp_f([l0, x, u0])))   (graph_conv.py:90-95) ---------------------------
constexpr uint32_t EMB_WBYTES = 2 * WPLANE;

__global__ void __launch_bounds__(128 * NWG, 1) k_tc_input_embed(GnnParams g, const float* __restrict__ lb0,
                                                                 const float* __restrict__ x, const float* __restrict__ ub0,
                                                                 uint16_t* __restrict__ mu0, RowMap map, int64_t rows) {
    const uint16_t* const wsrc[1] = {g.tc[INP_F_1]};
    const uint32_t woff[1] = {0};
    const uint32_t wlen[1] = {2 * WPLANE};
    CtaSetup s = cta_setup<true, 1>(smem_dyn(), EMB_WBYTES, wsrc, woff, wlen);
    Tail& tl = *s.tail;
    copy_vec(tl.bias[0], g.bias[INP_F_1], P); copy_vec(tl.bias[5], g.bias[INP_F], P); copy_vec(tl.w_small[0], g.wt[INP_F], 3 * P);
    __syncthreads();
    mbar_wait(smem_u32(&tl.mbar[0]), 0);
    pdl_trigger(); pdl_wait();
    WG c = make_wg(s, EMB_WBYTES);
    const int64_t ntiles = (rows + TILE - 1) / TILE;
    for (int64_t tile = (int64_t)blockIdx.x * NWG + c.wg; tile < ntiles; tile += (int64_t)gridDim.x * NWG) {
        const int64_t row0 = tile * TILE, grow = row0 + c.t;
        float feat[3] = {0.f, 0.f, 0.f};
        const int64_t nrow = grow < rows ? natural_row(map, grow) : -1;
        if (nrow >= 0) { feat[0] = lb0[nrow]; feat[1] = x[nrow]; feat[2] = ub0[nrow]; }
        first_layer_to_a<3>(c, feat, tl.w_small[0], tl.bias[5]);
        if (c.t == 0) bulk_wait_read();          // the previous tile's bulk store has read the staging buffer
        gemm_ts(c, s.w, s.w + WPLANE, 64, DCOL);
        epilogue_to_mu<false>(c, DCOL, tl.bias[0], 1.0f, nrow >= 0);
        commit_tile(c, mu0 + (size_t)tile * (ABUF / 2));
    }
    if (c.t == 0) bulk_wait_all();
    cta_teardown(s);
}

// ---- input update: mu0 = inp_b2_2(relu(inp_b2([inp_b_1(relu(inp_b([l0,u0]))), nb])))   (graph_conv.py:380-385) ----
//      = inp_b2_2(relu(Wi relu(inp_b([l0,u0])) + Wn nb + bi)),  Wi = W_b2[:, :64] W_b1,  Wn = W_b2[:, 64:]
constexpr uint32_t INU_WI = 0, INU_WN = 2 * WPLANE, INU_B22 = 4 * WPLANE, INU_WBYTES = 6 * WPLANE;

__global__ void __launch_bounds__(128 * NWG, 1) k_tc_input_update(GnnParams g, const float* __restrict__ lb0,
                                                                  const float* __restrict__ ub0, const uint16_t* __restrict__ nb_img,
                                                                  uint16_t* __restrict__ mu0, RowMap map, int64_t rows) {
    const uint16_t* const wsrc[3] = {g.tcx_w[T_INP_C], g.tcx_w[T_INP_NB], g.tc[INP_B2_2]};
    const uint32_t woff[3] = {INU_WI, INU_WN, INU_B22};
    const uint32_t wlen[3] = {2 * WPLANE, 2 * WPLANE, 2 * WPLANE};
    CtaSetup s = cta_setup<true, 3>(smem_dyn(), INU_WBYTES, wsrc, woff, wlen);
    Tail& tl = *s.tail;
    copy_vec(tl.bias[0], g.tcx_b[T_INP_C], P); copy_vec(tl.bias[1], g.bias[INP_B2_2], P);
    copy_vec(tl.bias[5], g.bias[INP_B], P); copy_vec(tl.w_small[0], g.wt[INP_B], 2 * P);
    __syncthreads();
    mbar_wait(smem_u32(&tl.mbar[0]), 0);
    pdl_trigger(); pdl_wait();
    WG c = make_wg(s, INU_WBYTES);
    const uint32_t W = s.w;
    const int64_t ntiles = (rows + TILE - 1) / TILE;
    const int64_t tile_step = (int64_t)gridDim.x * NWG;
    for (int64_t tile = (int64_t)blockIdx.x * NWG + c.wg; tile < ntiles; tile += tile_step) {
        const int64_t row0 = tile * TILE, grow = row0 + c.t;
        request_nb(c, nb_img + (size_t)tile * (ABUF / 2));
        float feat[2] = {0.f, 0.f};
        const int64_t nrow = grow < rows ? natural_row(map, grow) : -1;
        if (nrow >= 0) { feat[0] = lb0[nrow]; feat[1] = ub0[nrow]; }
        first_layer_to_a<2>(c, feat, tl.w_small[0], tl.bias[5]);
        // D = Wi relu(inp_b(.)) + Wn nb: both products into the one accumulator, one commit
        gemm_sync(c);
        if (c.lead_warp) {
            tc_fence_after();
            if (elect_one()) issue_ts(c, W + INU_WI, W + INU_WI + WPLANE, 64, DCOL, false);
            __syncwarp();
            mbar_wait(c.mbar_tma, c.ph_tma);
            if (elect_one()) {
                issue_ss(c, W + INU_WN, W + INU_WN + WPLANE, 64, DCOL, true);
                umma_commit(c.mbar_mma);
            }
            __syncwarp();
        }
        c.ph_tma ^= 1u;
        gemm_finish(c);
        epilogue_to_a<true>(c, DCOL, tl.bias[0]);
        gemm_ts(c, W + INU_B22, W + INU_B22 + WPLANE, 64, DCOL);
        epilogue_to_mu<false>(c, DCOL, tl.bias[1], 1.0f, nrow >= 0);
        commit_tile(c, mu0 + (size_t)tile * (ABUF / 2));
    }
    if (c.t == 0) bulk_wait_all();
    cta_teardown(s);
}

constexpr size_t smem_bytes(uint32_t wbytes, bool land) { return 1024 + wbytes + (land ? NWG * ABUF : 0) + sizeof(Tail); }

int grid_for(int64_t rows) {
    const int64_t tiles = (rows + TILE - 1) / TILE, ctas = (tiles + NWG - 1) / NWG;
    return (int)(ctas < 1 ? 1 : (ctas < 148 ? ctas : 148));
}

// tile images (hi + lo planes, scaled domain) -> fp32 [rows][64]; debugging snapshots and the output-node kernel's view
__global__ void k_unpack_tile_image(const uint16_t* __restrict__ img, float* __restrict__ out, RowMap map, int64_t rows,
                                    int piece_major) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;      // one thread per (slot row, 8-channel chunk)
    if (i >= rows * 8) return;
    const int64_t row = i >> 3;
    const int64_t nrow = natural_row(map, row);
    if (nrow < 0) return;
    const int chunk = (int)(i & 7);
    const int64_t tile = row / TILE;
    const uint32_t r = (uint32_t)(row % TILE);
    const uint32_t off = piece_major ? (uint32_t)chunk * NB_PIECE + r * 16u : swz(r, (uint32_t)chunk);
    const __half* hi = reinterpret_cast<const __half*>(img) + tile * (ABUF / 2) + off / 2;
    const __half* lo = hi + APLANE / 2;
    for (int j = 0; j < 8; ++j) out[nrow * P + chunk * 8 + j] = (__half2float(hi[j]) + __half2float(lo[j])) * AINV;
}

// ---- compaction of the ambiguous rows (three small launches per layer and chunk) ---------------------------------
__device__ __forceinline__ bool row_is_ambiguous(const float* __restrict__ lb, const float* __restrict__ ub, const RowMap& map,
                                                 int64_t row, int64_t rows) {
    const int64_t nrow = row < rows ? natural_row(map, row) : -1;
    return nrow >= 0 && compute_ratio(lb[nrow], ub[nrow]).amb != 0.0f;
}
__global__ void __launch_bounds__(TILE) k_amb_count(const float* __restrict__ lb, const float* __restrict__ ub, RowMap map,
                                                    int64_t rows, int32_t* __restrict__ cnt) {
    const int64_t row = (int64_t)blockIdx.x * TILE + threadIdx.x;
    const bool amb = row_is_ambiguous(lb, ub, map, row, rows);
    const int total = __syncthreads_count(amb);
    if (threadIdx.x == 0) cnt[blockIdx.x] = total;
}
// exclusive scan of cnt[0 .. n) into base[0 .. n], base[n] = total; one block
__global__ void __launch_bounds__(1024) k_amb_scan(const int32_t* __restrict__ cnt, int32_t* __restrict__ base, int n) {
    __shared__ int32_t part[1024];
    const int per = (n + 1023) / 1024, lo = threadIdx.x * per, hi = min(n, lo + per);
    int32_t sum = 0;
    for (int i = lo; i < hi; ++i) sum += cnt[i];
    part[threadIdx.x] = sum;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {
        const int32_t v = threadIdx.x >= off ? part[threadIdx.x - off] : 0;
        __syncthreads();
        part[threadIdx.x] += v;
        __syncthreads();
    }
    int32_t run = part[threadIdx.x] - sum;
    for (int i = lo; i < hi; ++i) { base[i] = run; run += cnt[i]; }
    if (threadIdx.x == 1023) base[n] = part[1023];
}
__global__ void __launch_bounds__(TILE) k_amb_fill(const float* __restrict__ lb, const float* __restrict__ ub, RowMap map,
                                                   int64_t rows, const int32_t* __restrict__ base, int32_t* __restrict__ amb_rows) {
    __shared__ int32_t wc[4];
    const int64_t row = (int64_t)blockIdx.x * TILE + threadIdx.x;
    const bool amb = row_is_ambiguous(lb, ub, map, row, rows);
    const unsigned bal = __ballot_sync(0xffffffffu, amb);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) wc[warp] = __popc(bal);
    __syncthreads();
    int slot = base[blockIdx.x] + __popc(bal & ((1u << lane) - 1u));
    for (int w = 0; w < warp; ++w) slot += wc[w];
    if (amb) amb_rows[slot] = (int32_t)row;
}

// the same three steps for every hidden layer of a wave in three launches (a block finds its layer from the tile offsets)
__device__ __forceinline__ int amb_layer_of(const AmbLayers& a, int tile) {
    int k = 0;
    while (k + 1 < a.n && tile >= a.tile0[k + 1]) ++k;
    return k;
}
__global__ void __launch_bounds__(TILE) k_amb_count_all(AmbLayers a) {
    const int k = amb_layer_of(a, (int)blockIdx.x), tile = (int)blockIdx.x - a.tile0[k];
    const int64_t row = (int64_t)tile * TILE + threadIdx.x;
    const bool amb = row_is_ambiguous(a.lb[k], a.ub[k], a.map[k], row, a.rows[k]);
    const int total = __syncthreads_count(amb);
    if (threadIdx.x == 0) a.cnt[k][tile] = total;
}
__global__ void __launch_bounds__(1024) k_amb_scan_all(AmbLayers a) {
    __shared__ int32_t part[1024];
    const int k = blockIdx.x, n = a.tile0[k + 1] - a.tile0[k];
    const int32_t* __restrict__ cnt = a.cnt[k];
    int32_t* __restrict__ base = a.base[k];
    const int per = (n + 1023) / 1024, lo = threadIdx.x * per, hi = min(n, lo + per);
    int32_t sum = 0;
    for (int i = lo; i < hi; ++i) sum += cnt[i];
    part[threadIdx.x] = sum;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {
        const int32_t v = threadIdx.x >= off ? part[threadIdx.x - off] : 0;
        __syncthreads();
        part[threadIdx.x] += v;
        __syncthreads();
    }
    int32_t run = part[threadIdx.x] - sum;
    for (int i = lo; i < hi; ++i) { base[i] = run; run += cnt[i]; }
    if (threadIdx.x == 1023) base[n] = part[1023];
}
__global__ void __launch_bounds__(TILE) k_amb_fill_all(AmbLayers a) {
    __shared__ int32_t wc[4];
    const int k = amb_layer_of(a, (int)blockIdx.x), tile = (int)blockIdx.x - a.tile0[k];
    const int64_t row = (int64_t)tile * TILE + threadIdx.x;
    const bool amb = row_is_ambiguous(a.lb[k], a.ub[k], a.map[k], row, a.rows[k]);
    const unsigned bal = __ballot_sync(0xffffffffu, amb);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) wc[warp] = __popc(bal);
    __syncthreads();
    int slot = a.base[k][tile] + __popc(bal & ((1u << lane) - 1u));
    for (int w = 0; w < warp; ++w) slot += wc[w];
    if (amb) a.out_rows[k][slot] = (int32_t)row;
}

}  // namespace

void amb_compact_all(AmbLayers a, cudaStream_t st, int64_t* launches) {
    a.tile0[0] = 0;
    for (int k = 0; k < a.n; ++k) a.tile0[k + 1] = a.tile0[k] + (int)((a.rows[k] + TILE - 1) / TILE);
    k_amb_count_all<<<a.tile0[a.n], TILE, 0, st>>>(a);
    k_amb_scan_all<<<a.n, 1024, 0, st>>>(a);
    k_amb_fill_all<<<a.tile0[a.n], TILE, 0, st>>>(a);
    *launches += 3;
}

void amb_compact(const float* lb, const float* ub, RowMap map, int64_t rows, int32_t* cnt, int32_t* amb_base, int32_t* amb_rows,
                 cudaStream_t st, int64_t* launches) {
    const int ntiles = (int)((rows + TILE - 1) / TILE);
    k_amb_count<<<ntiles, TILE, 0, st>>>(lb, ub, map, rows, cnt);
    k_amb_scan<<<1, 1024, 0, st>>>(cnt, amb_base, ntiles);
    k_amb_fill<<<ntiles, TILE, 0, st>>>(lb, ub, map, rows, amb_base, amb_rows);
    *launches += 3;
}

bool tc_available() { return true; }

int tc_init() {
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(k_tc_update, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes(UPD_WBYTES, true))) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_tc_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fz::SMEM_MAX)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_tc_fused_input, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fz::SMEM_MAX)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_tc_relax, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes(RLX_WBYTES, false))) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_tc_input_embed, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes(EMB_WBYTES, true))) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_tc_input_update, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes(INU_WBYTES, true))) != cudaSuccess) return e;
    return 0;
}

// packed layout of one linear weight W[64][K], K = 64 * nblk:  [hi plane of K-block 0 .. nblk-1][lo plane 0 .. nblk-1],
// each plane 64 (n) x 64 (k) fp16 in the K-major SWIZZLE_128B shared-memory image (8 KB), so that the planes of
// consecutive K-blocks also read as one (64 * nblk)-row B tile
int64_t tc_packed_elems(int K) { return (int64_t)2 * (K / 64) * 64 * 64; }

int64_t tc_pack_weight(const float* w, int K, uint16_t* dst) {
    const int nblk = K / 64;
    for (int n = 0; n < 64; ++n)
        for (int k = 0; k < K; ++k) {
            uint16_t hi, lo;
            split_host(w[(size_t)n * K + k], hi, lo);
            const int kb = k / 64, kk = k % 64;
            const size_t e = (size_t)(swz((uint32_t)n, (uint32_t)(kk / 8)) + (kk % 8) * 2) / 2;
            dst[(size_t)kb * 4096 + e] = hi;
            dst[(size_t)(nblk + kb) * 4096 + e] = lo;
        }
    return tc_packed_elems(K);
}

void tc_relax(const GnnParams& g, const NodeInputs* in, float* const* relax_f, float* const* relax_b, int n_layers, cudaStream_t st,
              int64_t* launches) {
    RelaxLayers rl;
    rl.n = n_layers;
    int64_t rows = 0;
    for (int k = 0; k < n_layers; ++k) { rl.in[k] = in[k]; rl.rlx_f[k] = relax_f[k]; rl.rlx_b[k] = relax_b[k]; rows += in[k].rows; }
    launch_pdl(k_tc_relax, grid_for(rows), 128 * NWG, smem_bytes(RLX_WBYTES, false), st, g, rl);
    ++*launches;
}

namespace {
UpdArgs make_upd_args(const GnnParams& g, bool backward, const float* lb, const float* ub, const float* nb, const float* relax,
                      const int32_t* amb_base, float* mu_out, float* scores, RowMap map, int64_t score_stride, int64_t score_off,
                      int64_t rows, unsigned long long* nan_count, const NanDoms& nan_doms) {
    UpdArgs a;
    a.g = g; a.backward = backward ? 1 : 0; a.lb = lb; a.ub = ub; a.nb_img = reinterpret_cast<const uint16_t*>(nb); a.rlx = relax;
    a.amb_base = amb_base; a.mu_out = reinterpret_cast<uint16_t*>(mu_out); a.scores = scores; a.map = map;
    a.score_stride = score_stride; a.score_off = score_off; a.Bc = (int)(rows / map.nslots); a.nan_count = nan_count;
    a.nan_doms = nan_doms;
    return a;
}
}  // namespace

void tc_update(const GnnParams& g, bool backward, const float* lb, const float* ub, const float* nb, const float* relax,
               const int32_t* amb_base, float* mu_out, float* scores, RowMap map, int64_t score_stride, int64_t score_off, int64_t rows,
               unsigned long long* nan_count, const NanDoms& nan_doms, cudaStream_t st, int64_t* launches) {
    const UpdArgs a = make_upd_args(g, backward, lb, ub, nb, relax, amb_base, mu_out, scores, map, score_stride, score_off, rows, nan_count,
                                    nan_doms);
    const int64_t nitems = (int64_t)(map.nslots / TILE) * ((a.Bc + NWG - 1) / NWG);
    launch_pdl(k_tc_update, (int)(nitems < 1 ? 1 : (nitems < 148 ? nitems : 148)), 128 * NWG, smem_bytes(UPD_WBYTES, true), st, a);
    ++*launches;
}

void tc_fused(const GnnParams& g, const PropPlan* plan, const float* mu_in, bool backward, const float* lb, const float* ub,
              const float* relax, const int32_t* amb_base, float* mu_out, float* scores, RowMap map, int64_t score_stride, int64_t score_off,
              int64_t rows, unsigned long long* nan_count, const NanDoms& nan_doms, float* nb_dbg, bool input_layer, cudaStream_t st,
              int64_t* launches) {
    FusedArgs fa;
    fa.input_layer = input_layer ? 1 : 0;
    fa.u = make_upd_args(g, backward, lb, ub, nullptr, relax, amb_base, mu_out, scores, map, score_stride, score_off, rows, nan_count,
                         nan_doms);
    fa.plan = prop_plan_dev(plan);
    fa.mu_in = reinterpret_cast<const uint16_t*>(mu_in);
    fa.nb_dbg = reinterpret_cast<uint16_t*>(nb_dbg);
    const uint32_t wbytes = scores ? UPD_WBYTES : UPD_FN;
    const int staging = mu_out == nullptr ? 0 : (scores ? 1 : 2);
    const int ns = (int)((fz::SMEM_MAX - fz::smem_for(wbytes, staging, 0)) / fz::STAGE);
    fa.n_stages = ns > fz::NS_MAX ? fz::NS_MAX : ns;
    // layers with long K loops are bound by the propagation's issue loop, layers with short ones by the chains, whose GEMMs queue
    // behind whatever the propagation has issued: groups of 4 K steps for the former, pairs of steps for the latter
    // (a chain takes ~11 000 cycles per item, a K step 192 cycles of tensor time: only K loops of 48+ steps outlast the chains)
    fa.mma_group = prop_plan_ksteps_per_tile(plan) >= 48.0 ? 4 : 2;      // (2 instead of 1 for the short loops: +1 % on the base step)
    if (fa.mma_group > fa.n_stages / 2) fa.mma_group = fa.n_stages / 2;
    const int64_t nitems = (int64_t)fa.plan.ntiles * ((fa.u.Bc + fz::PD - 1) / fz::PD);
    launch_pdl(input_layer ? k_tc_fused_input : k_tc_fused, (int)(nitems < 1 ? 1 : (nitems < 148 ? nitems : 148)), fz::THREADS,
               fz::smem_for(wbytes, staging, fa.n_stages), st, fa);
    ++*launches;
}

void tc_input_embed(const GnnParams& g, const float* lb0, const float* x, const float* ub0, float* mu0, RowMap map, int64_t rows,
                    cudaStream_t st, int64_t* launches) {
    launch_pdl(k_tc_input_embed, grid_for(rows), 128 * NWG, smem_bytes(EMB_WBYTES, true), st, g, lb0, x, ub0, reinterpret_cast<uint16_t*>(mu0), map, rows);
    ++*launches;
}

void tc_input_update(const GnnParams& g, const float* lb0, const float* ub0, const float* nb, float* mu0, RowMap map, int64_t rows,
                     cudaStream_t st, int64_t* launches) {
    launch_pdl(k_tc_input_update, grid_for(rows), 128 * NWG, smem_bytes(INU_WBYTES, true), st,
               g, lb0, ub0, reinterpret_cast<const uint16_t*>(nb), reinterpret_cast<uint16_t*>(mu0), map, (int64_t)rows);
    ++*launches;
}

void tc_unpack_tile_image(const float* img, float* out, RowMap map, int64_t rows, bool piece_major, cudaStream_t st) {
    const int64_t n = rows * 8;
    k_unpack_tile_image<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(reinterpret_cast<const uint16_t*>(img), out, map, rows, piece_major ? 1 : 0);
}

}  // namespace gnnb
