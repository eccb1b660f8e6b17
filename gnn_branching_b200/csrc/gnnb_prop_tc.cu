// Propagation of the node embeddings through the verified network's edge sets on the tensor cores.
//
// Every edge set (conv2d, conv_transpose2d / freq, W @ mu, W^T @ mu; graph_conv.py:110-132, 299-322, 361-376) is a
// sparse matrix product  nb[b] = Wmat * mu[b]  with Wmat [n_out x n_in] built from the verified network's own
// weights.  At gnnb_set_network the matrix is cut into dense blocks ("plan", gnnb_prop_body.cuh): a tile is 128 output nodes
// chosen so that they share inputs (all channels of a small spatial patch), its K dimension is the sorted list of input nodes
// any of them touches, padded to K steps of 16, and its values are stored per K step as fp16 hi/lo planes in the UMMA K-major
// image without swizzle.  conv_transpose's 1/freq tap-count normalisation is folded into the rows.
//
// The kernel (k_tc_prop below) is a warp-specialised gather-GEMM over (tile, 4 subdomains) items; its input is the mu
// tile image of the producing layer and its output the piece-major nb tile image the node-update kernels TMA in
// (formats: gnnb_umma.cuh).  The fused kernel k_tc_fused (gnnb_tc.cu) reads the same plans.
#include <algorithm>
#include <functional>
#include <map>
#include <vector>

#include "gnnb_prop_body.cuh"
#include "gnnb_umma.cuh"

namespace gnnb {

using namespace tcx;

struct PropPlan {
    PropPlanDev dev{};
    void* blob = nullptr;
    int nksteps = 0;
    double density = 0.0;         // useful MACs / issued MACs
};

namespace prop {

// ---- the gather-GEMM kernel ---------------------------------------------------------------------------------
// A persistent CTA (1 per SM) walks items = (tile of 128 output nodes, group of PD = 4 subdomains); per chunk of up to 4 K steps
//   D[128 nodes x (4 subdomains x 64 channels)] += Wblock[128 x 64] * Mu[64 input nodes x (4 x 64)]
// as tcgen05.mma M = 128, N = 256, K = 16, three passes for the fp16 hi/lo split (Wh Mh + Wl Mh + Wh Ml).
// Warp roles (14 warps), decoupled by mbarrier rings:
//   warp 0      TMA: the chunk's weight blocks (plan.ks_w, 8 KB per K step, K-major without swizzle; one bulk copy of the
//               chunk's steps, which are contiguous)                                               -> W ring, 3 stages of 32 KB
//   warp 1      MMA issue + tcgen05.commit (frees ring stages, publishes accumulators): all 32 lanes walk the loop with
//               uniform operands, one elected lane issues (6 back-to-back UTCHMMA per half chunk)
//   warps 2-5   gather, one subdomain each: the half chunk's input-node rows (plan.ks_rows) are copied with 16-byte cp.async
//               straight from the mu tile images (already fp16 hi/lo, scaled) into the MN-major SWIZZLE_128B B operand — no
//               registers, no conversion; half a chunk (32 rows x 4 subdomains x 2 planes = 32 KB) per stage, 4 stages
//   warps 6-13  two epilogue warpgroups, alternating items on a double-buffered accumulator (2 x 256 TMEM columns):
//               tcgen05.ld -> fp16 hi/lo split -> piece-major nb tile image (consecutive rows = consecutive 16 bytes)
constexpr int PD = 4;
constexpr int W_STAGES = 3, B_STAGES = 4;
constexpr int CHUNK_KS = 4;                               // K steps per chunk = per W stage
constexpr uint32_t W_KS = 8192;                           // weight block of one K step: [hi 128 x 16][lo 128 x 16] fp16
constexpr uint32_t W_STAGE_BYTES = CHUNK_KS * W_KS;       // 32 KB
constexpr uint32_t B_ROWS = 32;                           // input nodes per B stage (half a chunk = 2 K steps)
constexpr uint32_t B_DOM_BYTES = B_ROWS * 128;            // 4 KB: one plane of one subdomain
constexpr uint32_t B_PLANE_BYTES = PD * B_DOM_BYTES;      // 16 KB
constexpr uint32_t B_STAGE_BYTES = 2 * B_PLANE_BYTES;     // 32 KB
constexpr int PROP_WARPS = 14, PROP_THREADS = PROP_WARPS * 32;
constexpr int GATHER_WARP0 = 2, EPI_WARP0 = 6;

struct PropTail {
    uint64_t w_full[W_STAGES], w_empty[W_STAGES], b_full[B_STAGES], b_empty[B_STAGES], acc_full[2], acc_empty[2];
    uint32_t tmem_slot;
};
constexpr size_t PROP_SMEM = 1024 + W_STAGES * W_STAGE_BYTES + B_STAGES * B_STAGE_BYTES + sizeof(PropTail);

}  // namespace prop

namespace {

__global__ void __launch_bounds__(prop::PROP_THREADS, 1) k_tc_prop(PropPlanDev plan, const uint16_t* __restrict__ mu_img,
                                                                   uint16_t* __restrict__ nb_img, int Bc) {
    using namespace prop;
    extern __shared__ unsigned char smem_raw[];
    unsigned char* base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);   // keeps the shared address space
    const uint32_t w_ring = smem_u32(base), b_ring = w_ring + W_STAGES * W_STAGE_BYTES;
    PropTail* tail = reinterpret_cast<PropTail*>(base + W_STAGES * W_STAGE_BYTES + B_STAGES * B_STAGE_BYTES);
    const int warp = uniform((int)(threadIdx.x >> 5)), lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int i = 0; i < W_STAGES; ++i) { mbar_init(smem_u32(&tail->w_full[i]), 1); mbar_init(smem_u32(&tail->w_empty[i]), 1); }
        for (int i = 0; i < B_STAGES; ++i) { mbar_init(smem_u32(&tail->b_full[i]), PD * 32); mbar_init(smem_u32(&tail->b_empty[i]), 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(smem_u32(&tail->acc_full[i]), 1); mbar_init(smem_u32(&tail->acc_empty[i]), 128); }
        fence_mbar_init();
    }
    __syncwarp();
    if (warp == 0) tmem_alloc(smem_u32(&tail->tmem_slot), 512);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tail->tmem_slot;
    pdl_trigger(); pdl_wait();          // prologue done; the mu images are the predecessor's output

    const int rank = (int)blockIdx.x, nranks = (int)gridDim.x;
    const int ngroups = (Bc + PD - 1) / PD;
    const int64_t nitems = (int64_t)plan.ntiles * ngroups;       // item = group * ntiles + tile

    if (warp == 0) {
        // ---- weight blocks: a chunk's K steps are contiguous in plan.ks_w ----
        if (lane == 0) {
            uint32_t ws = 0, wph = 0;
            for (int64_t item = rank; item < nitems; item += nranks) {
                const int tile = (int)(item % plan.ntiles);
                const int ks0 = plan.tile_ks0[tile], ks1 = plan.tile_ks0[tile + 1];
                for (int ks = ks0; ks < ks1; ks += CHUNK_KS) {
                    const uint32_t bytes = (uint32_t)min(CHUNK_KS, ks1 - ks) * W_KS;
                    mbar_wait(smem_u32(&tail->w_empty[ws]), wph ^ 1u);
                    const uint32_t full = smem_u32(&tail->w_full[ws]);
                    mbar_expect_tx(full, bytes);
                    bulk_g2s(w_ring + ws * W_STAGE_BYTES, plan.ks_w + (size_t)ks * (W_KS / 2), bytes, full);
                    if (++ws == W_STAGES) { ws = 0; wph ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ---- MMA issue: the whole warp walks the loop (uniform control and operands), one elected lane issues ----
        // D fp32, A fp16 K-major, B fp16 MN-major (bit 16), M = 128, N = 256
        const uint32_t idesc = (1u << 4) | (1u << 16) | ((uint32_t)(PD * 64 >> 3) << 17) | ((uint32_t)(TILE >> 4) << 24);
        constexpr uint64_t KS_DESC = W_KS >> 4;                    // one K step further in the W stage (descriptor address units)
        uint32_t ws = 0, wph = 0, bs = 0, bph = 0, it = 0;
#ifdef GNNB_TRACE
        long long t_acc = 0, t_w = 0, t_b = 0, t_all = clock64(), t0_;
        int n_chunks = 0;
#define PTR_BEGIN() t0_ = clock64()
#define PTR_END(x) x += clock64() - t0_
#else
#define PTR_BEGIN()
#define PTR_END(x)
#endif
        for (int64_t item = rank; item < nitems; item += nranks, ++it) {
            const int tile = (int)(item % plan.ntiles);
            const int ks0 = uniform(plan.tile_ks0[tile]), ks1 = uniform(plan.tile_ks0[tile + 1]);
            const uint32_t a = it & 1u, aph = (it >> 1) & 1u;
            PTR_BEGIN();
            mbar_wait(smem_u32(&tail->acc_empty[a]), aph ^ 1u);      // the epilogue has drained this accumulator
            PTR_END(t_acc);
            tc_fence_after();
            const uint32_t d = (tmem_base & 0x0000FFFFu) + a * 256u;
            uint32_t accum = 0;
            for (int ks = ks0; ks < ks1; ks += CHUNK_KS) {
                PTR_BEGIN();
                mbar_wait(smem_u32(&tail->w_full[ws]), wph);
                PTR_END(t_w);
                const int nks = min(CHUNK_KS, ks1 - ks);
                const uint32_t wa = w_ring + ws * W_STAGE_BYTES;
                const uint64_t a_hi = make_desc_nosw(wa, NB_PIECE, 128u), a_lo = make_desc_nosw(wa + W_KS / 2, NB_PIECE, 128u);
                for (int h = 0; 2 * h < nks; ++h) {
                    PTR_BEGIN();
                    mbar_wait(smem_u32(&tail->b_full[bs]), bph);
                    PTR_END(t_b);
                    tc_fence_after();
                    const uint32_t ba = b_ring + bs * B_STAGE_BYTES;
                    const uint64_t b_hi = make_desc_mn(ba, B_DOM_BYTES), b_lo = make_desc_mn(ba + B_PLANE_BYTES, B_DOM_BYTES);
                    const bool two = nks - 2 * h >= 2;             // K steps of this half chunk that hold data: 1 or 2
                    const uint64_t ah0 = a_hi + 2 * h * KS_DESC, al0 = a_lo + 2 * h * KS_DESC;
                    if (elect_one()) {
                        umma(d, ah0, b_hi, idesc, accum);                      // Wh Mh
                        if (two) umma(d, ah0 + KS_DESC, b_hi + 128, idesc, 1u);
                        umma(d, al0, b_hi, idesc, 1u);                         // Wl Mh
                        if (two) umma(d, al0 + KS_DESC, b_hi + 128, idesc, 1u);
                        umma(d, ah0, b_lo, idesc, 1u);                         // Wh Ml
                        if (two) umma(d, ah0 + KS_DESC, b_lo + 128, idesc, 1u);
                        umma_commit(smem_u32(&tail->b_empty[bs]));
                    }
                    __syncwarp();
                    accum = 1u;
                    if (++bs == B_STAGES) { bs = 0; bph ^= 1u; }
                }
                if (elect_one()) umma_commit(smem_u32(&tail->w_empty[ws]));
                __syncwarp();
                if (++ws == W_STAGES) { ws = 0; wph ^= 1u; }
#ifdef GNNB_TRACE
                ++n_chunks;
#endif
            }
            if (elect_one()) umma_commit(smem_u32(&tail->acc_full[a]));
            __syncwarp();
        }
#ifdef GNNB_TRACE
        if (rank == 1 && lane == 0) printf("TRACE prop-mma: items %u chunks %d total %lld | wait acc_empty %lld, w_full %lld, b_full %lld\n", it, n_chunks,
                                           clock64() - t_all, t_acc, t_w, t_b);
#endif
    } else if (warp < EPI_WARP0) {
        // ---- gather: warp g copies the rows of subdomain d0 + g, half a chunk (2 K steps, 32 rows) per stage ----
        const int g = warp - GATHER_WARP0;
        const unsigned char* mu_bytes = reinterpret_cast<const unsigned char*>(mu_img);
        uint32_t bs = 0, bph = 0;
#ifdef GNNB_TRACE
        long long g_wait = 0, g_all = clock64(), g0_;
#endif
        for (int64_t item = rank; item < nitems; item += nranks) {
            const int tile = (int)(item % plan.ntiles);
            const int d = (int)(item / plan.ntiles) * PD + g;
            const bool dom_ok = d < Bc;
            const int64_t drow = (int64_t)d * plan.nslots_in;
            const int ks0 = plan.tile_ks0[tile], ks1 = plan.tile_ks0[tile + 1];
            for (int ks = ks0; ks < ks1; ks += 2) {
                // a lane past the tile's last K step (odd step count) is a zero row, like the padding rows of a step
                const int krow = ks * 16 + lane;
                const int idx = krow < ks1 * 16 ? __ldg(plan.ks_rows + krow) : -1;
#ifdef GNNB_TRACE
                g0_ = clock64();
#endif
                mbar_wait(smem_u32(&tail->b_empty[bs]), bph ^ 1u);
#ifdef GNNB_TRACE
                g_wait += clock64() - g0_;
#endif
                const uint32_t dst0 = b_ring + bs * B_STAGE_BYTES + (uint32_t)g * B_DOM_BYTES;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int k = i * 4 + (lane >> 3);               // row of the stage: 4 rows x 8 chunks per instruction
                    const int node = __shfl_sync(0xffffffffu, idx, k);
                    const bool ok = dom_ok && node >= 0;
                    const int64_t grow = ok ? drow + node : 0;
                    const uint32_t r = (uint32_t)(grow & (TILE - 1));
                    const uint32_t jp = (uint32_t)(lane & 7);       // physical 16-byte chunk of the row in the mu image
                    const unsigned char* src = mu_bytes + (grow >> 7) * (int64_t)ABUF + (r >> 3) * 1024u + (r & 7u) * 128u + jp * 16u;
                    const uint32_t dst = dst0 + swz((uint32_t)k, jp ^ (r & 7u));   // logical chunk = physical ^ (row & 7)
                    cp_async16(dst, src, ok);
                    cp_async16(dst + B_PLANE_BYTES, src + APLANE, ok);
                }
                cp_async_arrive(smem_u32(&tail->b_full[bs]));
                if (++bs == B_STAGES) { bs = 0; bph ^= 1u; }
            }
        }
#ifdef GNNB_TRACE
        if (rank == 1 && g == 0 && lane == 0) printf("TRACE prop-gather: total %lld, wait b_empty %lld\n", clock64() - g_all, g_wait);
#endif
    } else if (warp < EPI_WARP0 + 8) {
        // ---- epilogue: warpgroup ew takes the items it & 1 == ew ----
        const int ew = (warp - EPI_WARP0) >> 2;
        const int m = (warp & 3) * 32 + lane;                      // TMEM lane = tile row (a warp reaches lanes 32 * (warp % 4) ..)
        const uint32_t tmem = tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + (uint32_t)ew * 256u;
        const uint32_t full = smem_u32(&tail->acc_full[ew]), empty = smem_u32(&tail->acc_empty[ew]);
        uint32_t aph = 0, it = 0;
#ifdef GNNB_TRACE
        long long e_wait = 0, e_work = 0, e0_;
#endif
        for (int64_t item = rank; item < nitems; item += nranks, ++it) {
            if ((int)(it & 1u) != ew) continue;
            const int tile = (int)(item % plan.ntiles);
            const int d0 = (int)(item / plan.ntiles) * PD;
#ifdef GNNB_TRACE
            e0_ = clock64();
#endif
            mbar_wait(full, aph);
            aph ^= 1u;
            tc_fence_after();
#ifdef GNNB_TRACE
            e_wait += clock64() - e0_; e0_ = clock64();
#endif
#pragma unroll 1
            for (int dom = 0; dom < PD; ++dom) {
                if (d0 + dom >= Bc) break;
                // slot order: the tile's 128 rows are one tile image of the output layer; thread = row, so a warp's store
                // instruction writes 512 contiguous bytes of a piece
                unsigned char* img = reinterpret_cast<unsigned char*>(nb_img) +
                                     ((int64_t)(d0 + dom) * plan.ntiles + tile) * (int64_t)ABUF + (uint32_t)m * 16u;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    float x[16];
                    tmem_ld16_sync(tmem + (uint32_t)(dom * 64 + q * 16), x);
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        uint4 hi, lo;
                        split2(x[h * 8 + 0], x[h * 8 + 1], hi.x, lo.x);
                        split2(x[h * 8 + 2], x[h * 8 + 3], hi.y, lo.y);
                        split2(x[h * 8 + 4], x[h * 8 + 5], hi.z, lo.z);
                        split2(x[h * 8 + 6], x[h * 8 + 7], hi.w, lo.w);
                        const uint32_t off = (uint32_t)(q * 2 + h) * NB_PIECE;
                        *reinterpret_cast<uint4*>(img + off) = hi;
                        *reinterpret_cast<uint4*>(img + APLANE + off) = lo;
                    }
                }
            }
            tc_fence_before();
            mbar_arrive(empty);
#ifdef GNNB_TRACE
            e_work += clock64() - e0_;
#endif
        }
#ifdef GNNB_TRACE
        if (rank == 1 && m == 0) printf("TRACE prop-epi wg %d: wait acc_full %lld, work %lld\n", ew, e_wait, e_work);
#endif
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tmem_base, 512);
}

// ---- host-side plan construction ------------------------------------------------------------------------
struct Edge { int in; float w; };
using EdgeFn = std::function<void(int, std::vector<Edge>&)>;

// tiles of <= 128 nodes on a (C, H, W) grid: all channels (in blocks of <= 128) of a spatial patch
std::vector<std::vector<int>> grid_tiles(int C, int H, int W) {
    const int Cb = std::min(C, TILE), Pp = std::max(1, TILE / Cb);
    int bestY = 1, bestX = 1;
    long bestTiles = -1;
    for (int Yb = 1; Yb <= std::min(H, Pp); ++Yb)
        for (int Xb = 1; Xb <= std::min(W, Pp / Yb); ++Xb) {
            const long tiles = (long)((H + Yb - 1) / Yb) * ((W + Xb - 1) / Xb);
            const bool better = bestTiles < 0 || tiles < bestTiles ||
                                (tiles == bestTiles && std::abs(Yb - Xb) < std::abs(bestY - bestX));
            if (better) { bestTiles = tiles; bestY = Yb; bestX = Xb; }
        }
    std::vector<std::vector<int>> tiles;
    for (int c0 = 0; c0 < C; c0 += Cb)
        for (int y0 = 0; y0 < H; y0 += bestY)
            for (int x0 = 0; x0 < W; x0 += bestX) {
                std::vector<int> rows;
                for (int c = c0; c < std::min(C, c0 + Cb); ++c)
                    for (int y = y0; y < std::min(H, y0 + bestY); ++y)
                        for (int x = x0; x < std::min(W, x0 + bestX); ++x) rows.push_back((c * H + y) * W + x);
                tiles.push_back(rows);
            }
    return tiles;
}

std::vector<std::vector<int>> range_tiles(int n) {
    std::vector<std::vector<int>> tiles;
    for (int r0 = 0; r0 < n; r0 += TILE) {
        std::vector<int> rows;
        for (int r = r0; r < std::min(n, r0 + TILE); ++r) rows.push_back(r);
        tiles.push_back(rows);
    }
    return tiles;
}

PropPlan* build_plan(const LayerTiling& out, const LayerTiling& in, const EdgeFn& edges) {
    std::vector<int32_t> tile_ks0, ks_rows;
    std::vector<uint16_t> ks_w;
    std::vector<Edge> ev;
    std::vector<float> dense;
    double useful = 0.0, issued = 0.0;
    for (int t = 0; t < out.ntiles; ++t) {
        const int32_t* rows = &out.node_of_slot[(size_t)t * TILE];       // -1 = padding slot
        std::vector<std::vector<Edge>> row_edges(TILE);
        std::map<int, int> col;                     // input SLOT -> K index (sorted by slot: neighbouring K rows are neighbouring rows of the mu image)
        for (int m = 0; m < TILE; ++m) {
            if (rows[m] < 0) continue;
            ev.clear();
            edges(rows[m], ev);
            for (Edge& e : ev) { e.in = in.slot_of_node[e.in]; col[e.in] = 0; }
            row_edges[m] = ev;
            useful += (double)ev.size();
        }
        int K = 0;
        for (auto& kv : col) kv.second = K++;
        dense.assign((size_t)TILE * K, 0.f);
        for (int m = 0; m < TILE; ++m)
            for (const Edge& e : row_edges[m]) dense[(size_t)m * K + col[e.in]] += e.w;
        // K steps [0, ceil(K / 16)) of this tile, at least one
        const int nks = std::max(1, (K + 15) / 16);
        issued += 128.0 * 16.0 * nks;
        tile_ks0.push_back((int32_t)(ks_rows.size() / 16));
        const size_t r0 = ks_rows.size(), w0 = ks_w.size();
        ks_rows.resize(r0 + (size_t)nks * 16, -1);
        for (const auto& kv : col) ks_rows[r0 + kv.second] = kv.first;
        ks_w.resize(w0 + (size_t)nks * 4096, 0);                        // 8 KB = 4096 fp16 per K step
        for (int m = 0; m < TILE; ++m)
            for (int k = 0; k < K; ++k) {
                const float x = dense[(size_t)m * K + k];
                if (x == 0.f) continue;
                uint16_t hi, lo;
                split_host(x, hi, lo);
                const int j = k / 16, pce = (k % 16) / 8, e = k % 8;
                const size_t el = w0 + (size_t)j * 4096 + (size_t)pce * 1024 + (size_t)m * 8 + e;      // fp16 elements: piece 2 KB = 1024
                ks_w[el] = hi;
                ks_w[el + 2048] = lo;                                                                  // lo plane 4 KB further
            }
    }
    tile_ks0.push_back((int32_t)(ks_rows.size() / 16));
    PropPlan* p = new PropPlan();
    p->nksteps = (int)(ks_rows.size() / 16);
    p->density = issued > 0 ? useful / issued : 0.0;
    const size_t b_tk = tile_ks0.size() * 4, b_kr = ks_rows.size() * 4, b_kw = ks_w.size() * sizeof(uint16_t);
    auto up = [](size_t x) { return (x + 255) & ~size_t(255); };
    const size_t total = up(b_tk) + up(b_kr) + up(b_kw);
    if (cudaMalloc(&p->blob, total) != cudaSuccess) { delete p; return nullptr; }
    unsigned char* d = reinterpret_cast<unsigned char*>(p->blob);
    size_t off = 0;
    auto put = [&](const void* src, size_t bytes) {
        void* dst = d + off;
        cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice);
        off += up(bytes);
        return dst;
    };
    p->dev.ks_w = reinterpret_cast<const uint16_t*>(put(ks_w.data(), b_kw));
    p->dev.tile_ks0 = reinterpret_cast<const int32_t*>(put(tile_ks0.data(), b_tk));
    p->dev.ks_rows = reinterpret_cast<const int32_t*>(put(ks_rows.data(), b_kr));
    p->dev.ntiles = out.ntiles;
    p->dev.nslots_in = (int)in.node_of_slot.size();
    p->dev.nslots_out = (int)out.node_of_slot.size();
    if (cudaGetLastError() != cudaSuccess) { cudaFree(p->blob); delete p; return nullptr; }
    return p;
}

}  // namespace

LayerTiling make_tiling(int C, int H, int W) {
    const std::vector<std::vector<int>> tiles = (H == 1 && W == 1) ? range_tiles(C) : grid_tiles(C, H, W);
    LayerTiling t;
    t.ntiles = (int)tiles.size();
    t.node_of_slot.assign((size_t)t.ntiles * TILE, -1);
    t.slot_of_node.assign((size_t)C * H * W, -1);
    for (int i = 0; i < t.ntiles; ++i)
        for (size_t m = 0; m < tiles[i].size(); ++m) {
            t.node_of_slot[(size_t)i * TILE + m] = tiles[i][m];
            t.slot_of_node[tiles[i][m]] = i * TILE + (int)m;
        }
    return t;
}

int prop_tc_init() {
    return cudaFuncSetAttribute(k_tc_prop, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)prop::PROP_SMEM);
}

// plan for  nb = A_k(mu)  (forward) or  nb = A_k^T(mu) [/ freq]  (backward) of one verified-network layer;
// `w` is the layer's HOST weight (conv [co,ci,k,k] / linear [out,in])
PropPlan* prop_plan_build(const LayerDev& L, const float* w, bool backward, bool normalise, const LayerTiling& out,
                          const LayerTiling& in) {
    const int k = L.ksize, s = L.stride, p = L.pad;
    if (L.kind == GNNB_LAYER_CONV) {
        const int hw_in = L.h_in * L.w_in, hw_out = L.h_out * L.w_out;
        if (!backward) {
            EdgeFn f = [=](int node, std::vector<Edge>& ev) {
                const int co = node / hw_out, y = (node % hw_out) / L.w_out, x = node % L.w_out;
                for (int ci = 0; ci < L.c_in; ++ci)
                    for (int ky = 0; ky < k; ++ky) {
                        const int yy = y * s + ky - p;
                        if (yy < 0 || yy >= L.h_in) continue;
                        for (int kx = 0; kx < k; ++kx) {
                            const int xx = x * s + kx - p;
                            if (xx < 0 || xx >= L.w_in) continue;
                            ev.push_back({ci * hw_in + yy * L.w_in + xx, w[((co * L.c_in + ci) * k + ky) * k + kx]});
                        }
                    }
            };
            return build_plan(out, in, f);
        }
        EdgeFn f = [=](int node, std::vector<Edge>& ev) {
            const int ci = node / hw_in, yi = (node % hw_in) / L.w_in, xi = node % L.w_in;
            int taps = 0;
            const size_t first = ev.size();
            for (int ky = 0; ky < k; ++ky) {
                const int ty = yi + p - ky;
                if (ty < 0 || ty % s != 0 || ty / s >= L.h_out) continue;
                for (int kx = 0; kx < k; ++kx) {
                    const int tx = xi + p - kx;
                    if (tx < 0 || tx % s != 0 || tx / s >= L.w_out) continue;
                    ++taps;
                    for (int co = 0; co < L.c_out; ++co)
                        ev.push_back({co * hw_out + (ty / s) * L.w_out + tx / s, w[((co * L.c_in + ci) * k + ky) * k + kx]});
                }
            }
            if (normalise && taps > 0)      // conv_transpose2d(.) / freq, freq = tap count (graph_conv.py:306-312)
                for (size_t i = first; i < ev.size(); ++i) ev[i].w = ev[i].w / (float)taps;
        };
        return build_plan(out, in, f);
    }
    if (!backward) {
        EdgeFn f = [=](int node, std::vector<Edge>& ev) {
            for (int i = 0; i < L.n_in; ++i) ev.push_back({i, w[(size_t)node * L.n_in + i]});
        };
        return build_plan(out, in, f);
    }
    EdgeFn f = [=](int node, std::vector<Edge>& ev) {
        for (int o = 0; o < L.n_out; ++o) ev.push_back({o, w[(size_t)o * L.n_in + node]});
    };
    return build_plan(out, in, f);
}

void prop_plan_free(PropPlan* p) {
    if (!p) return;
    if (p->blob) cudaFree(p->blob);
    delete p;
}

double prop_plan_density(const PropPlan* p) { return p ? p->density : 0.0; }
const PropPlanDev& prop_plan_dev(const PropPlan* p) { return p->dev; }
double prop_plan_ksteps_per_tile(const PropPlan* p) { return p->dev.ntiles > 0 ? (double)p->nksteps / p->dev.ntiles : 1.0; }

void prop_tc_run(const PropPlan* plan, const float* mu_img, float* nb_img, int Bc, cudaStream_t st, int64_t* launches) {
    const int64_t nitems = (int64_t)plan->dev.ntiles * ((Bc + prop::PD - 1) / prop::PD);
    const int grid = (int)(nitems < 1 ? 1 : (nitems < 148 ? nitems : 148));
    launch_pdl(k_tc_prop, grid, prop::PROP_THREADS, prop::PROP_SMEM, st, plan->dev,
               reinterpret_cast<const uint16_t*>(mu_img), reinterpret_cast<uint16_t*>(nb_img), Bc);
    ++*launches;
}

// nb[b, n, :] = Wp[b, n] * mu[L+1][b, :] (graph_conv.py:324-326) written as the fp16 tile image
namespace {
__global__ void k_property_backward_img(const float* __restrict__ wp, const float* __restrict__ mu_out,
                                        uint16_t* __restrict__ nb_img, int nL, int nslots, int64_t total8) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total8; i += (int64_t)gridDim.x * blockDim.x) {
        const int chunk = (int)(i & 7);
        const int64_t row = i >> 3;              // b * nslots + slot; the last hidden layer is flat: slot = node
        const int64_t b = row / nslots;
        const int node = (int)(row - b * nslots);
        const float w = node < nL ? wp[b * nL + node] * ASCALE : 0.f;
        const float4 m0 = *reinterpret_cast<const float4*>(mu_out + b * P + chunk * 8);
        const float4 m1 = *reinterpret_cast<const float4*>(mu_out + b * P + chunk * 8 + 4);
        uint4 hi, lo;
        split2(w * m0.x, w * m0.y, hi.x, lo.x);
        split2(w * m0.z, w * m0.w, hi.y, lo.y);
        split2(w * m1.x, w * m1.y, hi.z, lo.z);
        split2(w * m1.z, w * m1.w, hi.w, lo.w);
        unsigned char* img = reinterpret_cast<unsigned char*>(nb_img) + (row / TILE) * (int64_t)ABUF;
        const uint32_t off = (uint32_t)chunk * NB_PIECE + (uint32_t)(row % TILE) * 16u;     // piece-major nb image
        *reinterpret_cast<uint4*>(img + off) = hi;
        *reinterpret_cast<uint4*>(img + APLANE + off) = lo;
    }
}
}  // namespace

void prop_tc_property_backward(const float* wp, const float* mu_out, float* nb_img, int nL, int nslots, int Bc, cudaStream_t st, int64_t* launches) {
    const int64_t total8 = (int64_t)Bc * nslots * 8;
    const int64_t blocks = (total8 + 255) / 256;
    k_property_backward_img<<<(unsigned)(blocks < 1 ? 1 : (blocks < 148 * 16 ? blocks : 148 * 16)), 256, 0, st>>>(
        wp, mu_out, reinterpret_cast<uint16_t*>(nb_img), nL, nslots, total8);
    ++*launches;
}

}  // namespace gnnb
