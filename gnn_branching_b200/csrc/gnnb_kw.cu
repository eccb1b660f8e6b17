// Batched KW (Wong & Kolter) intermediate bounds on the GPU — the bound producer in front of the scoring path
// (SURVEY §8f rank 3): gnnb_kw_bounds (the bounds of init_kw_bounds) and gnnb_child_bounds (the bounds part of
// update_the_model: KW pass from the parent's bounds with one ReLU fixed, interval pass, second KW pass where needed).
//
// Reference: DualNetwork.__init__ of the vendored convex_adversarial (dual_network.py:15-101, dual_layers.py:207-312,
// dual_inputs.py:24-70) as called from init_kw_bounds / update_kw_bounds (plnn/dual_network_linear_approximation.py:205-451)
// and KWConvGen.update_the_model (plnn/conv_kwinter_gen.py:558-660).  The reference
// pushes x, the n0 x n0 identity, the biases and one scaled unit vector per ambiguous ReLU FORWARD through the layers; the
// number of columns depends on the domain.  Here the same numbers are computed by the transposed recursion, whose column
// count is fixed (one column per output neuron), so B domains x 64-column groups batch into the existing propagation
// kernels (oracle/kw_bounds_oracle.py states the forward form and is pinned to the reference; both forms are the same sums).
//
// For output neuron o of layer k:   s_k = e_o;   for j = k-1 .. 1:  t_j = A_{j+1}^T s_{j+1},  s_j = d_j * t_j;   t_0 = A_1^T s_1
//     centre = t_0 . x + sum_{j<=k} s_j . b_j
//     zl_k[o] = centre - eps |t_0|_1 + sum_{j<k} sum_{i in I_j} zl_j[i] relu(-s_j[i])
//     zu_k[o] = centre + eps |t_0|_1 - sum_{j<k} sum_{i in I_j} zl_j[i] relu(+s_j[i])
// with d_j = [zl_j >= 0] + I_j zu_j / (zu_j - zl_j), I_j = [zl_j < 0 < zu_j] from the (already final) bounds of layer j, then
// intersected with the provided bounds of the parent domain (dual_network.py:85-86).  A_j^T is prop_backward without the
// tap-count normalisation (gnnb_prop.cu), 64 columns riding in the 64 "embedding channels" of a [pairs, n, 64] tensor,
// pair = (domain, column group).  A pass may run on a subset of the domains (dom_list) and may leave the first hidden
// layers of a domain untouched (keep_upto: update_kw_bounds keeps the layers up to the split).
#include <string>
#include <vector>

#include "gnnb_common.cuh"
#include "gnnb_umma.cuh"

namespace gnnb {
namespace {

constexpr int KW_COLS = P;          // columns per pair = the channel width of the propagation kernels
constexpr int KW_MAX_LAYERS = 30;   // hidden layers a child-bounds call can handle (pointer tables passed by value)

// s_k of a column group: buf[pair][node][c] = (node == g * 64 + c)
__global__ void k_kw_onehot(float* __restrict__ buf, int n, int G, int64_t p0, int64_t total4) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total4) return;
    const int c4 = (int)(i & 15);
    const int64_t row = i >> 4;                      // pair_local * n + node
    const int node = (int)(row % n);
    const int g = (int)((p0 + row / n) % G);
    const int c = node - g * KW_COLS;                // the column whose unit vector has its 1 at this node
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c >= c4 * 4 && c < c4 * 4 + 4) reinterpret_cast<float*>(&v)[c - c4 * 4] = 1.0f;
    reinterpret_cast<float4*>(buf)[i] = v;
}

// t_L of the property output: column 0 = Wp[b, :], the other columns 0 (one pair per domain)
__global__ void k_kw_wp_col(float* __restrict__ buf, const float* __restrict__ wp, int nL, int64_t b0, int64_t total4,
                            const int32_t* __restrict__ dom_list) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total4) return;
    const int c4 = (int)(i & 15);
    const int64_t row = i >> 4;                      // pair_local * nL + node
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    const int64_t bl = b0 + row / nL, b = dom_list ? dom_list[bl] : bl;
    if (c4 == 0) v.x = wp[b * nL + row % nL];
    reinterpret_cast<float4*>(buf)[i] = v;
}

struct KwAcc { float *cx, *l1, *bias, *low, *up; };      // [pairs][64] each

// t_j -> s_j = d_j * t_j in place, and the three sums over the nodes of layer j.  One block per pair, thread = (part, column).
__global__ void __launch_bounds__(256) k_kw_reduce_layer(float* __restrict__ t, const float* __restrict__ zl, const float* __restrict__ zu,
                                                         const float* __restrict__ bias_node, int n, int G, int64_t p0, KwAcc acc,
                                                         const int32_t* __restrict__ dom_list) {
    __shared__ float red[3][4][KW_COLS];
    const int64_t pl = blockIdx.x, bl = (p0 + pl) / G, b = dom_list ? dom_list[bl] : bl;
    const int c = threadIdx.x & 63, part = threadIdx.x >> 6;
    float sb = 0.f, sl = 0.f, su = 0.f;
    for (int i = part; i < n; i += 4) {
        const float l = zl[b * n + i], u = zu[b * n + i];
        const bool I = (u > 0.f) && (l < 0.f);
        float d = (l >= 0.f) ? 1.0f : 0.0f;
        if (I) d += __fdiv_rn(u, u - l);
        float* q = t + ((int64_t)pl * n + i) * KW_COLS + c;
        const float s = *q * d;
        *q = s;
        sb = fmaf(s, bias_node[i], sb);
        if (I) { sl = fmaf(l, fmaxf(-s, 0.f), sl); su = fmaf(l, fmaxf(s, 0.f), su); }
    }
    red[0][part][c] = sb; red[1][part][c] = sl; red[2][part][c] = su;
    __syncthreads();
    if (part == 0) {
        const int64_t o = pl * KW_COLS + c;
        acc.bias[o] += (red[0][0][c] + red[0][1][c]) + (red[0][2][c] + red[0][3][c]);
        acc.low[o] += (red[1][0][c] + red[1][1][c]) + (red[1][2][c] + red[1][3][c]);
        acc.up[o] += (red[2][0][c] + red[2][1][c]) + (red[2][2][c] + red[2][3][c]);
    }
}

// t_0 . x and |t_0|_1
__global__ void __launch_bounds__(256) k_kw_reduce_input(const float* __restrict__ t, const float* __restrict__ x, int n0, int G, int64_t p0,
                                                         KwAcc acc, const int32_t* __restrict__ dom_list) {
    __shared__ float red[2][4][KW_COLS];
    const int64_t pl = blockIdx.x, bl = (p0 + pl) / G, b = dom_list ? dom_list[bl] : bl;
    const int c = threadIdx.x & 63, part = threadIdx.x >> 6;
    float sx = 0.f, s1 = 0.f;
    for (int i = part; i < n0; i += 4) {
        const float v = t[((int64_t)pl * n0 + i) * KW_COLS + c];
        sx = fmaf(v, x[b * n0 + i], sx);
        s1 += fabsf(v);
    }
    red[0][part][c] = sx; red[1][part][c] = s1;
    __syncthreads();
    if (part == 0) {
        const int64_t o = pl * KW_COLS + c;
        acc.cx[o] = (red[0][0][c] + red[0][1][c]) + (red[0][2][c] + red[0][3][c]);
        acc.l1[o] = (red[1][0][c] + red[1][1][c]) + (red[1][2][c] + red[1][3][c]);
    }
}

// bounds of the group's columns, intersected with the provided ones; own_bias: bias of the layer per node (hidden layers) or
// the property bias per domain (ncols == 1); layer: 1-based index of the layer, left untouched for domains with
// keep_upto[b] >= layer
__global__ void k_kw_finish(KwAcc acc, int ncols, int G, int64_t p0, int64_t npairs, float eps, const float* __restrict__ bias_node,
                            const float* __restrict__ bp, const float* prov_lb, const float* prov_ub,      // may alias out_lb / out_ub
                            float* out_lb, float* out_ub, const int32_t* __restrict__ dom_list,
                            const int32_t* __restrict__ keep_upto, int layer) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npairs * KW_COLS) return;
    const int64_t pl = i / KW_COLS, p = p0 + pl, bl = p / G, b = dom_list ? dom_list[bl] : bl;
    const int o = (int)(p % G) * KW_COLS + (int)(i % KW_COLS);
    if (o >= ncols) return;
    if (keep_upto && keep_upto[b] >= layer) return;
    const float own = bias_node ? bias_node[o] : bp[b];
    const float centre = acc.cx[i] + (acc.bias[i] + own);
    float zl = centre - eps * acc.l1[i] + acc.low[i];
    float zu = centre + eps * acc.l1[i] - acc.up[i];
    const int64_t at = b * ncols + o;
    if (prov_lb) zl = fmaxf(zl, prov_lb[at]);
    if (prov_ub) zu = fminf(zu, prov_ub[at]);
    out_lb[at] = zl;
    out_ub[at] = zu;
}

__global__ void k_kw_input_box(const float* __restrict__ x, float eps, int64_t total, float* __restrict__ lb, float* __restrict__ ub) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    lb[i] = x[i] - eps;
    ub[i] = x[i] + eps;
}

unsigned blocks_of(int64_t n, int per) { return (unsigned)((n + per - 1) / per < 1 ? 1 : (n + per - 1) / per); }

// ---- child domains (update_the_model) -----------------------------------------------------------------------------------
// the split of update_kw_bounds (plnn/dual_network_linear_approximation.py:313-319): u = 0 (choice 0) or l = 0 (choice 1) at
// the decided ReLU; keep_upto[b] = 1-based index of the decided layer (its bounds and those in front of it are final)
struct BoundPtrs { float* lb[KW_MAX_LAYERS + 2]; float* ub[KW_MAX_LAYERS + 2]; int n[KW_MAX_LAYERS + 2]; };
__global__ void k_child_split(BoundPtrs o, int L, int B, const int32_t* __restrict__ dec_layer, const int32_t* __restrict__ dec_index,
                              const int32_t* __restrict__ choice, int32_t* __restrict__ keep_upto, int32_t* __restrict__ changed) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int lay = dec_layer[b], idx = dec_index[b];
    changed[b] = 0;
    if (lay < 0 || lay >= L || idx < 0 || idx >= o.n[lay + 1]) { keep_upto[b] = L; return; }      // no valid decision: nothing behind it to refresh
    keep_upto[b] = lay + 1;
    if (choice[b] == 0) o.ub[lay + 1][(int64_t)b * o.n[lay + 1] + idx] = 0.f;
    else o.lb[lay + 1][(int64_t)b * o.n[lay + 1] + idx] = 0.f;
}

// Does an interval bound that beats the current one call for the second KW pass?  The reference repeats the pass on ANY strict
// improvement (:630-641), which includes last-bit differences between two evaluations of the same sum: root bounds are
// themselves KW bounds intersected with interval bounds, so wherever the interval bound was the tighter one at the root the
// child's interval bound is the same number up to summation order.  The tighter bound is always taken; the pass is repeated
// only for gains above rounding (1e-6 relative), whose effect on later layers is above rounding too.
__device__ __forceinline__ bool interval_gain_counts(float better, float current) {
    return fabsf(better - current) > 1e-6f * fmaxf(1.0f, fabsf(current));
}

// the tighter of the interval and the current bound, and the note for the second KW pass.  Child domains (root = 0): changed = 1
// when a hidden layer's bound moved (conv_kwinter_gen.py:652).  Root (build_the_model, :262-267): changed = the FIRST hidden
// layer whose bound moved by more than 1e-4 (the reference's test), kept as a minimum over the nodes.
__device__ __forceinline__ void interval_commit(float lo, float hi, float* lb, float* ub, int32_t* changed, int layer, bool hidden, int root) {
    bool ch = false;
    const float l0 = *lb, u0 = *ub;
    if (lo > l0) { ch |= root ? (lo - l0 > 1e-4f) : interval_gain_counts(lo, l0); *lb = lo; }
    if (hi < u0) { ch |= root ? (u0 - hi > 1e-4f) : interval_gain_counts(hi, u0); *ub = hi; }
    if (ch && hidden) { if (root) atomicMin(changed, layer); else *changed = 1; }
}

// interval bounds of one layer from the post-ReLU box of the layer in front of it, intersected with the current bounds
// (plnn/conv_kwinter_gen.py:594-641: W+ l + W- u + b / W+ u + W- l + b); only for domains whose split lies in front of the
// layer; changed[b] is raised when a HIDDEN layer's bound moved (:652: only then the KW pass is repeated)
__global__ void __launch_bounds__(256) k_interval_conv(LayerDev Ld, const float* __restrict__ lb_in, const float* __restrict__ ub_in,
                                                       float* __restrict__ lb, float* __restrict__ ub, int B, int layer,
                                                       const int32_t* __restrict__ keep_upto, int32_t* __restrict__ changed, int root) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)B * Ld.n_out) return;
    const int b = (int)(i / Ld.n_out), node = (int)(i % Ld.n_out);
    if (keep_upto[b] >= layer) return;
    const int hw = Ld.h_out * Ld.w_out, co = node / hw, y = (node % hw) / Ld.w_out, x = node % Ld.w_out;
    const float* li = lb_in + (int64_t)b * Ld.n_in;
    const float* ui = ub_in + (int64_t)b * Ld.n_in;
    float lo = Ld.bias_node[node], hi = lo;
    for (int ci = 0; ci < Ld.c_in; ++ci)
        for (int ky = 0; ky < Ld.ksize; ++ky) {
            const int yy = y * Ld.stride + ky - Ld.pad;
            if (yy < 0 || yy >= Ld.h_in) continue;
            for (int kx = 0; kx < Ld.ksize; ++kx) {
                const int xx = x * Ld.stride + kx - Ld.pad;
                if (xx < 0 || xx >= Ld.w_in) continue;
                const float w = Ld.weight[((co * Ld.c_in + ci) * Ld.ksize + ky) * Ld.ksize + kx];
                const int at = (ci * Ld.h_in + yy) * Ld.w_in + xx;
                const bool raw = root && layer == 1;                     // the first layer reads the input box itself
                const float l = raw ? li[at] : fmaxf(li[at], 0.f), u = raw ? ui[at] : fmaxf(ui[at], 0.f);
                lo = fmaf(w, w > 0.f ? l : u, lo);
                hi = fmaf(w, w > 0.f ? u : l, hi);
            }
        }
    interval_commit(lo, hi, lb + i, ub + i, changed + b, layer, true, root);
}

// linear layer (and, with per-domain weights wp / bias bp, the property output): one warp per (domain, output)
__global__ void __launch_bounds__(256) k_interval_linear(const float* __restrict__ W, const float* __restrict__ bias, int64_t w_dom_stride,
                                                         int n_in, int n_out, const float* __restrict__ lb_in, const float* __restrict__ ub_in,
                                                         float* __restrict__ lb, float* __restrict__ ub, int B, int layer, bool hidden,
                                                         const int32_t* __restrict__ keep_upto, int32_t* __restrict__ changed, int root) {
    const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (wid >= (int64_t)B * n_out) return;
    const int b = (int)(wid / n_out), o = (int)(wid % n_out);
    if (keep_upto[b] >= layer) return;
    const float* w = W + (int64_t)b * w_dom_stride + (int64_t)o * n_in;
    const float* li = lb_in + (int64_t)b * n_in;
    const float* ui = ub_in + (int64_t)b * n_in;
    float lo = 0.f, hi = 0.f;
    for (int i = lane; i < n_in; i += 32) {
        const bool raw = root && layer == 1;
        const float wv = w[i], l = raw ? li[i] : fmaxf(li[i], 0.f), u = raw ? ui[i] : fmaxf(ui[i], 0.f);
        lo = fmaf(wv, wv > 0.f ? l : u, lo);
        hi = fmaf(wv, wv > 0.f ? u : l, hi);
    }
    for (int d = 16; d > 0; d >>= 1) { lo += __shfl_xor_sync(0xffffffffu, lo, d); hi += __shfl_xor_sync(0xffffffffu, hi, d); }
    if (lane != 0) return;
    const float bv = w_dom_stride ? bias[b] : bias[o];
    lo += bv; hi += bv;
    interval_commit(lo, hi, lb + wid, ub + wid, changed + b, layer, hidden, root);
}

// the domains whose hidden bounds moved, in index order (one block; B is a frontier batch, thousands at most)
__global__ void __launch_bounds__(1024) k_collect_changed(const int32_t* __restrict__ changed, int B, int32_t* __restrict__ list, int32_t* __restrict__ count) {
    __shared__ int32_t warp_tot[32];
    __shared__ int32_t base;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (int b0 = 0; b0 < B; b0 += 1024) {
        const int b = b0 + threadIdx.x;
        const bool f = b < B && changed[b] != 0;
        const unsigned bal = __ballot_sync(0xffffffffu, f);
        if ((threadIdx.x & 31) == 0) warp_tot[threadIdx.x >> 5] = __popc(bal);
        __syncthreads();
        int before = base;
        for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) before += warp_tot[w];
        if (f) list[before + __popc(bal & ((1u << (threadIdx.x & 31)) - 1u))] = b;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < 32; ++w) t += warp_tot[w]; base += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = base;
}

// root: first changed layer (or INT_MAX) -> keep_upto (that layer stays as the interval pass left it; nothing to redo: L) and the
// 0 / 1 flag of the domains that need the KW pass
__global__ void k_root_prepare(int32_t* __restrict__ changed, int32_t* __restrict__ keep, int B, int L) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int c = changed[b];
    keep[b] = c <= L ? c : L;
    changed[b] = c <= L ? 1 : 0;
}

// ReLU phase of every hidden node from its pre-activation bounds, in the BaB convention (plnn/conv_kwinter_gen.py:696-713:
// passing 1, blocked 0, ambiguous -1)
__global__ void k_mask_from_bounds(const float* __restrict__ lb, const float* __restrict__ ub, int8_t* __restrict__ mask, int64_t total) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const float l = lb[i], u = ub[i];
    mask[i] = (l >= 0.f && u >= 0.f) ? 1 : ((l <= 0.f && u <= 0.f) ? 0 : -1);
}


// ---- dense layers on the tensor cores ------------------------------------------------------------------------------------
// The column blocks of the dense recursion are exactly what the GNN's propagation kernel moves: [pairs, n, 64] with 64 columns
// in the 64 "embedding channels".  With the un-normalised transposed plans (KwTc::plans) k_tc_prop computes t_j = A_{j+1}^T s_{j+1}
// on the tensor cores (fp16 hi / lo split, three passes, fp32 accumulate: 2^-22 per product, bounds are held to 2e-5); the
// tensors travel in the tile-image formats of that kernel (gnnb_umma.cuh): s_j as a mu image (slot order, K-major
// SWIZZLE_128B planes), t_j as the piece-major nb image.  Unscaled values: |t| stays far below fp16's range.
using namespace tcx;

// s_k of a column group as a mu image: row of slot r, channel c = (node_of_slot[r] == g * 64 + c)
__global__ void k_kw_img_onehot(uint16_t* __restrict__ mu_img, RowMap map, int G, int64_t p0, int64_t total) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;       // (pair-local row, chunk of 8 channels)
    if (i >= total) return;
    const int chunk = (int)(i & 7);
    const int64_t row = i >> 3, pl = row / map.nslots;
    const int slot = (int)(row - pl * map.nslots);
    const int node = map.node_of_slot[slot];
    const int g = (int)((p0 + pl) % G);
    const int c = node - g * KW_COLS - chunk * 8;                            // position of the 1 inside this chunk, if any
    uint4 hi = make_uint4(0u, 0u, 0u, 0u);
    if (node >= 0 && c >= 0 && c < 8) reinterpret_cast<uint16_t*>(&hi)[c] = 0x3C00u;      // fp16 1.0
    unsigned char* img = reinterpret_cast<unsigned char*>(mu_img) + (row / TILE) * (int64_t)ABUF;
    const uint32_t off = swz((uint32_t)(row % TILE), (uint32_t)chunk);
    *reinterpret_cast<uint4*>(img + off) = hi;
    *reinterpret_cast<uint4*>(img + APLANE + off) = make_uint4(0u, 0u, 0u, 0u);
}

// t_L of the property output as an nb image: channel 0 = Wp[b, node], the other channels 0 (one pair per domain)
__global__ void k_kw_img_wp(uint16_t* __restrict__ nb_img, const float* __restrict__ wp, RowMap map, int64_t p0, int64_t total,
                            const int32_t* __restrict__ dom_list) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;       // (pair-local row, piece of 8 channels)
    if (i >= total) return;
    const int piece = (int)(i & 7);
    const int64_t row = i >> 3, pl = row / map.nslots;
    const int slot = (int)(row - pl * map.nslots);
    const int node = map.node_of_slot[slot];
    const int64_t b = dom_list ? dom_list[p0 + pl] : p0 + pl;
    uint4 hi = make_uint4(0u, 0u, 0u, 0u), lo = hi;
    if (piece == 0 && node >= 0) split2(wp[b * map.n + node], 0.f, hi.x, lo.x);
    unsigned char* img = reinterpret_cast<unsigned char*>(nb_img) + (row / TILE) * (int64_t)ABUF;
    const uint32_t off = (uint32_t)piece * NB_PIECE + (uint32_t)(row % TILE) * 16u;
    *reinterpret_cast<uint4*>(img + off) = hi;
    *reinterpret_cast<uint4*>(img + APLANE + off) = lo;
}

__device__ __forceinline__ void unpack8(const uint4& hi, const uint4& lo, float (&v)[8]) {
    const __half2* h = reinterpret_cast<const __half2*>(&hi);
    const __half2* l = reinterpret_cast<const __half2*>(&lo);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        v[2 * q] = __low2float(h[q]) + __low2float(l[q]);
        v[2 * q + 1] = __high2float(h[q]) + __high2float(l[q]);
    }
}

// t_j (nb image) -> s_j = d_j * t_j (mu image) and the layer's three sums per column.  One block per pair, which walks the tiles of
// the layer in order (deterministic sums): thread = (row of the tile, half of the channels) in phase 1, (row quarter, column)
// in phase 2.  layer_is_input: t_0 instead — t_0 . x and |t_0|_1, nothing written back.
__global__ void __launch_bounds__(256) k_kw_img_reduce(const uint16_t* __restrict__ t_img, uint16_t* __restrict__ s_img, RowMap map,
                                                       const float* __restrict__ zl, const float* __restrict__ zu,
                                                       const float* __restrict__ bias_node, const float* __restrict__ x, int G, int64_t p0,
                                                       KwAcc acc, const int32_t* __restrict__ dom_list, int layer_is_input) {
    __shared__ float S[TILE][KW_COLS + 1];
    __shared__ float rowA[TILE], rowB[TILE];        // hidden: l (0 unless the row is in I) and bias; input: x and unused
    __shared__ float red[3][4][KW_COLS];
    const int64_t pl = blockIdx.x, bl = (p0 + pl) / G, b = dom_list ? dom_list[bl] : bl;
    const int tid = threadIdx.x, r = tid >> 1, half = tid & 1;
    const int q = tid >> 6, c = tid & 63;
    const int ntiles = map.nslots / TILE;
    float s0 = 0.f, s1 = 0.f, s2 = 0.f;
    for (int tile = 0; tile < ntiles; ++tile) {
        const int node = map.node_of_slot[tile * TILE + r];
        float d = 0.f, la = 0.f, bi = 0.f;
        if (node >= 0) {
            if (layer_is_input) { la = x[b * map.n + node]; d = 1.0f; }
            else {
                const float l = zl[b * map.n + node], u = zu[b * map.n + node];
                const bool I = (u > 0.f) && (l < 0.f);
                d = (l >= 0.f) ? 1.0f : 0.0f;
                if (I) { d += __fdiv_rn(u, u - l); la = l; }
                bi = bias_node[node];
            }
        }
        if (half == 0) { rowA[r] = la; rowB[r] = bi; }
        const unsigned char* ti = reinterpret_cast<const unsigned char*>(t_img) + ((int64_t)pl * ntiles + tile) * ABUF;
        unsigned char* si = reinterpret_cast<unsigned char*>(s_img) + ((int64_t)pl * ntiles + tile) * ABUF;
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) {
            const int chunk = half * 4 + cc;
            const uint32_t toff = (uint32_t)chunk * NB_PIECE + (uint32_t)r * 16u;
            float v[8];
            unpack8(*reinterpret_cast<const uint4*>(ti + toff), *reinterpret_cast<const uint4*>(ti + APLANE + toff), v);
#pragma unroll
            for (int e = 0; e < 8; ++e) { v[e] *= d; S[r][chunk * 8 + e] = v[e]; }
            if (!layer_is_input) {
                uint4 hi, lo;
                split2(v[0], v[1], hi.x, lo.x); split2(v[2], v[3], hi.y, lo.y); split2(v[4], v[5], hi.z, lo.z); split2(v[6], v[7], hi.w, lo.w);
                const uint32_t soff = swz((uint32_t)r, (uint32_t)chunk);
                *reinterpret_cast<uint4*>(si + soff) = hi;
                *reinterpret_cast<uint4*>(si + APLANE + soff) = lo;
            }
        }
        __syncthreads();
        for (int rr = q * 32; rr < q * 32 + 32; ++rr) {
            const float sv = S[rr][c], a = rowA[rr];
            if (layer_is_input) { s0 = fmaf(sv, a, s0); s1 += fabsf(sv); }
            else {
                s0 = fmaf(sv, rowB[rr], s0);
                s1 = fmaf(a, fmaxf(-sv, 0.f), s1);        // a = l for rows in I, 0 otherwise
                s2 = fmaf(a, fmaxf(sv, 0.f), s2);
            }
        }
        __syncthreads();
    }
    red[0][q][c] = s0; red[1][q][c] = s1; red[2][q][c] = s2;
    __syncthreads();
    if (q == 0) {
        const int64_t o = pl * KW_COLS + c;
        const float a0 = (red[0][0][c] + red[0][1][c]) + (red[0][2][c] + red[0][3][c]);
        const float a1 = (red[1][0][c] + red[1][1][c]) + (red[1][2][c] + red[1][3][c]);
        const float a2 = (red[2][0][c] + red[2][1][c]) + (red[2][2][c] + red[2][3][c]);
        if (layer_is_input) { acc.cx[o] = a0; acc.l1[o] = a1; }
        else { acc.bias[o] += a0; acc.low[o] += a1; acc.up[o] += a2; }
    }
}

// ---- conv layers: one column's backward cone is local -------------------------------------------------------------------
// For a conv layer k whose predecessors are all conv layers, the column e_o of output o = (co, y, x) touches only the kernel
// footprint of (y, x) in layer k - 1, the footprint of that in layer k - 2, ... : a window of a few hundred nodes per layer
// instead of the whole layer (base conv2: 128 of 2 048 nodes of layer 1, 300 of 3 072 input pixels).  The dense recursion above
// spends > 95 % of its work on zeros there.  This kernel runs the same recursion on the windows: one block per (domain,
// position (y, x)), columns = the C_k output channels at that position (they share the cone), the window tensors
// [element][column] in shared memory, ping-pong.  Same sums as the dense form, different summation order.
constexpr int CONE_MAX_DEPTH = 8;
constexpr int CONE_MAX_SMEM = 200 * 1024;     // dynamic shared memory of k_kw_cone, opted in per device by kw_init
struct ConeArgs {
    LayerDev layer[CONE_MAX_DEPTH];      // A_1 .. A_k
    const float* zl[CONE_MAX_DEPTH];     // bounds of layers 1 .. k - 1 (index j - 1), [B, n_j]
    const float* zu[CONE_MAX_DEPTH];
    int k;                               // the layer whose bounds are computed (1-based), 2 <= k <= CONE_MAX_DEPTH
    int cols, R;                         // columns = C_k; threads = cols * R
    int buf_elems;                       // floats per ping-pong buffer
    const float* x;                      // [B, n0]
    float eps;
    float* out_lb; float* out_ub;        // [B, n_k], provided bounds on entry (intersection in place)
    const int32_t* dom_list; const int32_t* keep_upto;
};

__global__ void __launch_bounds__(256) k_kw_cone(const __grid_constant__ ConeArgs a) {
    extern __shared__ float cone_smem[];
    const int k = a.k, cols = a.cols;
    const int bl = blockIdx.y, b = a.dom_list ? a.dom_list[bl] : bl;
    if (a.keep_upto && a.keep_upto[b] >= k) return;
    const LayerDev& Lk = a.layer[k - 1];
    const int y = blockIdx.x / Lk.w_out, x = blockIdx.x % Lk.w_out;
    // windows of layers k-1 .. 0: [ylo, yhi] x [xlo, xhi], all channels (one table per block in shared memory: indexed by a loop
    // variable, a per-thread copy would live in local memory)
    __shared__ int ylo[CONE_MAX_DEPTH + 1], yhi[CONE_MAX_DEPTH + 1], xlo[CONE_MAX_DEPTH + 1], xhi[CONE_MAX_DEPTH + 1];
    if (threadIdx.x == 0) {
        ylo[k] = yhi[k] = y; xlo[k] = xhi[k] = x;
        for (int j = k; j >= 1; --j) {
            const LayerDev& L = a.layer[j - 1];
            ylo[j - 1] = max(0, ylo[j] * L.stride - L.pad); yhi[j - 1] = min(L.h_in - 1, yhi[j] * L.stride - L.pad + L.ksize - 1);
            xlo[j - 1] = max(0, xlo[j] * L.stride - L.pad); xhi[j - 1] = min(L.w_in - 1, xhi[j] * L.stride - L.pad + L.ksize - 1);
        }
    }
    __syncthreads();
    float* cur = cone_smem;
    float* nxt = cone_smem + a.buf_elems;
    const int tid = threadIdx.x, nthr = cols * a.R, col = tid % cols;
    float acc_bias = 0.f, acc_low = 0.f, acc_up = 0.f, acc_cx = 0.f, acc_l1 = 0.f;
    // t_{k-1} = A_k^T e_o: the kernel footprint of (y, x), column co = row co of the kernel
    {
        const int hj = yhi[k - 1] - ylo[k - 1] + 1, wj = xhi[k - 1] - xlo[k - 1] + 1, E = Lk.c_in * hj * wj;
        for (int idx = tid; idx < E * cols; idx += nthr) {
            const int e = idx / cols, ci = e / (hj * wj), wy = (e / wj) % hj, wx = e % wj;
            const int ky = ylo[k - 1] + wy - (y * Lk.stride - Lk.pad), kx = xlo[k - 1] + wx - (x * Lk.stride - Lk.pad);
            cur[idx] = Lk.weight[((col * Lk.c_in + ci) * Lk.ksize + ky) * Lk.ksize + kx];
        }
    }
    __syncthreads();
    for (int j = k - 1; j >= 1; --j) {
        const LayerDev& Lj = a.layer[j - 1];          // A_j: layer j - 1 -> layer j
        const int hj = yhi[j] - ylo[j] + 1, wj = xhi[j] - xlo[j] + 1, E = Lj.c_out * hj * wj;
        const float* zl = a.zl[j - 1] + (int64_t)b * Lj.n_out;
        const float* zu = a.zu[j - 1] + (int64_t)b * Lj.n_out;
        // s_j = d_j t_j and the layer's three sums
        for (int idx = tid; idx < E * cols; idx += nthr) {
            const int e = idx / cols, c = e / (hj * wj), wy = (e / wj) % hj, wx = e % wj;
            const int node = (c * Lj.h_out + ylo[j] + wy) * Lj.w_out + xlo[j] + wx;
            const float l = zl[node], u = zu[node];
            const bool I = (u > 0.f) && (l < 0.f);
            float d = (l >= 0.f) ? 1.0f : 0.0f;
            if (I) d += __fdiv_rn(u, u - l);
            const float sv = cur[idx] * d;
            cur[idx] = sv;
            acc_bias = fmaf(sv, Lj.bias_node[node], acc_bias);
            if (I) { acc_low = fmaf(l, fmaxf(-sv, 0.f), acc_low); acc_up = fmaf(l, fmaxf(sv, 0.f), acc_up); }
        }
        __syncthreads();
        // t_{j-1} = A_j^T s_j on the window of layer j - 1.  Columns in blocks of 8 per thread when they come in eights (a weight is
        // loaded once per 8 products, the 8 column values with two 16-byte shared-memory loads), one by one otherwise
        const int hi = yhi[j - 1] - ylo[j - 1] + 1, wi = xhi[j - 1] - xlo[j - 1] + 1, Ei = Lj.c_in * hi * wi;
        const int64_t wstride = (int64_t)Lj.c_in * Lj.ksize * Lj.ksize;
        const int cstride = hj * wj * cols;
        if ((cols & 7) == 0) {
            const int CG = cols >> 3;
            for (int idx = tid; idx < Ei * CG; idx += nthr) {
                const int e = idx / CG, cg = idx - e * CG, ci = e / (hi * wi), yy = ylo[j - 1] + (e / wi) % hi, xx = xlo[j - 1] + e % wi;
                float sum[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                for (int ky = 0; ky < Lj.ksize; ++ky) {
                    const int ty = yy + Lj.pad - ky;
                    if (ty < 0 || ty % Lj.stride != 0) continue;
                    const int oy = ty / Lj.stride;
                    if (oy < ylo[j] || oy > yhi[j]) continue;
                    for (int kx = 0; kx < Lj.ksize; ++kx) {
                        const int tx = xx + Lj.pad - kx;
                        if (tx < 0 || tx % Lj.stride != 0) continue;
                        const int ox = tx / Lj.stride;
                        if (ox < xlo[j] || ox > xhi[j]) continue;
                        const float* w = Lj.weight + (ci * Lj.ksize + ky) * Lj.ksize + kx;
                        const float* sp = cur + ((oy - ylo[j]) * wj + (ox - xlo[j])) * cols + cg * 8;
                        for (int c = 0; c < Lj.c_out; ++c) {
                            const float wv = __ldg(w + c * wstride);
                            const float4 s0 = *reinterpret_cast<const float4*>(sp + c * cstride);
                            const float4 s1 = *reinterpret_cast<const float4*>(sp + c * cstride + 4);
                            sum[0] = fmaf(wv, s0.x, sum[0]); sum[1] = fmaf(wv, s0.y, sum[1]); sum[2] = fmaf(wv, s0.z, sum[2]); sum[3] = fmaf(wv, s0.w, sum[3]);
                            sum[4] = fmaf(wv, s1.x, sum[4]); sum[5] = fmaf(wv, s1.y, sum[5]); sum[6] = fmaf(wv, s1.z, sum[6]); sum[7] = fmaf(wv, s1.w, sum[7]);
                        }
                    }
                }
                float4* o = reinterpret_cast<float4*>(nxt + e * cols + cg * 8);
                o[0] = make_float4(sum[0], sum[1], sum[2], sum[3]);
                o[1] = make_float4(sum[4], sum[5], sum[6], sum[7]);
            }
        } else {
            for (int idx = tid; idx < Ei * cols; idx += nthr) {
                const int e = idx / cols, ci = e / (hi * wi), yy = ylo[j - 1] + (e / wi) % hi, xx = xlo[j - 1] + e % wi;
                float sum = 0.f;
                for (int ky = 0; ky < Lj.ksize; ++ky) {
                    const int ty = yy + Lj.pad - ky;
                    if (ty < 0 || ty % Lj.stride != 0) continue;
                    const int oy = ty / Lj.stride;
                    if (oy < ylo[j] || oy > yhi[j]) continue;
                    for (int kx = 0; kx < Lj.ksize; ++kx) {
                        const int tx = xx + Lj.pad - kx;
                        if (tx < 0 || tx % Lj.stride != 0) continue;
                        const int ox = tx / Lj.stride;
                        if (ox < xlo[j] || ox > xhi[j]) continue;
                        const float* w = Lj.weight + (ci * Lj.ksize + ky) * Lj.ksize + kx;
                        const float* sp = cur + ((oy - ylo[j]) * wj + (ox - xlo[j])) * cols + col;
                        for (int c = 0; c < Lj.c_out; ++c) sum = fmaf(w[c * wstride], sp[c * cstride], sum);
                    }
                }
                nxt[idx] = sum;
            }
        }
        __syncthreads();
        float* t = cur; cur = nxt; nxt = t;
    }
    // t_0 . x and |t_0|_1 on the input window
    {
        const LayerDev& L1 = a.layer[0];
        const int hi = yhi[0] - ylo[0] + 1, wi = xhi[0] - xlo[0] + 1, Ei = L1.c_in * hi * wi;
        const float* xb = a.x + (int64_t)b * L1.n_in;
        for (int idx = tid; idx < Ei * cols; idx += nthr) {
            const int e = idx / cols, ci = e / (hi * wi), yy = ylo[0] + (e / wi) % hi, xx = xlo[0] + e % wi;
            const float v = cur[idx];
            acc_cx = fmaf(v, xb[(ci * L1.h_in + yy) * L1.w_in + xx], acc_cx);
            acc_l1 += fabsf(v);
        }
    }
    __syncthreads();
    // the R partial sums of every column
    float* red = cone_smem;                   // 5 * nthr floats <= buf_elems (checked on the host)
    red[0 * nthr + tid] = acc_bias; red[1 * nthr + tid] = acc_low; red[2 * nthr + tid] = acc_up; red[3 * nthr + tid] = acc_cx; red[4 * nthr + tid] = acc_l1;
    __syncthreads();
    if (tid < cols) {
        float v[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        for (int r = 0; r < a.R; ++r)
#pragma unroll
            for (int q = 0; q < 5; ++q) v[q] += red[q * nthr + r * cols + tid];
        const int node = (tid * Lk.h_out + y) * Lk.w_out + x;
        const float centre = v[3] + (v[0] + Lk.bias_node[node]);
        const int64_t at = (int64_t)b * Lk.n_out + node;
        a.out_lb[at] = fmaxf(centre - a.eps * v[4] + v[1], a.out_lb[at]);
        a.out_ub[at] = fminf(centre + a.eps * v[4] - v[2], a.out_ub[at]);
    }
}

// bounds of conv layer k through the cone kernel; false when the layer does not qualify (a linear layer in front of it, too
// deep, too many channels, windows too large for shared memory): the caller takes the dense path
bool kw_cone_layer(const std::vector<LayerDev>& layers, const std::vector<int>& n, int k, int ND, const float* x, float eps,
                   float* const* out_lb, float* const* out_ub, const int32_t* dom_list, const int32_t* keep_upto, cudaStream_t st,
                   int64_t* launches) {
    if (k < 2 || k > CONE_MAX_DEPTH) return false;
    for (int j = 1; j <= k; ++j) if (layers[j - 1].kind != GNNB_LAYER_CONV) return false;
    const LayerDev& Lk = layers[k - 1];
    const int cols = Lk.c_out;
    if (cols > 256) return false;
    const int R = 256 / cols < 1 ? 1 : 256 / cols;
    // largest (unclipped) window per layer
    int h = 1, w = 1;
    size_t max_elems = 0;
    for (int j = k; j >= 1; --j) {
        const LayerDev& L = layers[j - 1];
        h = (h - 1) * L.stride + L.ksize; w = (w - 1) * L.stride + L.ksize;
        h = h < L.h_in ? h : L.h_in; w = w < L.w_in ? w : L.w_in;
        const size_t e = (size_t)L.c_in * h * w;
        max_elems = e > max_elems ? e : max_elems;
    }
    size_t buf = max_elems * cols;
    if (buf < (size_t)5 * cols * R) buf = (size_t)5 * cols * R;
    const size_t smem = 2 * buf * sizeof(float);
    if (smem > CONE_MAX_SMEM) return false;
    ConeArgs a{};
    for (int j = 1; j <= k; ++j) a.layer[j - 1] = layers[j - 1];
    for (int j = 1; j < k; ++j) { a.zl[j - 1] = out_lb[j]; a.zu[j - 1] = out_ub[j]; }
    a.k = k; a.cols = cols; a.R = R; a.buf_elems = (int)buf; a.x = x; a.eps = eps;
    a.out_lb = out_lb[k]; a.out_ub = out_ub[k]; a.dom_list = dom_list; a.keep_upto = keep_upto;
    for (int d0 = 0; d0 < ND; d0 += 65535) {
        const int nd = ND - d0 < 65535 ? ND - d0 : 65535;
        ConeArgs b = a;
        // domains beyond the first 65 535: shift the per-domain views (dom_list is indexed by the local domain; without it the
        // arrays themselves are)
        if (d0) {
            if (dom_list) b.dom_list = dom_list + d0;
            else {
                b.x = x + (size_t)d0 * n[0];
                for (int j = 1; j < k; ++j) { b.zl[j - 1] = out_lb[j] + (size_t)d0 * n[j]; b.zu[j - 1] = out_ub[j] + (size_t)d0 * n[j]; }
                b.out_lb = out_lb[k] + (size_t)d0 * n[k]; b.out_ub = out_ub[k] + (size_t)d0 * n[k];
                if (keep_upto) b.keep_upto = keep_upto + d0;
            }
        }
        k_kw_cone<<<dim3((unsigned)(Lk.h_out * Lk.w_out), (unsigned)nd), cols * R, smem, st>>>(b);
        ++*launches;
    }
    return true;
}

}  // namespace

// The shared-memory opt-in is a property of the device's context, so every context sets it (gnnb_create), not once per process
int kw_init() {
    return cudaFuncSetAttribute(k_kw_cone, cudaFuncAttributeMaxDynamicSharedMemorySize, CONE_MAX_SMEM);
}

// One KW pass.  Every pointer is a device pointer.  x [B, n0]; wp [B, n_L]; bp [B]; prov_lb / prov_ub: L + 1 arrays [B, n_k]
// (k = 1..L+1, the last one — the property output — may be null) or null; out_lb / out_ub: L + 2 arrays [B, n_k] (k = 0..L+1),
// may alias the provided arrays.  first_layer: first layer (1-based) whose bounds are computed (layers in front of it must
// already be in out_*; 1 also writes the input box).  dom_list / n_dom: the pass runs on these domains only (rows of the same
// arrays), null = all B.  keep_upto [B] or null: layers <= keep_upto[b] of domain b are left as they are.
// *ws / *ws_cap (floats): caller-kept scratch, grown when too small.
int kw_pass(const std::vector<LayerDev>& layers, const std::vector<int>& n, int B, const float* x, float eps, const float* wp, const float* bp,
            const float* const* prov_lb, const float* const* prov_ub, float* const* out_lb, float* const* out_ub, int first_layer,
            const int32_t* dom_list, int n_dom, const int32_t* keep_upto, const KwTc* tc, float** ws, size_t* ws_cap, cudaStream_t st,
            int64_t* launches, std::string* err) {
    const int L = (int)layers.size();
    const int ND = dom_list ? n_dom : B;          // domains of this pass
    static const bool use_cone = !(getenv("GNNB_KW_DENSE") && atoi(getenv("GNNB_KW_DENSE")) != 0);      // debugging: dense recursion everywhere
    if (ND < 1) return GNNB_OK;
    static const bool use_tc = !(getenv("GNNB_KW_SIMT") && atoi(getenv("GNNB_KW_SIMT")) != 0);        // debugging: exact-fp32 propagation everywhere
    if (!use_tc) tc = nullptr;
    int nmax = 0;
    for (int k = 0; k <= L; ++k) {
        const int rows = tc ? (*tc->maps)[k].nslots : n[k];          // the tile images are padded to whole tiles
        nmax = rows > nmax ? rows : nmax;
    }
    int64_t max_pairs = 0;
    for (int k = 1; k <= L; ++k) {
        const int64_t pairs = (int64_t)ND * ((n[k] + KW_COLS - 1) / KW_COLS);
        max_pairs = pairs > max_pairs ? pairs : max_pairs;
    }
    const int64_t PMAX = max_pairs < 1024 ? (max_pairs < 1 ? 1 : max_pairs) : 1024;      // pairs per pass: two [PMAX, nmax, 64] buffers
    const size_t buf_elems = (size_t)PMAX * nmax * KW_COLS, acc_elems = (size_t)PMAX * KW_COLS;
    const size_t need = 2 * buf_elems + 5 * acc_elems + 64;
    if (*ws_cap < need) {
        if (*ws) { cudaStreamSynchronize(st); cudaFree(*ws); }
        *ws = nullptr; *ws_cap = 0;
        const cudaError_t e = cudaMalloc(ws, need * sizeof(float));
        if (e != cudaSuccess) { *err = std::string("KW bounds workspace: ") + cudaGetErrorString(e); return GNNB_ERR_CUDA; }
        *ws_cap = need;
    }
    float* buf[2] = {*ws, *ws + buf_elems};
    float* accp = *ws + 2 * buf_elems;
    KwAcc acc{accp, accp + acc_elems, accp + 2 * acc_elems, accp + 3 * acc_elems, accp + 4 * acc_elems};

    if (first_layer <= 1) {
        k_kw_input_box<<<blocks_of((int64_t)B * n[0], 256), 256, 0, st>>>(x, eps, (int64_t)B * n[0], out_lb[0], out_ub[0]);
        ++*launches;
    }
    for (int k = first_layer < 1 ? 1 : first_layer; k <= L + 1; ++k) {
        const bool out_layer = k == L + 1;
        const int ncols = out_layer ? 1 : n[k];
        const int G = (ncols + KW_COLS - 1) / KW_COLS;
        const int64_t pairs = (int64_t)ND * G;
        // conv layers behind conv layers: the windowed recursion.  It intersects with the bounds already in out_*, so it needs them
        // there: true for every caller that provides bounds (they alias out_*); without provided bounds the dense path runs.
        if (use_cone && !out_layer && prov_lb && prov_ub && prov_lb[k - 1] == out_lb[k] && prov_ub[k - 1] == out_ub[k] &&
            kw_cone_layer(layers, n, k, ND, x, eps, out_lb, out_ub, dom_list, keep_upto, st, launches))
            continue;
        for (int64_t p0 = 0; p0 < pairs; p0 += PMAX) {
            const int64_t np = (pairs - p0) < PMAX ? (pairs - p0) : PMAX;
            cudaMemsetAsync(accp, 0, 5 * acc_elems * sizeof(float), st);
            int cur = 0;
            int j = k - 1;                          // layer whose post-activation space buf[cur] is about to hold (t_j)
            if (tc) {
                // tensor-core form: buf[0] holds mu images (s), buf[1] nb images (t)
                uint16_t* s_img = reinterpret_cast<uint16_t*>(buf[0]);
                uint16_t* t_img = reinterpret_cast<uint16_t*>(buf[1]);
                const std::vector<RowMap>& M = *tc->maps;
                if (!out_layer) {
                    const int64_t total = np * M[k].nslots * 8;
                    k_kw_img_onehot<<<blocks_of(total, 256), 256, 0, st>>>(s_img, M[k], G, p0, total);                  // s_k
                    ++*launches;
                    prop_tc_run((*tc->plans)[k - 1], buf[0], buf[1], (int)np, st, launches);                            // t_{k-1} = A_k^T s_k
                } else {
                    const int64_t total = np * M[L].nslots * 8;
                    k_kw_img_wp<<<blocks_of(total, 256), 256, 0, st>>>(t_img, wp, M[L], p0, total, dom_list);           // t_L (G = 1: pair = domain)
                    ++*launches;
                }
                for (; j >= 1; --j) {
                    k_kw_img_reduce<<<(unsigned)np, 256, 0, st>>>(t_img, s_img, M[j], out_lb[j], out_ub[j], layers[j - 1].bias_node, nullptr, G, p0, acc,
                                                                  dom_list, 0);                                       // s_j = d_j t_j
                    ++*launches;
                    prop_tc_run((*tc->plans)[j - 1], buf[0], buf[1], (int)np, st, launches);                            // t_{j-1} = A_j^T s_j
                }
                k_kw_img_reduce<<<(unsigned)np, 256, 0, st>>>(t_img, s_img, M[0], nullptr, nullptr, nullptr, x, G, p0, acc, dom_list, 1);
                ++*launches;
            } else {
            if (!out_layer) {
                const int64_t total4 = np * n[k] * 16;
                k_kw_onehot<<<blocks_of(total4, 256), 256, 0, st>>>(buf[cur], n[k], G, p0, total4);        // s_k
                ++*launches;
            } else {
                const int64_t total4 = np * n[L] * 16;
                k_kw_wp_col<<<blocks_of(total4, 256), 256, 0, st>>>(buf[cur], wp, n[L], p0, total4, dom_list);   // t_L (G = 1: pair = domain)
                ++*launches;
            }
            // walk down: buf[cur] holds s_{j+1} (or, for the output layer's first step, already t_L)
            bool have_t = out_layer;
            for (; j >= 1; --j) {
                if (!have_t) {
                    prop_backward(layers[j], buf[cur], buf[cur ^ 1], (int)np, false, st, launches);          // t_j = A_{j+1}^T s_{j+1}
                    cur ^= 1;
                }
                have_t = false;
                k_kw_reduce_layer<<<(unsigned)np, 256, 0, st>>>(buf[cur], out_lb[j], out_ub[j], layers[j - 1].bias_node, n[j], G, p0, acc, dom_list);
                ++*launches;
            }
            prop_backward(layers[0], buf[cur], buf[cur ^ 1], (int)np, false, st, launches);                  // t_0 = A_1^T s_1
            cur ^= 1;
            k_kw_reduce_input<<<(unsigned)np, 256, 0, st>>>(buf[cur], x, n[0], G, p0, acc, dom_list);
            ++*launches;
            }
            k_kw_finish<<<blocks_of(np * KW_COLS, 256), 256, 0, st>>>(acc, ncols, G, p0, np, eps, out_layer ? nullptr : layers[k - 1].bias_node, bp,
                                                                      prov_lb ? prov_lb[k - 1] : nullptr, prov_ub ? prov_ub[k - 1] : nullptr,
                                                                      out_lb[k], out_ub[k], dom_list, keep_upto, k);
            ++*launches;
        }
    }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { *err = std::string("KW bounds: ") + cudaGetErrorString(e); return GNNB_ERR_CUDA; }
    return GNNB_OK;
}

// init_kw_bounds for B domains: all layers, optional provided bounds of the hidden layers (L arrays)
int kw_bounds(const std::vector<LayerDev>& layers, const std::vector<int>& n, int B, const float* x, float eps, const float* wp, const float* bp,
              const float* const* prov_lb, const float* const* prov_ub, float* const* out_lb, float* const* out_ub, const KwTc* tc, float** ws,
              size_t* ws_cap, cudaStream_t st, int64_t* launches, std::string* err) {
    const int L = (int)layers.size();
    if (L > KW_MAX_LAYERS) { *err = "KW bounds: too many layers"; return GNNB_ERR_UNSUPPORTED; }
    const float* pl[KW_MAX_LAYERS + 1];
    const float* pu[KW_MAX_LAYERS + 1];
    for (int k = 0; k <= L; ++k) { pl[k] = (prov_lb && k < L) ? prov_lb[k] : nullptr; pu[k] = (prov_ub && k < L) ? prov_ub[k] : nullptr; }
    return kw_pass(layers, n, B, x, eps, wp, bp, prov_lb ? pl : nullptr, prov_ub ? pu : nullptr, out_lb, out_ub, 1, nullptr, 0, nullptr, tc, ws, ws_cap,
                   st, launches, err);
}

// Bounds part of update_the_model (plnn/conv_kwinter_gen.py:558-660) for B children at once.  parent_lb / parent_ub, out_lb /
// out_ub: L + 2 arrays [B, n_k] (k = 0..L+1); dec_layer (0-based hidden layer) / dec_index / choice: [B]; out_mask: L arrays
// [B, n_k] int8 or null; second_pass: [B] int32 or null (1 where the interval bounds tightened a hidden layer and the KW pass
// was repeated).  iscratch: 3 B + 1 int32 of caller-kept device scratch.  Synchronises `st` once (the number of domains that
// need the second pass).
int child_bounds(const std::vector<LayerDev>& layers, const std::vector<int>& n, int B, const float* x, float eps, const float* wp, const float* bp,
                 const float* const* parent_lb, const float* const* parent_ub, const int32_t* dec_layer, const int32_t* dec_index,
                 const int32_t* choice, float* const* out_lb, float* const* out_ub, int8_t* const* out_mask, int32_t* second_pass,
                 int32_t* iscratch, const KwTc* tc, float** ws, size_t* ws_cap, cudaStream_t st, int64_t* launches, std::string* err) {
    const int L = (int)layers.size();
    if (L > KW_MAX_LAYERS) { *err = "child bounds: too many layers"; return GNNB_ERR_UNSUPPORTED; }
    int32_t* keep = iscratch;
    int32_t* changed = iscratch + B;
    int32_t* list = iscratch + 2 * (size_t)B;
    int32_t* count = iscratch + 3 * (size_t)B;
    BoundPtrs o;
    for (int k = 0; k <= L + 1; ++k) {
        o.lb[k] = out_lb[k]; o.ub[k] = out_ub[k]; o.n[k] = n[k];
        if (out_lb[k] != parent_lb[k]) cudaMemcpyAsync(out_lb[k], parent_lb[k], (size_t)B * n[k] * sizeof(float), cudaMemcpyDeviceToDevice, st);
        if (out_ub[k] != parent_ub[k]) cudaMemcpyAsync(out_ub[k], parent_ub[k], (size_t)B * n[k] * sizeof(float), cudaMemcpyDeviceToDevice, st);
    }
    k_child_split<<<blocks_of(B, 256), 256, 0, st>>>(o, L, B, dec_layer, dec_index, choice, keep, changed);
    ++*launches;
    // first KW pass: the children's own (parent + split) bounds are the provided ones; layer 1 depends on no ReLU and never moves
    const float* pl[KW_MAX_LAYERS + 1];
    const float* pu[KW_MAX_LAYERS + 1];
    for (int k = 1; k <= L + 1; ++k) { pl[k - 1] = out_lb[k]; pu[k - 1] = out_ub[k]; }
    int rc = kw_pass(layers, n, B, x, eps, wp, bp, pl, pu, out_lb, out_ub, 2, nullptr, 0, keep, tc, ws, ws_cap, st, launches, err);
    if (rc != GNNB_OK) return rc;
    // interval pass, layer by layer behind the split
    for (int k = 2; k <= L + 1; ++k) {
        if (k <= L) {
            const LayerDev& Ld = layers[k - 1];
            if (Ld.kind == GNNB_LAYER_CONV)
                k_interval_conv<<<blocks_of((int64_t)B * n[k], 256), 256, 0, st>>>(Ld, out_lb[k - 1], out_ub[k - 1], out_lb[k], out_ub[k], B, k, keep, changed, 0);
            else
                k_interval_linear<<<blocks_of((int64_t)B * n[k] * 32, 256), 256, 0, st>>>(Ld.weight, Ld.bias_node, 0, n[k - 1], n[k], out_lb[k - 1], out_ub[k - 1],
                                                                                           out_lb[k], out_ub[k], B, k, true, keep, changed, 0);
        } else {
            k_interval_linear<<<blocks_of((int64_t)B * 32, 256), 256, 0, st>>>(wp, bp, n[L], n[L], 1, out_lb[L], out_ub[L], out_lb[k], out_ub[k], B, k, false,
                                                                                keep, changed, 0);
        }
        ++*launches;
    }
    k_collect_changed<<<1, 1024, 0, st>>>(changed, B, list, count);
    ++*launches;
    int32_t h_count = 0;
    cudaMemcpyAsync(&h_count, count, sizeof h_count, cudaMemcpyDeviceToHost, st);
    if (cudaStreamSynchronize(st) != cudaSuccess) { *err = std::string("child bounds: ") + cudaGetErrorString(cudaGetLastError()); return GNNB_ERR_CUDA; }
    if (h_count > 0) {
        rc = kw_pass(layers, n, B, x, eps, wp, bp, pl, pu, out_lb, out_ub, 2, list, h_count, keep, tc, ws, ws_cap, st, launches, err);
        if (rc != GNNB_OK) return rc;
    }
    if (second_pass) cudaMemcpyAsync(second_pass, changed, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToDevice, st);
    if (out_mask)
        for (int k = 1; k <= L; ++k) {
            const int64_t total = (int64_t)B * n[k];
            k_mask_from_bounds<<<blocks_of(total, 256), 256, 0, st>>>(out_lb[k], out_ub[k], out_mask[k - 1], total);
            ++*launches;
        }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { *err = std::string("child bounds: ") + cudaGetErrorString(e); return GNNB_ERR_CUDA; }
    return GNNB_OK;
}

// Bounds part of build_the_model (plnn/conv_kwinter_gen.py:199-270) for B root domains: KW bounds (init_kw_bounds), intersected
// layer by layer with interval bounds (the first layer from the input box itself); where a hidden layer moved by more than
// 1e-4, one KW pass from the first such layer with the intersected bounds provided.  Same arrays and scratch as child_bounds.
int root_bounds(const std::vector<LayerDev>& layers, const std::vector<int>& n, int B, const float* x, float eps, const float* wp, const float* bp,
                float* const* out_lb, float* const* out_ub, int8_t* const* out_mask, int32_t* second_pass, int32_t* iscratch, const KwTc* tc,
                float** ws, size_t* ws_cap, cudaStream_t st, int64_t* launches, std::string* err) {
    const int L = (int)layers.size();
    if (L > KW_MAX_LAYERS) { *err = "root bounds: too many layers"; return GNNB_ERR_UNSUPPORTED; }
    int32_t* keep = iscratch;
    int32_t* changed = iscratch + B;
    int32_t* list = iscratch + 2 * (size_t)B;
    int32_t* count = iscratch + 3 * (size_t)B;
    int rc = kw_bounds(layers, n, B, x, eps, wp, bp, nullptr, nullptr, out_lb, out_ub, tc, ws, ws_cap, st, launches, err);
    if (rc != GNNB_OK) return rc;
    cudaMemsetAsync(keep, 0, (size_t)B * sizeof(int32_t), st);                 // every layer takes part in the interval pass
    cudaMemsetAsync(changed, 0x7f, (size_t)B * sizeof(int32_t), st);           // "no layer moved"
    for (int k = 1; k <= L + 1; ++k) {
        if (k <= L) {
            const LayerDev& Ld = layers[k - 1];
            if (Ld.kind == GNNB_LAYER_CONV)
                k_interval_conv<<<blocks_of((int64_t)B * n[k], 256), 256, 0, st>>>(Ld, out_lb[k - 1], out_ub[k - 1], out_lb[k], out_ub[k], B, k, keep, changed, 1);
            else
                k_interval_linear<<<blocks_of((int64_t)B * n[k] * 32, 256), 256, 0, st>>>(Ld.weight, Ld.bias_node, 0, n[k - 1], n[k], out_lb[k - 1], out_ub[k - 1],
                                                                                           out_lb[k], out_ub[k], B, k, true, keep, changed, 1);
        } else {
            k_interval_linear<<<blocks_of((int64_t)B * 32, 256), 256, 0, st>>>(wp, bp, n[L], n[L], 1, out_lb[L], out_ub[L], out_lb[k], out_ub[k], B, k, false,
                                                                                keep, changed, 1);
        }
        ++*launches;
    }
    k_root_prepare<<<blocks_of(B, 256), 256, 0, st>>>(changed, keep, B, L);
    k_collect_changed<<<1, 1024, 0, st>>>(changed, B, list, count);
    *launches += 2;
    int32_t h_count = 0;
    cudaMemcpyAsync(&h_count, count, sizeof h_count, cudaMemcpyDeviceToHost, st);
    if (cudaStreamSynchronize(st) != cudaSuccess) { *err = std::string("root bounds: ") + cudaGetErrorString(cudaGetLastError()); return GNNB_ERR_CUDA; }
    if (h_count > 0) {
        const float* pl[KW_MAX_LAYERS + 1];
        const float* pu[KW_MAX_LAYERS + 1];
        for (int k = 1; k <= L + 1; ++k) { pl[k - 1] = out_lb[k]; pu[k - 1] = out_ub[k]; }
        rc = kw_pass(layers, n, B, x, eps, wp, bp, pl, pu, out_lb, out_ub, 2, list, h_count, keep, tc, ws, ws_cap, st, launches, err);
        if (rc != GNNB_OK) return rc;
    }
    if (second_pass) cudaMemcpyAsync(second_pass, changed, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToDevice, st);
    if (out_mask)
        for (int k = 1; k <= L; ++k) {
            const int64_t total = (int64_t)B * n[k];
            k_mask_from_bounds<<<blocks_of(total, 256), 256, 0, st>>>(out_lb[k], out_ub[k], out_mask[k - 1], total);
            ++*launches;
        }
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { *err = std::string("root bounds: ") + cudaGetErrorString(e); return GNNB_ERR_CUDA; }
    return GNNB_OK;
}

}  // namespace gnnb
