// Gradients of selected branching scores with respect to the 52 GNN tensors, and the Adam step — the device side of the
// online fine-tuning variant (reference: graphnet/graph_score_online.py:62-77, `loss = gnn_score - kw_score + improvement;
// loss.backward(); optimizer.step()`, called from plnn/relu_conv_online.py:198-211 on one subdomain at a time).
//
// The reference gets its gradients from PyTorch autograd over GraphNet.forward (graph_conv.py:77-388).  Here the same
// derivative is written out by hand: an exact-fp32 forward pass that keeps every activation a weight gradient needs (the
// "tape": inputs and ReLU outputs of each nn.Linear, per round and sweep), then the reverse sweep.  Rows are in node order
// (global row = b * n_k + node, 64 channels = 256 bytes per row), like the SIMT validation path.
//
// Building blocks:
//   k_lin_fwd   Y = rs_out * act(sum_seg (rs_seg * X_seg) W[:, seg]^T + b)       one nn.Linear with a concatenated input
//               (up to three 64-wide segments, each with an optional per-row scale: r0 / r1, -d2 / d1) or a K < 64 feature input
//   k_lin_bwd   its adjoint: dZ = dY * rs_out * [Y > 0];  dW[:, seg] += dZ^T (rs_seg X_seg);  db += colsum(dZ);
//               dX_seg (+)= rs_seg * dZ W[:, seg]
//   propagation adjoints reuse the forward kernels of gnnb_prop.cu: (A_k)^T is prop_backward without normalisation,
//               (A_k^T / freq)^T = A_k (. / freq) is k_div_freq + prop_forward, the rank-1 property edges are k_wp_reduce /
//               prop_property_backward
//   k_score_terms   score head on the few rows the loss names (forward + backward in one small kernel)
//   k_adam      torch.optim.Adam (L2 weight decay folded into the gradient, bias-corrected), one thread per parameter
//
// Dead work: the last round's input-layer update has no consumer (SURVEY §8a fact 2), so it gets no gradient; the
// round-independent relaxation features are evaluated once and receive the sum of the rounds' gradients.
#include <math.h>

#include <string>
#include <vector>

#include "gnnb_common.cuh"
#include "gnnb_train.cuh"

namespace gnnb {
namespace {

constexpr int TM = 64;        // rows per tile
constexpr int TMP = 68;       // padded leading dimension of transposed tiles
constexpr int NTH = 256;

struct LinSeg {
    const float* x;           // [rows][K]
    const float* rs;          // [rows] per-row scale of this segment, or null
    int K;                    // 64, or < 64 for the single-segment feature layers
};

struct LinFwdArgs {
    LinSeg seg[3];
    int nseg;
    const float* wt;          // [Ktot][64] transposed weight (GnnParams::wt)
    const float* bias;        // [64]
    int relu;
    const float* out_rs;      // [rows] or null
    float* y;                 // [rows][64]
    int64_t rows;
};

__device__ __forceinline__ float relu_keep_nan(float x) { return (x != x) ? x : fmaxf(x, 0.f); }

__global__ void __launch_bounds__(NTH) k_lin_fwd(LinFwdArgs a) {
    __shared__ __align__(16) float actT[64 * TMP];
    __shared__ __align__(16) float wbuf[64 * 64];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t ntiles = (a.rows + TM - 1) / TM;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t row0 = tile * TM;
        float acc[4][4];
        {
            const float4 b4 = *reinterpret_cast<const float4*>(a.bias + tx * 4);
#pragma unroll
            for (int i = 0; i < 4; ++i) { acc[i][0] = b4.x; acc[i][1] = b4.y; acc[i][2] = b4.z; acc[i][3] = b4.w; }
        }
        int koff = 0;
        for (int s = 0; s < a.nseg; ++s) {
            const LinSeg sg = a.seg[s];
            __syncthreads();
            for (int idx = threadIdx.x; idx < TM * sg.K; idx += NTH) {
                const int r = idx / sg.K, k = idx - r * sg.K;
                float v = 0.f;
                if (row0 + r < a.rows) {
                    v = sg.x[(row0 + r) * sg.K + k];
                    if (sg.rs) v *= sg.rs[row0 + r];
                }
                actT[k * TMP + r] = v;
            }
            for (int idx = threadIdx.x; idx < sg.K * 16; idx += NTH)
                reinterpret_cast<float4*>(wbuf)[idx] = reinterpret_cast<const float4*>(a.wt + (size_t)koff * 64)[idx];
            __syncthreads();
            for (int k = 0; k < sg.K; ++k) {
                const float4 x4 = *reinterpret_cast<const float4*>(actT + k * TMP + ty * 4);
                const float4 w4 = *reinterpret_cast<const float4*>(wbuf + k * 64 + tx * 4);
                const float xv[4] = {x4.x, x4.y, x4.z, x4.w};
                const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(xv[i], wv[j], acc[i][j]);
            }
            koff += sg.K;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int64_t row = row0 + ty * 4 + i;
            if (row >= a.rows) continue;
            const float s = a.out_rs ? a.out_rs[row] : 1.0f;
            float4 v;
            v.x = a.relu ? relu_keep_nan(acc[i][0]) : acc[i][0];
            v.y = a.relu ? relu_keep_nan(acc[i][1]) : acc[i][1];
            v.z = a.relu ? relu_keep_nan(acc[i][2]) : acc[i][2];
            v.w = a.relu ? relu_keep_nan(acc[i][3]) : acc[i][3];
            if (a.out_rs) { v.x *= s; v.y *= s; v.z *= s; v.w *= s; }
            *reinterpret_cast<float4*>(a.y + row * P + tx * 4) = v;
        }
    }
}

struct LinBwdArgs {
    LinSeg seg[3];
    float* dx[3];             // [rows][64] gradient of each segment's input, or null (feature inputs)
    int dx_acc[3];            // 1: add to dx, 0: overwrite
    int nseg;
    const float* w;           // [64][Ktot] nn.Linear layout
    int Ktot;
    const float* dy;          // [rows][64]
    const float* y_relu;      // [rows][64] the layer's ReLU output (mask = y > 0), or null when the layer has no ReLU
    const float* out_rs;      // [rows] or null
    float* dW;                // [64][Ktot]
    float* db;                // [64]
    int64_t rows;
};

struct BwdSmem {
    float dz[TM * 64];        // [r][n]
    float dzT[64 * TMP];      // [n][r]
    float xs[TM * 64];        // [r][k]  scaled input of the current segment, zero-padded to 64 columns
    float wb[64 * 64];        // [n][k]  weight slice of the current segment
};

__global__ void __launch_bounds__(NTH) k_lin_bwd(LinBwdArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    BwdSmem& s = *reinterpret_cast<BwdSmem*>(smem_raw);
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int64_t ntiles = (a.rows + TM - 1) / TM;
    float gw[3][4][4];        // this block's share of dW[ty*4 + i][koff + tx*4 + j]
    float gb[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int sg = 0; sg < 3; ++sg)
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) gw[sg][i][j] = 0.f;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int64_t row0 = tile * TM;
        __syncthreads();
        for (int idx = threadIdx.x; idx < TM * 16; idx += NTH) {
            const int r = idx >> 4, c4 = idx & 15;
            const int64_t row = row0 + r;
            float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
            if (row < a.rows) {
                g = *reinterpret_cast<const float4*>(a.dy + row * P + c4 * 4);
                if (a.out_rs) { const float q = a.out_rs[row]; g.x *= q; g.y *= q; g.z *= q; g.w *= q; }
                if (a.y_relu) {
                    const float4 y = *reinterpret_cast<const float4*>(a.y_relu + row * P + c4 * 4);
                    g.x = y.x > 0.f ? g.x : 0.f; g.y = y.y > 0.f ? g.y : 0.f;
                    g.z = y.z > 0.f ? g.z : 0.f; g.w = y.w > 0.f ? g.w : 0.f;
                }
            }
            *reinterpret_cast<float4*>(s.dz + r * 64 + c4 * 4) = g;
            s.dzT[(c4 * 4 + 0) * TMP + r] = g.x; s.dzT[(c4 * 4 + 1) * TMP + r] = g.y;
            s.dzT[(c4 * 4 + 2) * TMP + r] = g.z; s.dzT[(c4 * 4 + 3) * TMP + r] = g.w;
        }
        __syncthreads();
        if (tx == 0) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                float sum = 0.f;
                for (int r = 0; r < TM; ++r) sum += s.dz[r * 64 + ty * 4 + i];
                gb[i] += sum;
            }
        }
        int koff = 0;
#pragma unroll
        for (int sgi = 0; sgi < 3; ++sgi) {
            if (sgi >= a.nseg) break;
            const LinSeg sg = a.seg[sgi];
            __syncthreads();                       // previous users of xs / wb are done
            for (int idx = threadIdx.x; idx < TM * 64; idx += NTH) {
                const int r = idx >> 6, k = idx & 63;
                float v = 0.f;
                if (k < sg.K && row0 + r < a.rows) {
                    v = sg.x[(row0 + r) * sg.K + k];
                    if (sg.rs) v *= sg.rs[row0 + r];
                }
                s.xs[idx] = v;
            }
            if (a.dx[sgi] != nullptr)
                for (int idx = threadIdx.x; idx < 64 * 64; idx += NTH) {
                    const int n = idx >> 6, k = idx & 63;
                    s.wb[idx] = a.w[(size_t)n * a.Ktot + koff + k];
                }
            __syncthreads();
            // dW[n][koff + k] += sum_r dz[r][n] * xs[r][k]
            if (tx * 4 < sg.K) {
                for (int r = 0; r < TM; ++r) {
                    const float4 d4 = *reinterpret_cast<const float4*>(s.dz + r * 64 + ty * 4);
                    const float4 x4 = *reinterpret_cast<const float4*>(s.xs + r * 64 + tx * 4);
                    const float dv[4] = {d4.x, d4.y, d4.z, d4.w};
                    const float xv[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 4; ++j) gw[sgi][i][j] = fmaf(dv[i], xv[j], gw[sgi][i][j]);
                }
            }
            // dX[r][k] (+)= rs[r] * sum_n dz[r][n] * W[n][koff + k]
            if (a.dx[sgi] != nullptr) {
                float acc[4][4];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
                for (int n = 0; n < 64; ++n) {
                    const float4 d4 = *reinterpret_cast<const float4*>(s.dzT + n * TMP + ty * 4);
                    const float4 w4 = *reinterpret_cast<const float4*>(s.wb + n * 64 + tx * 4);
                    const float dv[4] = {d4.x, d4.y, d4.z, d4.w};
                    const float wv[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i)
#pragma unroll
                        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(dv[i], wv[j], acc[i][j]);
                }
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    const int64_t row = row0 + ty * 4 + i;
                    if (row >= a.rows) continue;
                    const float q = sg.rs ? sg.rs[row] : 1.0f;
                    float4* dst = reinterpret_cast<float4*>(a.dx[sgi] + row * P + tx * 4);
                    float4 v = make_float4(acc[i][0] * q, acc[i][1] * q, acc[i][2] * q, acc[i][3] * q);
                    if (a.dx_acc[sgi]) { const float4 o = *dst; v.x += o.x; v.y += o.y; v.z += o.z; v.w += o.w; }
                    *dst = v;
                }
            }
            koff += sg.K;
        }
    }
    // flush this block's partial sums
    int koff = 0;
#pragma unroll
    for (int sgi = 0; sgi < 3; ++sgi) {
        if (sgi >= a.nseg) break;
        const int K = a.seg[sgi].K;
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int k = tx * 4 + j;
                if (k < K && gw[sgi][i][j] != 0.f) atomicAdd(a.dW + (size_t)(ty * 4 + i) * a.Ktot + koff + k, gw[sgi][i][j]);
            }
        koff += K;
    }
    if (tx == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i)
            if (gb[i] != 0.f) atomicAdd(a.db + ty * 4 + i, gb[i]);
    }
}

// per-row scalars and feature vectors of a hidden layer (graph_conv.py:141-159, 253-279, 499-514)
// rs: [6][rows] = r0, r1, amb, gate (r0 != 0), d1, -d2;  featf / featb: [rows][7]
__global__ void k_row_scalars(const float* __restrict__ lb, const float* __restrict__ ub, const float* __restrict__ dual,
                              const float* __restrict__ pre, const float* __restrict__ post, const float* __restrict__ bias_node,
                              int n, int64_t rows, float* __restrict__ rs, float* __restrict__ featf, float* __restrict__ featb) {
    const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= rows) return;
    const float l = lb[row], u = ub[row], d1 = dual[row * 3 + 1], d2 = dual[row * 3 + 2], pp = pre[row], po = post[row];
    const float bs = bias_node[row % n];
    const Ratio q = compute_ratio(l, u);
    rs[0 * rows + row] = q.r0; rs[1 * rows + row] = q.r1; rs[2 * rows + row] = q.amb;
    rs[3 * rows + row] = (q.r0 != 0.0f) ? 1.0f : 0.0f; rs[4 * rows + row] = d1; rs[5 * rows + row] = -d2;
    float* f = featf + row * 7;
    f[0] = q.beta; f[1] = l; f[2] = u; f[3] = d1 - d2; f[4] = pp; f[5] = po; f[6] = bs;
    float* g = featb + row * 7;
    g[0] = l; g[1] = u; g[2] = q.beta; g[3] = -d2 + d1; g[4] = po; g[5] = pp; g[6] = bs;
}

// out[i][0..K) = (c0[i], c1[i], c2[i], c3[i]) — the 2 / 3 / 4-wide feature rows of the input and output nodes
__global__ void k_stack(const float* c0, const float* c1, const float* c2, const float* c3, int K, int64_t rows, float* out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows) return;
    const float* c[4] = {c0, c1, c2, c3};
    for (int k = 0; k < K; ++k) out[i * K + k] = c[k][i];
}

// out[b][c] (+)= sum_n wp[b][n] * x[b][n][c]   (graph_conv.py:196 forward; adjoint of the rank-1 edges of :324-326)
__global__ void __launch_bounds__(64) k_wp_reduce(const float* __restrict__ wp, const float* __restrict__ x, int nL, int accumulate,
                                                  float* __restrict__ out) {
    const int b = blockIdx.x, c = threadIdx.x;
    float acc = 0.f;
    for (int n = 0; n < nL; ++n) acc = fmaf(wp[(int64_t)b * nL + n], x[((int64_t)b * nL + n) * P + c], acc);
    if (accumulate) out[(int64_t)b * P + c] += acc; else out[(int64_t)b * P + c] = acc;
}

// x[b][(ci, yi, xi)][:] / freq(yi, xi): the adjoint of the tap-count normalisation of graph_conv.py:306-312
__global__ void k_div_freq(LayerDev L, const float* __restrict__ x, float* __restrict__ out, int64_t total4) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total4) return;
    const int64_t row = i >> 4;
    const int node = (int)(row % L.n_in);
    const int yx = node % (L.h_in * L.w_in), yi = yx / L.w_in, xi = yx % L.w_in;
    int ty = 0, tx = 0;
    for (int k = 0; k < L.ksize; ++k) {
        const int a = yi + L.pad - k;
        if (a >= 0 && a % L.stride == 0 && a / L.stride < L.h_out) ++ty;
        const int b = xi + L.pad - k;
        if (b >= 0 && b % L.stride == 0 && b / L.stride < L.w_out) ++tx;
    }
    const float freq = (float)(ty * tx);
    float4 v = reinterpret_cast<const float4*>(x)[i];
    v.x = __fdiv_rn(v.x, freq); v.y = __fdiv_rn(v.y, freq); v.z = __fdiv_rn(v.z, freq); v.w = __fdiv_rn(v.w, freq);
    reinterpret_cast<float4*>(out)[i] = v;
}

__global__ void k_add(float* __restrict__ dst, const float* __restrict__ src, int64_t n4) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n4) return;
    float4 a = reinterpret_cast<float4*>(dst)[i];
    const float4 b = reinterpret_cast<const float4*>(src)[i];
    a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
    reinterpret_cast<float4*>(dst)[i] = a;
}

// One block of 64 threads per loss term: score = fscore(relu(fnode(mu_row))) (graph_conv.py:448-449) and its backward with
// upstream gradient coeff.  A term is this wave's when its domain is valid and sits at list position row0 .. row0 + rows - 1
// (row_of); other terms (inactive, out of range, another wave's) return at once, and their score stays as it is.  The row of
// the term's node after the last backward sweep is found from the per-layer table (flat index -> layer, node).
struct ScoreTermArgs {
    const int32_t *domain, *index;  // [n_terms] the caller's terms
    const float* coeff;             // [n_terms]
    const int32_t* row_of;          // [B] position of a named subdomain in the list of named subdomains
    int B, n_hidden, row0, rows;
    const TermLayer* layers;        // [L] hidden layers k = 1..L
    int L;
    const float *w_fnode, *b_fnode, *w_fscore, *b_fscore;      // nn.Linear layouts
    float *dW_fnode, *db_fnode, *dW_fscore, *db_fscore;
    float* scores;                  // [n_terms]
};
__global__ void __launch_bounds__(64) k_score_terms(ScoreTermArgs a) {
    __shared__ float x[P], dh[P];
    __shared__ float red[2];
    const int t = blockIdx.x, c = threadIdx.x;
    const int d = a.domain[t], flat = a.index[t];
    if (d < 0 || d >= a.B || flat < 0 || flat >= a.n_hidden) return;
    const int r = a.row_of[d] - a.row0;
    if (r < 0 || r >= a.rows) return;
    int k = 0;
    while (k + 1 < a.L && flat >= a.layers[k + 1].off) ++k;
    const TermLayer lay = a.layers[k];
    const int64_t row = ((int64_t)r * lay.n + (flat - lay.off)) * P;
    x[c] = lay.mu[row + c];
    __syncthreads();
    float z = a.b_fnode[c];
    for (int k2 = 0; k2 < P; ++k2) z = fmaf(x[k2], a.w_fnode[c * P + k2], z);
    const float h = relu_keep_nan(z);
    float part = h * a.w_fscore[c];
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
    if ((c & 31) == 0) red[c >> 5] = part;
    __syncthreads();
    const float g = a.coeff[t];
    if (c == 0) {
        a.scores[t] = red[0] + red[1] + a.b_fscore[0];
        atomicAdd(a.db_fscore, g);
    }
    atomicAdd(a.dW_fscore + c, g * h);
    const float dd = (z > 0.f) ? g * a.w_fscore[c] : 0.f;
    dh[c] = dd;
    atomicAdd(a.db_fnode + c, dd);
    for (int k2 = 0; k2 < P; ++k2) atomicAdd(a.dW_fnode + c * P + k2, dd * x[k2]);
    __syncthreads();
    float dm = 0.f;
    for (int n = 0; n < P; ++n) dm = fmaf(dh[n], a.w_fnode[n * P + c], dm);
    atomicAdd(lay.dmu + row + c, dm);
}

// Terms -> named subdomains.  k_name_terms: every term's score is NaN until its wave writes it; an active term (domain >= 0)
// flags its domain, or counts as bad when its domain or index is out of range.  k_list_named (one block): the flagged domains
// in ascending order -> list, their positions -> row_of, the count -> cnt[0].  cnt = [named, bad].
__global__ void k_name_terms(const int32_t* __restrict__ domain, const int32_t* __restrict__ index, int n_terms, int B, int n_hidden,
                             float* __restrict__ scores, int32_t* __restrict__ cnt, int32_t* __restrict__ flag) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_terms) return;
    scores[t] = __int_as_float(0x7fc00000);
    const int d = domain[t], i = index[t];
    if (d < 0) return;
    if (d >= B || i < 0 || i >= n_hidden) { atomicAdd(cnt + 1, 1); return; }
    flag[d] = 1;
}

constexpr int LIST_TH = 1024;
__global__ void __launch_bounds__(LIST_TH) k_list_named(const int32_t* __restrict__ flag, int B, int32_t* __restrict__ list,
                                                        int32_t* __restrict__ row_of, int32_t* __restrict__ cnt) {
    __shared__ int warp_sum[LIST_TH / 32];
    __shared__ int base;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (int j0 = 0; j0 < B; j0 += LIST_TH) {
        const int j = j0 + threadIdx.x;
        const int v = (j < B && flag[j]) ? 1 : 0;
        const unsigned bal = __ballot_sync(0xffffffffu, v);
        if (lane == 0) warp_sum[wid] = __popc(bal);
        __syncthreads();
        int before = base + __popc(bal & ((1u << lane) - 1u));
        for (int w = 0; w < wid; ++w) before += warp_sum[w];
        if (v) { list[before] = j; row_of[j] = before; }
        __syncthreads();
        if (threadIdx.x == 0) {
            int s = 0;
            for (int w = 0; w < LIST_TH / 32; ++w) s += warp_sum[w];
            base += s;
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) cnt[0] = base;
}

// torch.optim.Adam (amsgrad = False, maximize = False): weight decay is added to the gradient, moments are bias-corrected
__global__ void k_adam(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, int64_t n,
                       float lr, float b1, float b2, float eps, float wd, float bc1, float bc2_sqrt) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float gi = g[i];
    if (wd != 0.f) gi = fmaf(wd, p[i], gi);
    const float mi = m[i] + (gi - m[i]) * (1.0f - b1);             // exp_avg.lerp_(grad, 1 - beta1)
    const float vi = fmaf(1.0f - b2, gi * gi, v[i] * b2);          // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
    m[i] = mi; v[i] = vi;
    const float denom = __fdiv_rn(sqrtf(vi), bc2_sqrt) + eps;
    p[i] = p[i] - (lr / bc1) * __fdiv_rn(mi, denom);
}

int blocks_for(int64_t n, int per) { return (int)((n + per - 1) / per < 1 ? 1 : (n + per - 1) / per); }
int tile_grid(int64_t rows) {
    const int64_t t = (rows + TM - 1) / TM;
    return (int)(t < 1 ? 1 : (t < 148 * 4 ? t : 148 * 4));
}

struct Ctx {      // launch helpers bound to one call
    const GnnParams& g;
    const TrainParams& tp;
    cudaStream_t st;
    int64_t* launches;

    void fwd(int l, std::initializer_list<LinSeg> segs, bool relu, const float* out_rs, float* y, int64_t rows) const {
        LinFwdArgs a{};
        int i = 0;
        for (const LinSeg& s : segs) a.seg[i++] = s;
        a.nseg = i; a.wt = g.wt[l]; a.bias = g.bias[l]; a.relu = relu ? 1 : 0; a.out_rs = out_rs; a.y = y; a.rows = rows;
        k_lin_fwd<<<tile_grid(rows), NTH, 0, st>>>(a);
        ++*launches;
    }
    struct BSeg { LinSeg s; float* dx; bool acc; };
    void bwd(int l, std::initializer_list<BSeg> segs, const float* dy, const float* y_relu, const float* out_rs, int64_t rows) const {
        LinBwdArgs a{};
        int i = 0;
        for (const BSeg& s : segs) { a.seg[i] = s.s; a.dx[i] = s.dx; a.dx_acc[i] = s.acc ? 1 : 0; ++i; }
        a.nseg = i; a.w = tp.w[l]; a.Ktot = lin_in(l); a.dy = dy; a.y_relu = y_relu; a.out_rs = out_rs;
        a.dW = tp.dw[l]; a.db = tp.db[l]; a.rows = rows;
        k_lin_bwd<<<tile_grid(rows), NTH, sizeof(BwdSmem), st>>>(a);
        ++*launches;
    }
    void add(float* dst, const float* src, int64_t numel) const {
        k_add<<<blocks_for(numel / 4, 256), 256, 0, st>>>(dst, src, numel / 4);
        ++*launches;
    }
    void zero(float* p, int64_t numel) const { cudaMemsetAsync(p, 0, (size_t)numel * sizeof(float), st); }
};

// Offsets (floats) of a wave's activation tape and gradient temporaries in the arena, laid out for waves of up to Bcap
// subdomains; a smaller wave uses the first rows of each array.
struct Tape {
    struct Layer { size_t rs, featf, featb, h1, rlxf, g1, g2, s1, g3, rlxb, drlxf, drlxb; std::vector<size_t> nbF, h3F, eF, h4F, nbB, h3B, eB, h4B; };
    std::vector<Layer> lt;
    size_t o_f3, o_f2, o_f4, o_e1, o_i1, o_i2, o_dout, o_dsm, o_bufA, o_bufB, o_bufC, o_bufD, o_tab;
    std::vector<size_t> o_nb0, o_i3, o_o1, o_nbo, o_o2, o_mu, o_dF, o_dB;
    size_t total = 0;

    Tape(const std::vector<int>& n, int T, int Bcap) {
        const int L = (int)n.size() - 2;
        auto R = [&](int k) { return (int64_t)Bcap * n[k]; };
        auto take = [&](int64_t elems) { size_t o = total; total += ((size_t)elems + 63) & ~size_t(63); return o; };
        int64_t rmax = 0;
        for (int k = 0; k <= L; ++k) rmax = R(k) > rmax ? R(k) : rmax;
        lt.resize(L + 1);
        for (int k = 1; k <= L; ++k) {
            Layer& q = lt[k];
            const int64_t r = R(k);
            q.rs = take(6 * r); q.featf = take(7 * r); q.featb = take(7 * r);
            q.h1 = take(r * P); q.rlxf = take(r * P); q.g1 = take(r * P); q.g2 = take(r * P); q.s1 = take(r * P); q.g3 = take(r * P);
            q.rlxb = take(r * P); q.drlxf = take(r * P); q.drlxb = take(r * P);
            for (int t = 0; t < T; ++t) {
                q.nbF.push_back(take(r * P)); q.h3F.push_back(take(r * P)); q.eF.push_back(take(r * P)); q.h4F.push_back(take(r * P));
                q.nbB.push_back(take(r * P)); q.h3B.push_back(take(r * P)); q.eB.push_back(take(r * P)); q.h4B.push_back(take(r * P));
            }
        }
        const int64_t r0n = R(0);
        o_f3 = take(r0n * 3); o_f2 = take(r0n * 2); o_f4 = take((int64_t)Bcap * 4);
        o_e1 = take(r0n * P); o_i1 = take(r0n * P); o_i2 = take(r0n * P);
        o_nb0.assign(T, 0); o_i3.assign(T, 0); o_o1.assign(T, 0); o_nbo.assign(T, 0); o_o2.assign(T, 0);
        for (int t = 0; t < T; ++t) {
            if (t < T - 1) { o_nb0[t] = take(r0n * P); o_i3[t] = take(r0n * P); }
            o_o1[t] = take((int64_t)Bcap * P); o_nbo[t] = take((int64_t)Bcap * P); o_o2[t] = take((int64_t)Bcap * P);
        }
        o_mu.assign(L + 2, 0); o_dF.assign(L + 1, 0); o_dB.assign(L + 1, 0);
        for (int k = 0; k <= L; ++k) { o_mu[k] = take(R(k) * P); o_dF[k] = take(R(k) * P); o_dB[k] = take(R(k) * P); }
        o_mu[L + 1] = take((int64_t)Bcap * P);
        o_dout = take((int64_t)Bcap * P); o_dsm = take(4 * (int64_t)Bcap * P);
        o_bufA = take(rmax * P); o_bufB = take(rmax * P); o_bufC = take(rmax * P); o_bufD = take(rmax * P);
        o_tab = take((int64_t)((L * sizeof(TermLayer) + sizeof(float) - 1) / sizeof(float)));
    }
};

}  // namespace

int train_init() {
    cudaError_t e = cudaFuncSetAttribute(k_lin_bwd, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(BwdSmem));
    return (int)e;
}

size_t train_tape_floats(const std::vector<int>& n, int T, int Bcap) { return Tape(n, T, Bcap).total; }

void name_terms(const int32_t* domain, const int32_t* index, int n_terms, int B, int n_hidden, float* scores, int32_t* cnt,
                int32_t* flag, int32_t* list, int32_t* row_of, cudaStream_t st, int64_t* launches) {
    k_name_terms<<<blocks_for(n_terms, 256), 256, 0, st>>>(domain, index, n_terms, B, n_hidden, scores, cnt, flag);
    k_list_named<<<1, LIST_TH, 0, st>>>(flag, B, list, row_of, cnt);
    *launches += 2;
}

int train_wave(const GnnParams& g, const TrainParams& tp, const std::vector<LayerDev>& layers, const std::vector<int>& n,
               const std::vector<int>& hidden_off, const GnnInputs& in, int Bcap, int B, const WaveTerms& wt, float* arena,
               cudaStream_t st, int64_t* launches) {
    const int L = (int)layers.size(), T = g.T;
    auto R = [&](int k) { return (int64_t)B * n[k]; };
    const Tape tz(n, T, Bcap);
    using LayerTape = Tape::Layer;
    const std::vector<LayerTape>& lt = tz.lt;
    const size_t o_f3 = tz.o_f3, o_f2 = tz.o_f2, o_f4 = tz.o_f4, o_e1 = tz.o_e1, o_i1 = tz.o_i1, o_i2 = tz.o_i2;
    const size_t o_dout = tz.o_dout, o_dsm = tz.o_dsm;
    const std::vector<size_t>&o_nb0 = tz.o_nb0, &o_i3 = tz.o_i3, &o_o1 = tz.o_o1, &o_nbo = tz.o_nbo, &o_o2 = tz.o_o2;
    const std::vector<size_t>&o_mu = tz.o_mu, &o_dF = tz.o_dF, &o_dB = tz.o_dB;
    const int64_t r0n = R(0);
    float* base = arena;
    auto Pp = [&](size_t off) { return base + off; };
    Ctx c{g, tp, st, launches};

    // ---- forward with tape ----
    for (int k = 1; k <= L; ++k) {
        const LayerTape& q = lt[k];
        const int64_t r = R(k);
        float* rs = Pp(q.rs);
        k_row_scalars<<<blocks_for(r, 256), 256, 0, st>>>(in.lb[k], in.ub[k], in.dual[k - 1], in.pre[k - 1], in.post[k - 1],
                                                          layers[k - 1].bias_node, n[k], r, rs, Pp(q.featf), Pp(q.featb));
        ++*launches;
        const float *amb = rs + 2 * r, *d1 = rs + 4 * r, *nd2 = rs + 5 * r;
        c.fwd(FC1, {{Pp(q.featf), nullptr, 7}}, true, nullptr, Pp(q.h1), r);
        c.fwd(FC1_1, {{Pp(q.h1), nullptr, P}}, false, amb, Pp(q.rlxf), r);
        c.fwd(BC1, {{Pp(q.featb), nullptr, 7}}, true, nullptr, Pp(q.g1), r);
        c.fwd(BC1_1, {{Pp(q.g1), nullptr, P}}, true, nullptr, Pp(q.g2), r);
        c.fwd(BC1_2, {{Pp(q.g2), nullptr, P}}, false, nullptr, Pp(q.s1), r);
        c.fwd(BC2, {{Pp(q.s1), nullptr, P}, {Pp(q.s1), nd2, P}, {Pp(q.s1), d1, P}}, true, nullptr, Pp(q.g3), r);
        c.fwd(BC2_1, {{Pp(q.g3), nullptr, P}}, false, amb, Pp(q.rlxb), r);
        c.zero(Pp(q.drlxf), r * P); c.zero(Pp(q.drlxb), r * P);
    }
    k_stack<<<blocks_for(r0n, 256), 256, 0, st>>>(in.lb[0], in.pin, in.ub[0], nullptr, 3, r0n, Pp(o_f3));
    k_stack<<<blocks_for(r0n, 256), 256, 0, st>>>(in.lb[0], in.ub[0], nullptr, nullptr, 2, r0n, Pp(o_f2));
    k_stack<<<blocks_for(B, 256), 256, 0, st>>>(in.lb[L + 1], in.ub[L + 1], in.pout, in.bp, 4, B, Pp(o_f4));
    *launches += 3;
    c.fwd(INP_F, {{Pp(o_f3), nullptr, 3}}, true, nullptr, Pp(o_e1), r0n);
    c.fwd(INP_F_1, {{Pp(o_e1), nullptr, P}}, false, nullptr, Pp(o_mu[0]), r0n);
    if (T > 1) {
        c.fwd(INP_B, {{Pp(o_f2), nullptr, 2}}, true, nullptr, Pp(o_i1), r0n);
        c.fwd(INP_B_1, {{Pp(o_i1), nullptr, P}}, false, nullptr, Pp(o_i2), r0n);
    }
    for (int t = 0; t < T; ++t) {
        for (int k = 1; k <= L; ++k) {
            const LayerTape& q = lt[k];
            const int64_t r = R(k);
            const float* rs = Pp(q.rs);
            prop_forward(layers[k - 1], Pp(o_mu[k - 1]), Pp(q.nbF[t]), B, st, launches);
            c.fwd(FC3, {{Pp(q.nbF[t]), rs, P}, {Pp(q.nbF[t]), rs + r, P}}, true, nullptr, Pp(q.h3F[t]), r);
            c.fwd(FC3_2, {{Pp(q.h3F[t]), nullptr, P}}, false, nullptr, Pp(q.eF[t]), r);
            c.fwd(FC4, {{Pp(q.rlxf), nullptr, P}, {Pp(q.eF[t]), nullptr, P}}, true, nullptr, Pp(q.h4F[t]), r);
            c.fwd(FC4_2, {{Pp(q.h4F[t]), nullptr, P}}, false, rs + 3 * r, Pp(o_mu[k]), r);
        }
        k_wp_reduce<<<B, 64, 0, st>>>(in.wp, Pp(o_mu[L]), n[L], 0, Pp(o_nbo[t]));
        ++*launches;
        c.fwd(OUT1, {{Pp(o_f4), nullptr, 4}}, true, nullptr, Pp(o_o1[t]), B);
        c.fwd(OUT2, {{Pp(o_o1[t]), nullptr, P}, {Pp(o_nbo[t]), nullptr, P}}, true, nullptr, Pp(o_o2[t]), B);
        c.fwd(OUT3, {{Pp(o_o2[t]), nullptr, P}}, false, nullptr, Pp(o_mu[L + 1]), B);
        for (int k = L; k >= 1; --k) {
            const LayerTape& q = lt[k];
            const int64_t r = R(k);
            const float* rs = Pp(q.rs);
            if (k == L) prop_property_backward(in.wp, Pp(o_mu[L + 1]), Pp(q.nbB[t]), n[L], B, st, launches);
            else prop_backward(layers[k], Pp(o_mu[k + 1]), Pp(q.nbB[t]), B, true, st, launches);
            c.fwd(BC3, {{Pp(q.nbB[t]), rs, P}, {Pp(q.nbB[t]), rs + r, P}}, true, nullptr, Pp(q.h3B[t]), r);
            c.fwd(BC3_1, {{Pp(q.h3B[t]), nullptr, P}}, false, nullptr, Pp(q.eB[t]), r);
            c.fwd(BC4, {{Pp(q.rlxb), nullptr, P}, {Pp(q.eB[t]), nullptr, P}}, true, nullptr, Pp(q.h4B[t]), r);
            c.fwd(BC4_1, {{Pp(q.h4B[t]), nullptr, P}}, false, rs + 3 * r, Pp(o_mu[k]), r);
        }
        if (t < T - 1) {
            prop_backward(layers[0], Pp(o_mu[1]), Pp(o_nb0[t]), B, false, st, launches);
            c.fwd(INP_B2, {{Pp(o_i2), nullptr, P}, {Pp(o_nb0[t]), nullptr, P}}, true, nullptr, Pp(o_i3[t]), r0n);
            c.fwd(INP_B2_2, {{Pp(o_i3[t]), nullptr, P}}, false, nullptr, Pp(o_mu[0]), r0n);
        }
    }

    // ---- backward ----
    for (int k = 1; k <= L; ++k) c.zero(Pp(o_dB[k]), R(k) * P);
    {   // score head on the rows the loss names; the layer table points into this arena (a stream-ordered copy from pageable
        // memory returns after the source has been read)
        std::vector<TermLayer> tab(L);
        for (int k = 1; k <= L; ++k) tab[k - 1] = TermLayer{Pp(o_mu[k]), Pp(o_dB[k]), hidden_off[k], n[k]};
        TermLayer* d_tab = reinterpret_cast<TermLayer*>(Pp(tz.o_tab));
        cudaMemcpyAsync(d_tab, tab.data(), L * sizeof(TermLayer), cudaMemcpyHostToDevice, st);
        ScoreTermArgs a{};
        a.domain = wt.domain; a.index = wt.index; a.coeff = wt.coeff; a.row_of = wt.row_of;
        a.B = wt.B; a.n_hidden = wt.n_hidden; a.row0 = wt.row0; a.rows = B;
        a.layers = d_tab; a.L = L;
        a.w_fnode = tp.w[FNODE]; a.b_fnode = tp.b[FNODE]; a.w_fscore = tp.w[FSCORE]; a.b_fscore = tp.b[FSCORE];
        a.dW_fnode = tp.dw[FNODE]; a.db_fnode = tp.db[FNODE]; a.dW_fscore = tp.dw[FSCORE]; a.db_fscore = tp.db[FSCORE];
        a.scores = wt.scores;
        k_score_terms<<<wt.n_terms, 64, 0, st>>>(a);
        ++*launches;
    }
    float *bufA = Pp(tz.o_bufA), *bufB = Pp(tz.o_bufB), *bufC = Pp(tz.o_bufC), *bufD = Pp(tz.o_bufD);
    for (int t = T - 1; t >= 0; --t) {
        if (t < T - 1) {
            // input-layer update of round t produced the mu[0] that round t + 1 read: its gradient is dF[0] (graph_conv.py:360-385)
            float* dmu0 = Pp(o_dF[0]);
            c.bwd(INP_B2_2, {{{Pp(o_i3[t]), nullptr, P}, bufA, false}}, dmu0, nullptr, nullptr, r0n);                       // dI3
            c.bwd(INP_B2, {{{Pp(o_i2), nullptr, P}, bufB, false}, {{Pp(o_nb0[t]), nullptr, P}, bufC, false}}, bufA, Pp(o_i3[t]), nullptr, r0n);
            c.bwd(INP_B_1, {{{Pp(o_i1), nullptr, P}, bufA, false}}, bufB, nullptr, nullptr, r0n);                           // dI1
            c.bwd(INP_B, {{{Pp(o_f2), nullptr, 2}, nullptr, false}}, bufA, Pp(o_i1), nullptr, r0n);
            prop_forward(layers[0], bufC, bufD, B, st, launches);                 // (A_1^T)^T dnb0
            c.add(Pp(o_dB[1]), bufD, R(1) * P);
        }
        c.zero(Pp(o_dout), (int64_t)B * P);
        for (int k = 1; k <= L; ++k) {       // reverse of the backward sweep (it ran k = L .. 1)
            const LayerTape& q = lt[k];
            const int64_t r = R(k);
            const float* rs = Pp(q.rs);
            c.bwd(BC4_1, {{{Pp(q.h4B[t]), nullptr, P}, bufA, false}}, Pp(o_dB[k]), nullptr, rs + 3 * r, r);                 // dH4
            c.bwd(BC4, {{{Pp(q.rlxb), nullptr, P}, Pp(q.drlxb), true}, {{Pp(q.eB[t]), nullptr, P}, bufB, false}}, bufA, Pp(q.h4B[t]), nullptr, r);
            c.bwd(BC3_1, {{{Pp(q.h3B[t]), nullptr, P}, bufA, false}}, bufB, nullptr, nullptr, r);                           // dH3
            c.bwd(BC3, {{{Pp(q.nbB[t]), rs, P}, bufB, false}, {{Pp(q.nbB[t]), rs + r, P}, bufB, true}}, bufA, Pp(q.h3B[t]), nullptr, r);   // dNB
            if (k == L) {
                k_wp_reduce<<<B, 64, 0, st>>>(in.wp, bufB, n[L], 1, Pp(o_dout));
                ++*launches;
            } else {
                const LayerDev& nx = layers[k];
                const float* src = bufB;
                if (nx.kind == GNNB_LAYER_CONV) {
                    k_div_freq<<<blocks_for(r * 16, 256), 256, 0, st>>>(nx, bufB, bufC, r * 16);
                    ++*launches;
                    src = bufC;
                }
                prop_forward(nx, src, bufD, B, st, launches);
                c.add(Pp(o_dB[k + 1]), bufD, R(k + 1) * P);
            }
        }
        // output node (graph_conv.py:196-210)
        c.bwd(OUT3, {{{Pp(o_o2[t]), nullptr, P}, Pp(o_dsm), false}}, Pp(o_dout), nullptr, nullptr, B);
        c.bwd(OUT2, {{{Pp(o_o1[t]), nullptr, P}, Pp(o_dsm) + (size_t)B * P, false}, {{Pp(o_nbo[t]), nullptr, P}, Pp(o_dsm) + 2 * (size_t)B * P, false}},
              Pp(o_dsm), Pp(o_o2[t]), nullptr, B);
        c.bwd(OUT1, {{{Pp(o_f4), nullptr, 4}, nullptr, false}}, Pp(o_dsm) + (size_t)B * P, Pp(o_o1[t]), nullptr, B);
        prop_property_backward(in.wp, Pp(o_dsm) + 2 * (size_t)B * P, Pp(o_dF[L]), n[L], B, st, launches);
        for (int k = L; k >= 1; --k) {       // reverse of the forward sweep
            const LayerTape& q = lt[k];
            const int64_t r = R(k);
            const float* rs = Pp(q.rs);
            c.bwd(FC4_2, {{{Pp(q.h4F[t]), nullptr, P}, bufA, false}}, Pp(o_dF[k]), nullptr, rs + 3 * r, r);
            c.bwd(FC4, {{{Pp(q.rlxf), nullptr, P}, Pp(q.drlxf), true}, {{Pp(q.eF[t]), nullptr, P}, bufB, false}}, bufA, Pp(q.h4F[t]), nullptr, r);
            c.bwd(FC3_2, {{{Pp(q.h3F[t]), nullptr, P}, bufA, false}}, bufB, nullptr, nullptr, r);
            c.bwd(FC3, {{{Pp(q.nbF[t]), rs, P}, bufB, false}, {{Pp(q.nbF[t]), rs + r, P}, bufB, true}}, bufA, Pp(q.h3F[t]), nullptr, r);
            prop_backward(layers[k - 1], bufB, Pp(o_dF[k - 1]), B, false, st, launches);     // (A_k)^T dnb
        }
        if (t == 0) {
            c.bwd(INP_F_1, {{{Pp(o_e1), nullptr, P}, bufA, false}}, Pp(o_dF[0]), nullptr, nullptr, r0n);
            c.bwd(INP_F, {{{Pp(o_f3), nullptr, 3}, nullptr, false}}, bufA, Pp(o_e1), nullptr, r0n);
        } else {
            for (int k = 1; k <= L; ++k) c.zero(Pp(o_dB[k]), R(k) * P);
        }
    }
    for (int k = 1; k <= L; ++k) {           // relaxation features: the sum of the rounds' gradients
        const LayerTape& q = lt[k];
        const int64_t r = R(k);
        const float* rs = Pp(q.rs);
        const float *amb = rs + 2 * r, *d1 = rs + 4 * r, *nd2 = rs + 5 * r;
        c.bwd(FC1_1, {{{Pp(q.h1), nullptr, P}, bufA, false}}, Pp(q.drlxf), nullptr, amb, r);
        c.bwd(FC1, {{{Pp(q.featf), nullptr, 7}, nullptr, false}}, bufA, Pp(q.h1), nullptr, r);
        c.bwd(BC2_1, {{{Pp(q.g3), nullptr, P}, bufA, false}}, Pp(q.drlxb), nullptr, amb, r);
        c.bwd(BC2, {{{Pp(q.s1), nullptr, P}, bufB, false}, {{Pp(q.s1), nd2, P}, bufB, true}, {{Pp(q.s1), d1, P}, bufB, true}}, bufA, Pp(q.g3), nullptr, r);
        c.bwd(BC1_2, {{{Pp(q.g2), nullptr, P}, bufA, false}}, bufB, nullptr, nullptr, r);
        c.bwd(BC1_1, {{{Pp(q.g1), nullptr, P}, bufB, false}}, bufA, Pp(q.g2), nullptr, r);
        c.bwd(BC1, {{{Pp(q.featb), nullptr, 7}, nullptr, false}}, bufB, Pp(q.g1), nullptr, r);
    }
    return (int)cudaGetLastError();
}

void adam_step(float* p, const float* grad, float* m, float* v, int64_t numel, float lr, float b1, float b2, float eps, float wd,
               int step, cudaStream_t st, int64_t* launches) {
    const float bc1 = 1.0f - (float)pow((double)b1, step);
    const float bc2_sqrt = (float)sqrt(1.0 - pow((double)b2, step));
    k_adam<<<blocks_for(numel, 256), 256, 0, st>>>(p, grad, m, v, numel, lr, b1, b2, eps, wd, bc1, bc2_sqrt);
    ++*launches;
}

}  // namespace gnnb
