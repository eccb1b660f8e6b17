// Propagation of the 64-channel node embeddings through the verified network's own edges, plus the
// single-node output update and the masked argmax.  fp32 on CUDA cores, embeddings node-major
// [Bc, n_k, 64] so every access is a 256-byte row per node.
//
//   prop_forward   nb = A_k applied to mu[k-1] per embedding channel, bias NOT added
//                  (graph_conv.py:110-121 conv2d over the (B*p)-batched embeddings; :130-132 W @ mu)
//   prop_backward  nb = A_{k+1}^T applied to mu[k+1]; conv: conv_transpose2d / freq with freq the tap count
//                  per input position (graph_conv.py:299-318), not divided for the input layer (:361-372);
//                  linear: W^T @ mu (:320-322)
//   prop_property_backward   nb[b,n,:] = Wp[b,n] * mu[L+1][b,:]   (graph_conv.py:324-326, rank-1)
//   output_node    graph_conv.py:196-210
//   masked_argmax  torch.max over the candidate rows + index mapping (graph_score.py:41-47)
//   masked_topk    the k best candidates per row in the argmax's order (radix select + bitonic sort of at most 64 entries)
//   gather_rows / scatter_rescored   the sub-frontier of option "rescore" in, its results out
#include <cuda_fp16.h>
#include <math.h>

#include "gnnb_common.cuh"

namespace gnnb {
namespace {

constexpr int CG = 8;            // output channels accumulated per pass in the conv kernels

// one warp per output position (b, y, x); lane owns embedding channels 2*lane, 2*lane+1
__global__ void __launch_bounds__(256) k_conv_forward(LayerDev L, const float* __restrict__ mu_prev,
                                                      float* __restrict__ nb, int Bc) {
    extern __shared__ __align__(16) float wsm[];      // [(ci,ky,kx)][co]
    const int K = L.c_in * L.ksize * L.ksize;
    for (int i = threadIdx.x; i < K * L.c_out; i += blockDim.x) {
        const int co = i % L.c_out, kk = i / L.c_out;
        wsm[i] = L.weight[co * K + kk];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int hw_out = L.h_out * L.w_out, hw_in = L.h_in * L.w_in;
    const int64_t npos = (int64_t)Bc * hw_out;
    for (int64_t pos = (int64_t)blockIdx.x * wpb + warp; pos < npos; pos += (int64_t)gridDim.x * wpb) {
        const int b = (int)(pos / hw_out), yx = (int)(pos % hw_out);
        const int y = yx / L.w_out, x = yx % L.w_out;
        const float* src = mu_prev + (int64_t)b * L.n_in * P + lane * 2;
        float* dst = nb + (int64_t)b * L.n_out * P + lane * 2;
        for (int g0 = 0; g0 < L.c_out; g0 += CG) {
            float2 acc[CG];
#pragma unroll
            for (int j = 0; j < CG; ++j) acc[j] = make_float2(0.f, 0.f);
            for (int ci = 0; ci < L.c_in; ++ci)
                for (int ky = 0; ky < L.ksize; ++ky) {
                    const int yy = y * L.stride + ky - L.pad;
                    if (yy < 0 || yy >= L.h_in) continue;
                    for (int kx = 0; kx < L.ksize; ++kx) {
                        const int xx = x * L.stride + kx - L.pad;
                        if (xx < 0 || xx >= L.w_in) continue;
                        const float2 v = *reinterpret_cast<const float2*>(src + (int64_t)(ci * hw_in + yy * L.w_in + xx) * P);
                        const float* w = wsm + ((ci * L.ksize + ky) * L.ksize + kx) * L.c_out + g0;
#pragma unroll
                        for (int j = 0; j < CG; ++j)
                            if (g0 + j < L.c_out) {
                                acc[j].x = fmaf(w[j], v.x, acc[j].x);
                                acc[j].y = fmaf(w[j], v.y, acc[j].y);
                            }
                    }
                }
#pragma unroll
            for (int j = 0; j < CG; ++j)
                if (g0 + j < L.c_out)
                    *reinterpret_cast<float2*>(dst + (int64_t)((g0 + j) * hw_out + yx) * P) = acc[j];
        }
    }
}

// one warp per input position (b, yi, xi)
__global__ void __launch_bounds__(256) k_conv_backward(LayerDev L, const float* __restrict__ mu_next,
                                                       float* __restrict__ nb, int Bc, int normalise) {
    extern __shared__ __align__(16) float wsm[];      // [(co,ky,kx)][ci]
    const int kk2 = L.ksize * L.ksize;
    for (int i = threadIdx.x; i < L.c_out * kk2 * L.c_in; i += blockDim.x) {
        const int ci = i % L.c_in, r = i / L.c_in;
        const int co = r / kk2, t = r % kk2;
        wsm[i] = L.weight[(co * L.c_in + ci) * kk2 + t];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpb = blockDim.x >> 5;
    const int hw_out = L.h_out * L.w_out, hw_in = L.h_in * L.w_in;
    const int64_t npos = (int64_t)Bc * hw_in;
    for (int64_t pos = (int64_t)blockIdx.x * wpb + warp; pos < npos; pos += (int64_t)gridDim.x * wpb) {
        const int b = (int)(pos / hw_in), yx = (int)(pos % hw_in);
        const int yi = yx / L.w_in, xi = yx % L.w_in;
        const float* src = mu_next + (int64_t)b * L.n_out * P + lane * 2;
        float* dst = nb + (int64_t)b * L.n_in * P + lane * 2;
        for (int g0 = 0; g0 < L.c_in; g0 += CG) {
            float2 acc[CG];
#pragma unroll
            for (int j = 0; j < CG; ++j) acc[j] = make_float2(0.f, 0.f);
            int taps = 0;
            for (int ky = 0; ky < L.ksize; ++ky) {
                const int ty = yi + L.pad - ky;
                if (ty < 0 || ty % L.stride != 0) continue;
                const int yo = ty / L.stride;
                if (yo >= L.h_out) continue;
                for (int kx = 0; kx < L.ksize; ++kx) {
                    const int tx = xi + L.pad - kx;
                    if (tx < 0 || tx % L.stride != 0) continue;
                    const int xo = tx / L.stride;
                    if (xo >= L.w_out) continue;
                    ++taps;
                    for (int co = 0; co < L.c_out; ++co) {
                        const float2 v = *reinterpret_cast<const float2*>(src + (int64_t)(co * hw_out + yo * L.w_out + xo) * P);
                        const float* w = wsm + ((co * L.ksize + ky) * L.ksize + kx) * L.c_in + g0;
#pragma unroll
                        for (int j = 0; j < CG; ++j)
                            if (g0 + j < L.c_in) {
                                acc[j].x = fmaf(w[j], v.x, acc[j].x);
                                acc[j].y = fmaf(w[j], v.y, acc[j].y);
                            }
                    }
                }
            }
            // freq = conv_transpose2d(ones, ones): number of (output position, tap) pairs reaching this input
            const float freq = (float)taps;
#pragma unroll
            for (int j = 0; j < CG; ++j)
                if (g0 + j < L.c_in) {
                    float2 o = acc[j];
                    if (normalise) { o.x = __fdiv_rn(o.x, freq); o.y = __fdiv_rn(o.y, freq); }
                    *reinterpret_cast<float2*>(dst + (int64_t)((g0 + j) * hw_in + yx) * P) = o;
                }
        }
    }
}

// nb[b][m][c] = sum_k A(m,k) * mu[b][k][c],  A(m,k) = W[m*sm + k*sk]   (forward: sm = K, sk = 1; backward: sm = 1, sk = M)
__global__ void __launch_bounds__(256) k_linear(const float* __restrict__ W, int M, int K, int sm, int sk,
                                                const float* __restrict__ mu, float* __restrict__ nb) {
    __shared__ float As[32][33];
    __shared__ __align__(16) float Ms[32][64];
    const int b = blockIdx.y, m0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const float* mub = mu + (int64_t)b * K * P;
    float acc[2][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};
    for (int k0 = 0; k0 < K; k0 += 32) {
        __syncthreads();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int idx = threadIdx.x + i * 256;
            int kk, mm;
            if (sk == 1) { kk = idx & 31; mm = idx >> 5; } else { mm = idx & 31; kk = idx >> 5; }
            const int m = m0 + mm, k = k0 + kk;
            As[kk][mm] = (m < M && k < K) ? W[(int64_t)m * sm + (int64_t)k * sk] : 0.f;
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int idx = threadIdx.x + i * 256;
            const int kk = idx >> 4, c4 = idx & 15;
            const int k = k0 + kk;
            const float4 v = (k < K) ? *reinterpret_cast<const float4*>(mub + (int64_t)k * P + c4 * 4) : make_float4(0, 0, 0, 0);
            *reinterpret_cast<float4*>(&Ms[kk][c4 * 4]) = v;
        }
        __syncthreads();
#pragma unroll 8
        for (int kk = 0; kk < 32; ++kk) {
            const float a0 = As[kk][ty * 2], a1 = As[kk][ty * 2 + 1];
            const float4 v = *reinterpret_cast<const float4*>(&Ms[kk][tx * 4]);
            acc[0][0] = fmaf(a0, v.x, acc[0][0]); acc[0][1] = fmaf(a0, v.y, acc[0][1]);
            acc[0][2] = fmaf(a0, v.z, acc[0][2]); acc[0][3] = fmaf(a0, v.w, acc[0][3]);
            acc[1][0] = fmaf(a1, v.x, acc[1][0]); acc[1][1] = fmaf(a1, v.y, acc[1][1]);
            acc[1][2] = fmaf(a1, v.z, acc[1][2]); acc[1][3] = fmaf(a1, v.w, acc[1][3]);
        }
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const int m = m0 + ty * 2 + i;
        if (m < M)
            *reinterpret_cast<float4*>(nb + ((int64_t)b * M + m) * P + tx * 4) =
                make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    }
}

__global__ void k_property_backward(const float* __restrict__ wp, const float* __restrict__ mu_out,
                                    float* __restrict__ nb, int nL, int64_t total4) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
        const int c4 = (int)(i & 15);
        const int64_t row = i >> 4;              // b * nL + n
        const int64_t b = row / nL;
        const float w = wp[row];
        const float4 m = *reinterpret_cast<const float4*>(mu_out + b * P + c4 * 4);
        *reinterpret_cast<float4*>(nb + row * P + c4 * 4) = make_float4(w * m.x, w * m.y, w * m.z, w * m.w);
    }
}

// embedding channel c of global row `row`: fp32 [rows][64], or (mu_image) the tensor-core path's mu tile image —
// fp16 hi + lo planes, K-major SWIZZLE_128B, scaled by 1/8 (gnnb_umma.cuh)
__device__ __forceinline__ float mu_at(const float* __restrict__ mu, int mu_image, int64_t row, int c) {
    if (!mu_image) return mu[row * P + c];
    const uint32_t r = (uint32_t)(row & 127);
    const uint32_t off = (r >> 3) * 1024u + (r & 7u) * 128u + ((((uint32_t)c >> 3) ^ (r & 7u)) << 4) + ((uint32_t)c & 7u) * 2u;
    const unsigned char* tile = reinterpret_cast<const unsigned char*>(mu) + (row >> 7) * 32768;
    const __half hi = *reinterpret_cast<const __half*>(tile + off), lo = *reinterpret_cast<const __half*>(tile + 16384 + off);
    return (__half2float(hi) + __half2float(lo)) * 8.0f;
}

// one 256-thread block per subdomain: thread (part, c) sums every 4th node of channel c, so that four independent
// chains of loads are in flight per channel (the sum over the last hidden layer is latency-bound otherwise)
__global__ void __launch_bounds__(256) k_output_node(GnnParams g, const float* __restrict__ wp, const float* __restrict__ bp,
                                                     const float* __restrict__ mu_L, int mu_image, int mu_stride, const float* __restrict__ lb_out,
                                                     const float* __restrict__ ub_out, const float* __restrict__ prim_out,
                                                     float* __restrict__ mu_out, int nL) {
    __shared__ float part_s[4][P];
    __shared__ float cat[2 * P];
    __shared__ float h2[P];
    const int b = blockIdx.x, c = threadIdx.x & 63, part = threadIdx.x >> 6;
    float nbv = 0.f;                                       // prop.weight @ mu[L]  (graph_conv.py:196)
#pragma unroll 4
    for (int n = part; n < nL; n += 4) nbv = fmaf(wp[(int64_t)b * nL + n], mu_at(mu_L, mu_image, (int64_t)b * mu_stride + n, c), nbv);
    part_s[part][c] = nbv;
    __syncthreads();
    if (part != 0) return;
    nbv = (part_s[0][c] + part_s[1][c]) + (part_s[2][c] + part_s[3][c]);
    const float feat[4] = {lb_out[b], ub_out[b], prim_out[b], bp[b]};   // graph_conv.py:202-205
    float h = g.bias[OUT1][c];
#pragma unroll
    for (int k = 0; k < 4; ++k) h = fmaf(feat[k], g.wt[OUT1][k * P + c], h);
    cat[c] = (h != h) ? h : fmaxf(h, 0.f);
    cat[P + c] = nbv;
    asm volatile("bar.sync 1, 64;" ::: "memory");
    float a = g.bias[OUT2][c];
    for (int k = 0; k < 2 * P; ++k) a = fmaf(cat[k], g.wt[OUT2][k * P + c], a);
    h2[c] = (a != a) ? a : fmaxf(a, 0.f);
    asm volatile("bar.sync 1, 64;" ::: "memory");
    float o = g.bias[OUT3][c];
    for (int k = 0; k < P; ++k) o = fmaf(h2[k], g.wt[OUT3][k * P + c], o);
    mu_out[(int64_t)b * P + c] = o;
}

__device__ __forceinline__ bool better(float a, int ia, float b, int ib) {
    if (ib < 0) return ia >= 0;
    if (ia < 0) return false;
    const bool na = a != a, nbn = b != b;          // torch.max propagates NaN and returns the first one
    if (na || nbn) return na && (!nbn || ia < ib);
    return a > b || (a == b && ia < ib);
}

// one block per subdomain: max over rows with mask != 0, lowest index on ties
__global__ void __launch_bounds__(256) k_masked_argmax(const float* __restrict__ scores, const float* __restrict__ mask,
                                                       int n_hidden, float* __restrict__ best_score,
                                                       int32_t* __restrict__ best_idx, gnnb_winner* __restrict__ winners) {
    __shared__ float sv[8];
    __shared__ int si[8];
    const int b = blockIdx.x;
    const float* s = scores + (int64_t)b * n_hidden;
    const float* m = mask + (int64_t)b * n_hidden;
    float bv = -INFINITY;
    int bi = -1;
    for (int i = threadIdx.x; i < n_hidden; i += blockDim.x)
        if (m[i] != 0.f && better(s[i], i, bv, bi)) { bv = s[i]; bi = i; }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
        if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (lane == 0) { sv[warp] = bv; si[warp] = bi; }
    __syncthreads();
    if (warp == 0) {
        bv = lane < 8 ? sv[lane] : -INFINITY;
        bi = lane < 8 ? si[lane] : -1;
#pragma unroll
        for (int off = 4; off >= 1; off >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, bv, off);
            const int oi = __shfl_xor_sync(0xffffffffu, bi, off);
            if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
        }
        if (lane == 0) {
            const float v = bi < 0 ? -INFINITY : bv;
            if (best_score != nullptr) { best_score[b] = v; best_idx[b] = bi; }
            if (winners != nullptr) {      // one 8-byte store: the record the winner all-gather sends (gnn_branching_b200/dist.py)
                gnnb_winner w; w.score = v; w.index = bi;
                winners[b] = w;
            }
        }
    }
}

// Order-preserving key of a candidate's score: a larger key comes first in the order of better().  Every NaN maps above +inf
// (NaN first, and NaN ties go by index), -0.0 maps to the key of +0.0 (better() compares with a > b).  0 is no float's key
// (the smallest, -inf, is 0x007fffff) and marks an entry that is not a candidate.
__device__ __forceinline__ uint32_t topk_key(float s, float m) {
    if (m == 0.f) return 0u;
    if (s != s) return 0xffffffffu;
    const uint32_t u = s == 0.f ? 0u : __float_as_uint(s);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

constexpr int TOPK_BT = 256;             // threads per block; the 256 histogram bins are one per thread
constexpr int TOPK_SMEM_KEYS = 11264;    // rows up to this length keep their keys in shared memory (44 KB): the row is read once

// one block per row: the k best candidates, ordered by (key descending, index ascending); (-inf, -1) past the last candidate.
// 1. radix select with 8-bit digits (four histogram passes) finds T, the key of the kk-th candidate, kk = min(k, candidates),
//    and how many candidates with key T belong to the top kk;
// 2. one pass in index order takes every candidate above T and the first of those equal to T (ballot + block prefix count);
// 3. a bitonic sort orders the at most 64 taken entries.
// Histogram counts are integers and the sort sees a set of distinct (key, index) pairs: no result depends on the order of the
// atomics or on the block size.
__global__ void __launch_bounds__(TOPK_BT) k_masked_topk(const float* __restrict__ scores, const float* __restrict__ mask, int n,
                                                         int k, float* __restrict__ top_score, int32_t* __restrict__ top_idx) {
    extern __shared__ uint32_t skey[];                    // [n] when n <= TOPK_SMEM_KEYS
    __shared__ uint32_t hist[256];
    __shared__ uint32_t sel_key[GNNB_TOPK_MAX];
    __shared__ int sel_idx[GNNB_TOPK_MAX];
    __shared__ int wcnt[TOPK_BT / 32];
    __shared__ uint32_t s_prefix, s_rem, s_kk;
    __shared__ int s_above;
    const int b = blockIdx.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const float* s = scores + (int64_t)b * n;
    const float* m = mask ? mask + (int64_t)b * n : nullptr;
    const bool cached = n <= TOPK_SMEM_KEYS;
    auto key_at = [&](int i) { return cached ? skey[i] : topk_key(s[i], m ? m[i] : 1.f); };
    if (cached)
        for (int i = t; i < n; i += TOPK_BT) skey[i] = topk_key(s[i], m ? m[i] : 1.f);

    uint32_t prefix = 0u, pmask = 0u, rem = 0u;
    for (int shift = 24; shift >= 0; shift -= 8) {
        hist[t] = 0u;
        __syncthreads();
        for (int i = t; i < n; i += TOPK_BT) {
            const uint32_t key = key_at(i);
            if (key != 0u && (key & pmask) == prefix) atomicAdd(&hist[(key >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (warp == 0) {                                  // lane l holds digits 255 - 8 l - j, j = 0..7: descending digit order
            uint32_t c[8], sum = 0u;
#pragma unroll
            for (int j = 0; j < 8; ++j) { c[j] = hist[255 - 8 * lane - j]; sum += c[j]; }
            uint32_t incl = sum;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, incl, off);
                if (lane >= off) incl += v;
            }
            uint32_t r = rem;
            if (shift == 24) {                            // the first pass counts every candidate
                const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
                r = total < (uint32_t)k ? total : (uint32_t)k;
                if (lane == 0) s_kk = r;
            }
            const uint32_t excl = incl - sum;
            if (r > 0u && excl < r && r <= incl) {        // the digit of the r-th largest key lies in this lane's bins
                uint32_t acc = excl;
                int j = -1;
#pragma unroll
                for (int jj = 0; jj < 8; ++jj)           // unrolled: c stays in registers
                    if (j < 0) { if (acc + c[jj] >= r) j = jj; else acc += c[jj]; }
                s_prefix = prefix | ((uint32_t)(255 - 8 * lane - j) << shift);
                s_rem = r - acc;
            }
        }
        __syncthreads();
        if (s_kk == 0u) break;
        prefix = s_prefix;
        rem = s_rem;
        pmask |= 255u << shift;
    }
    const int kk = (int)s_kk;
    if (kk > 0) {
        const uint32_t T = prefix;
        const int need_eq = (int)rem, above = kk - (int)rem;
        if (t == 0) s_above = 0;
        __syncthreads();
        int eq_run = 0;
        for (int base = 0; base < n; base += TOPK_BT) {
            const int i = base + t;
            const uint32_t key = i < n ? key_at(i) : 0u;
            if (key > T) {
                const int slot = atomicAdd(&s_above, 1);
                sel_key[slot] = key; sel_idx[slot] = i;
            }
            const unsigned bal = __ballot_sync(0xffffffffu, key == T);
            if (lane == 0) wcnt[warp] = __popc(bal);
            __syncthreads();
            int pos = eq_run + __popc(bal & ((1u << lane) - 1u)), tile = 0;
#pragma unroll
            for (int w = 0; w < TOPK_BT / 32; ++w) { const int c = wcnt[w]; if (w < warp) pos += c; tile += c; }
            if (key == T && pos < need_eq) { sel_key[above + pos] = key; sel_idx[above + pos] = i; }
            eq_run += tile;
            const bool done = eq_run >= need_eq && s_above == above;
            __syncthreads();
            if (done) break;
        }
        if (t < GNNB_TOPK_MAX && t >= kk) { sel_key[t] = 0u; sel_idx[t] = 0x7fffffff; }     // padding sorts last
        __syncthreads();
        for (int size = 2; size <= GNNB_TOPK_MAX; size <<= 1)
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                if (t < GNNB_TOPK_MAX) {
                    const int p = t ^ stride;
                    if (p > t) {
                        const uint32_t ka = sel_key[t], kb = sel_key[p];
                        const int ia = sel_idx[t], ib = sel_idx[p];
                        const bool p_first = kb > ka || (kb == ka && ib < ia);
                        if (p_first == ((t & size) == 0)) {
                            sel_key[t] = kb; sel_key[p] = ka; sel_idx[t] = ib; sel_idx[p] = ia;
                        }
                    }
                }
                __syncthreads();
            }
    }
    for (int j = t; j < k; j += TOPK_BT) {
        float v = -INFINITY;
        int ix = -1;
        if (j < kk) { ix = sel_idx[j]; v = s[ix]; }       // the score's own bits (-0.0 stays -0.0)
        top_score[(int64_t)b * k + j] = v;
        top_idx[(int64_t)b * k + j] = ix;
    }
}

// block (i, a): row rows[i] of array a -> row i of its destination
__global__ void __launch_bounds__(256) k_gather_rows(const RowGather* __restrict__ tab, const int32_t* __restrict__ rows) {
    const RowGather t = tab[blockIdx.y];
    const float* src = t.src + (int64_t)rows[blockIdx.x] * t.per;
    float* dst = t.dst + (int64_t)blockIdx.x * t.per;
    for (int64_t j = threadIdx.x; j < t.per; j += blockDim.x) dst[j] = src[j];
}

// block i: the re-scored results of sub-frontier row i (k entries) -> row rows[i] of the call's outputs
__global__ void __launch_bounds__(256) k_scatter_rescored(const int32_t* __restrict__ rows, int k, const float* __restrict__ sub_best,
                                                          const int32_t* __restrict__ sub_idx, const float* __restrict__ sub_scores,
                                                          int n_hidden, float* __restrict__ best_score, int32_t* __restrict__ best_idx,
                                                          gnnb_winner* __restrict__ winners, float* __restrict__ scores,
                                                          int32_t* __restrict__ flag) {
    const int i = blockIdx.x;
    const int64_t b = rows[i];
    if (best_score != nullptr && threadIdx.x < k) {
        best_score[b * k + threadIdx.x] = sub_best[(int64_t)i * k + threadIdx.x];
        best_idx[b * k + threadIdx.x] = sub_idx[(int64_t)i * k + threadIdx.x];
    }
    if (threadIdx.x == 0) {
        if (winners != nullptr) {
            gnnb_winner w; w.score = sub_best[i]; w.index = sub_idx[i];
            winners[b] = w;
        }
        flag[b] = 0;
    }
    if (scores != nullptr)
        for (int j = threadIdx.x; j < n_hidden; j += blockDim.x) scores[b * n_hidden + j] = sub_scores[(int64_t)i * n_hidden + j];
}

int capped_grid(int64_t blocks) {
    const int64_t cap = 148 * 16;
    return (int)(blocks < 1 ? 1 : (blocks < cap ? blocks : cap));
}

}  // namespace

int prop_init(int max_smem_bytes) {
    cudaError_t e;
    if ((e = cudaFuncSetAttribute(k_conv_forward, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem_bytes)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(k_conv_backward, cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem_bytes)) != cudaSuccess) return e;
    return 0;
}

void prop_forward(const LayerDev& L, const float* mu_prev, float* nb, int Bc, cudaStream_t st, int64_t* launches) {
    if (L.kind == GNNB_LAYER_CONV) {
        const int64_t npos = (int64_t)Bc * L.h_out * L.w_out;
        const size_t smem = sizeof(float) * L.c_in * L.ksize * L.ksize * L.c_out;
        k_conv_forward<<<capped_grid((npos + 7) / 8), 256, smem, st>>>(L, mu_prev, nb, Bc);
    } else {
        dim3 grid((L.n_out + 31) / 32, Bc);
        k_linear<<<grid, 256, 0, st>>>(L.weight, L.n_out, L.n_in, L.n_in, 1, mu_prev, nb);
    }
    ++*launches;
}

void prop_backward(const LayerDev& L, const float* mu_next, float* nb, int Bc, bool normalise, cudaStream_t st, int64_t* launches) {
    if (L.kind == GNNB_LAYER_CONV) {
        const int64_t npos = (int64_t)Bc * L.h_in * L.w_in;
        const size_t smem = sizeof(float) * L.c_in * L.ksize * L.ksize * L.c_out;
        k_conv_backward<<<capped_grid((npos + 7) / 8), 256, smem, st>>>(L, mu_next, nb, Bc, normalise ? 1 : 0);
    } else {
        dim3 grid((L.n_in + 31) / 32, Bc);
        k_linear<<<grid, 256, 0, st>>>(L.weight, L.n_in, L.n_out, 1, L.n_in, mu_next, nb);
    }
    ++*launches;
}

void prop_property_backward(const float* wp, const float* mu_out, float* nb, int nL, int Bc, cudaStream_t st, int64_t* launches) {
    const int64_t total4 = (int64_t)Bc * nL * 16;
    k_property_backward<<<capped_grid((total4 + 255) / 256), 256, 0, st>>>(wp, mu_out, nb, nL, total4);
    ++*launches;
}

void output_node(const GnnParams& g, const float* wp, const float* bp, const float* mu_L, bool mu_image, int mu_stride, const float* lb_out,
                 const float* ub_out, const float* prim_out, float* mu_out, int nL, int Bc, cudaStream_t st, int64_t* launches) {
    k_output_node<<<Bc, 256, 0, st>>>(g, wp, bp, mu_L, mu_image ? 1 : 0, mu_stride, lb_out, ub_out, prim_out, mu_out, nL);
    ++*launches;
}

void masked_argmax(const float* scores, const float* mask, int n_hidden, int Bc, float* best_score, int32_t* best_idx,
                   gnnb_winner* winners, cudaStream_t st, int64_t* launches) {
    k_masked_argmax<<<Bc, 256, 0, st>>>(scores, mask, n_hidden, best_score, best_idx, winners);
    ++*launches;
}

void masked_topk(const float* scores, const float* mask, int n, int Bc, int k, float* top_score, int32_t* top_idx, cudaStream_t st,
                 int64_t* launches) {
    const size_t smem = n <= TOPK_SMEM_KEYS ? (size_t)n * sizeof(uint32_t) : 0;
    k_masked_topk<<<Bc, TOPK_BT, smem, st>>>(scores, mask, n, k, top_score, top_idx);
    ++*launches;
}

void gather_rows(const RowGather* tab, int n_arrays, const int32_t* rows, int n, cudaStream_t st, int64_t* launches) {
    k_gather_rows<<<dim3((unsigned)n, (unsigned)n_arrays), 256, 0, st>>>(tab, rows);
    ++*launches;
}

void scatter_rescored(const int32_t* rows, int n, int k, const float* sub_best, const int32_t* sub_idx, const float* sub_scores,
                      int n_hidden, float* best_score, int32_t* best_idx, gnnb_winner* winners, float* scores, int32_t* flag,
                      cudaStream_t st, int64_t* launches) {
    k_scatter_rescored<<<n, 256, 0, st>>>(rows, k, sub_best, sub_idx, sub_scores, n_hidden, best_score, best_idx, winners, scores, flag);
    ++*launches;
}

}  // namespace gnnb
