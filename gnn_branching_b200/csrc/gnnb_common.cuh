// Internal declarations shared by the libgnnb.so translation units.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/gnnb.h"

namespace gnnb {

constexpr int P = 64;                 // embedding size (GraphNet p; the shipped checkpoint and graph_score.py:9 use 64)

// The 26 nn.Linear modules of the GNN in state_dict order (graph_conv.py:36-74, 431-432).
enum Lin : int {
    INP_F = 0, INP_F_1, INP_B, INP_B_1, INP_B2, INP_B2_2, FC1, FC1_1, FC3, FC3_2, FC4, FC4_2,
    OUT1, OUT2, OUT3, BC1, BC1_1, BC1_2, BC2, BC2_1, BC3, BC3_1, BC4, BC4_1, FNODE, FSCORE, N_LIN
};

// in-features of each linear (out-features are P, except FSCORE = 1)
__host__ __device__ constexpr int lin_in(int l) {
    return l == INP_F ? 3 : l == INP_B ? 2 : (l == FC1 || l == BC1) ? 7 : l == OUT1 ? 4
         : (l == INP_B2 || l == FC3 || l == FC4 || l == OUT2 || l == BC3 || l == BC4) ? 2 * P
         : l == BC2 ? 3 * P : P;
}
__host__ __device__ constexpr int lin_out(int l) { return l == FSCORE ? 1 : P; }

// Composed linears used only by the tensor-core kernels (see gnnb_tc.cu header): products of two reference linears
// with nothing but a bias between them, formed once on the host in double precision.
enum TcLin : int {
    T_FWD_R = 0,   // fc4[:, :64] o fc1_1      bias = fc4[:, :64] b_fc1_1
    T_FWD_C,       // fc4[:, 64:] o fc3_2      bias = b_fc4 + fc4[:, 64:] b_fc3_2
    T_BWD_R,       // bc4[:, :64] o bc2_1
    T_BWD_C,       // bc4[:, 64:] o bc3_1      bias = b_bc4 + bc4[:, 64:] b_bc3_1
    T_INP_C,       // inp_b2[:, :64] o inp_b_1 bias = b_inp_b2 + inp_b2[:, :64] b_inp_b_1
    T_INP_NB,      // inp_b2[:, 64:]           (no bias)
    N_TCLIN
};

// GNN parameters on the device.
//   wt[l]   fp32 [K][64]   transposed weight (wt[k][n] = W[n][k]), SIMT kernels and first layers
//   bias[l] fp32 [64]
//   tc[l]   fp16 hi/lo planes in the UMMA shared-memory layout, one 16 KB block per 64 input features
//           (see gnnb_tc.cu for the layout); only for K >= 64 linears
struct GnnParams {
    const float* wt[N_LIN];
    const float* bias[N_LIN];
    const uint16_t* tc[N_LIN];
    const uint16_t* tcx_w[N_TCLIN];   // composed 64x64 linears, same plane layout as tc[]
    const float* tcx_b[N_TCLIN];      // their biases, fp32 [64]
    int T;
};

// One edge set of the verified network on the device.
struct LayerDev {
    int kind;
    int c_in, h_in, w_in, c_out, h_out, w_out, ksize, stride, pad;
    int n_in, n_out;
    const float* weight;      // as given (conv [co,ci,k,k], linear [out,in])
    const float* bias_node;   // [n_out] bias of the layer expanded per node (graph_conv.py:122-124, 133)
};

// Row order of the tensor-core path's private tensors ("slot order").  The nodes of a layer are grouped into tiles of
// <= 128 nodes that share inputs in the propagation plans (all channels of a spatial patch; 128 consecutive nodes for
// flat layers), each padded to 128 slots; a subdomain owns nslots consecutive rows, global row = b * nslots + slot.
// A propagation tile is therefore exactly one tile of the node kernels, and tiles never straddle subdomains.  The
// caller's arrays stay in the reference's NCHW-flat node order and are reached through node_of_slot.
struct RowMap {
    const int32_t* node_of_slot;   // [nslots] node of each slot, -1 = padding
    int n;                         // nodes per subdomain
    int nslots;                    // slots per subdomain (multiple of 128)
};
// index into a caller array [B, n] of global slot row `grow`, -1 for padding slots
__device__ __forceinline__ int64_t natural_row(const RowMap& m, int64_t grow) {
    const int64_t b = grow / m.nslots;
    const int node = __ldg(m.node_of_slot + (grow - b * m.nslots));
    return node < 0 ? -1 : b * m.n + node;
}
struct LayerTiling {               // host side of a RowMap
    std::vector<int32_t> node_of_slot, slot_of_node;
    int ntiles = 0;
};
LayerTiling make_tiling(int C, int H, int W);      // conv-shaped layer; H = W = 1: flat layer of C nodes

// Per-row (node) inputs of one hidden layer for one chunk of subdomains.  SIMT path: rows = Bc * n in node order;
// tensor-core path: rows = Bc * map.nslots in slot order, the arrays below are reached through `map`.
struct NodeInputs {
    const float* lb;          // [rows]
    const float* ub;          // [rows]
    const float* dual;        // [rows, 3]
    const float* prim_pre;    // [rows]
    const float* prim_post;   // [rows]
    const float* bias_node;   // [n]
    int n;                    // nodes per subdomain in this layer
    int64_t rows;
    // tensor-core path only: the ambiguous rows (beta > 0, the only ones whose relaxation features are non-zero,
    // graph_conv.py:161, 293), compacted in row order by amb_compact()
    const int32_t* amb_rows;  // [amb_base[ntiles]] global row of each compacted slot
    const int32_t* amb_base;  // [ntiles + 1] first slot of each tile of 128 rows; amb_base[ntiles] = number of ambiguous rows
    RowMap map;
};

// Subdomains in which the tensor-core pass of one scoring call met a NaN (option "rescore"), filled by the NaN watch of the
// tensor-core update kernels.  Subdomain numbers are indices into the call's frontier.  flag == null: not recorded.
struct NanDoms {
    int32_t* count;           // [1] entries of `list`
    int32_t* flag;            // [B] 1 once the subdomain is on the list (all 0 between calls)
    int32_t* list;            // [B] flagged subdomains, in the order the kernels found them
    int dom0;                 // first subdomain of the wave being scored
};

// ---- launchers (each enqueues on `st` and bumps *launches) -------------------------------------
// SIMT fp32 node kernels (gnnb_simt.cu)
void simt_relax(const GnnParams& g, const NodeInputs& in, float* relax_f, float* relax_b, cudaStream_t st, int64_t* launches);
void simt_update(const GnnParams& g, bool backward, const float* lb, const float* ub, const float* nb, const float* relax,
                 float* mu_out, float* scores /*or null*/, int n, int64_t score_stride, int64_t score_off, int64_t rows,
                 unsigned long long* nan_count, cudaStream_t st, int64_t* launches);
void simt_input_embed(const GnnParams& g, const float* lb0, const float* x, const float* ub0, float* mu0, int64_t rows,
                      cudaStream_t st, int64_t* launches);
void simt_input_update(const GnnParams& g, const float* lb0, const float* ub0, const float* nb, float* mu0, int64_t rows,
                       cudaStream_t st, int64_t* launches);

int simt_init();  // opt-in shared memory sizes; returns cudaError_t

// tcgen05 node kernels (gnnb_tc.cu) — same contracts as the SIMT ones
// relax' of n_layers <= AMB_MAX_LAYERS hidden layers in one launch (their ambiguous rows compacted by amb_compact_all)
void tc_relax(const GnnParams& g, const NodeInputs* in, float* const* relax_f, float* const* relax_b, int n_layers, cudaStream_t st,
              int64_t* launches);
void tc_update(const GnnParams& g, bool backward, const float* lb, const float* ub, const float* nb, const float* relax,
               const int32_t* amb_base, float* mu_out, float* scores, RowMap map, int64_t score_stride, int64_t score_off, int64_t rows,
               unsigned long long* nan_count, const NanDoms& nan_doms, cudaStream_t st, int64_t* launches);
// propagation (plan) + node update of one layer in ONE launch: the neighbour embeddings go from the propagation accumulator
// to the update chain through tensor memory and are never written (k_tc_fused); nb_dbg: the nb tile images for snapshots, or null;
// input_layer: the chain is the input-layer update (lb / ub = input bounds; backward, relax, amb_base, scores unused)
struct PropPlan;
void tc_fused(const GnnParams& g, const PropPlan* plan, const float* mu_in, bool backward, const float* lb, const float* ub,
              const float* relax, const int32_t* amb_base, float* mu_out, float* scores, RowMap map, int64_t score_stride, int64_t score_off,
              int64_t rows, unsigned long long* nan_count, const NanDoms& nan_doms, float* nb_dbg, bool input_layer, cudaStream_t st,
              int64_t* launches);
// slot of every ambiguous row of a layer, in row order: amb_base[tile] (+ the rank inside the tile), amb_rows[slot] = row;
// cnt is scratch of ntiles + 1 ints (three small launches: count per tile, scan, fill)
void amb_compact(const float* lb, const float* ub, RowMap map, int64_t rows, int32_t* cnt, int32_t* amb_base, int32_t* amb_rows,
                 cudaStream_t st, int64_t* launches);
// the same for up to AMB_MAX_LAYERS hidden layers of a wave in three launches
constexpr int AMB_MAX_LAYERS = 16;
struct AmbLayers {
    const float* lb[AMB_MAX_LAYERS];
    const float* ub[AMB_MAX_LAYERS];
    RowMap map[AMB_MAX_LAYERS];
    int64_t rows[AMB_MAX_LAYERS];
    int32_t* cnt[AMB_MAX_LAYERS];
    int32_t* base[AMB_MAX_LAYERS];
    int32_t* out_rows[AMB_MAX_LAYERS];
    int tile0[AMB_MAX_LAYERS + 1];      // filled by amb_compact_all
    int n;
};
void amb_compact_all(AmbLayers a, cudaStream_t st, int64_t* launches);
void tc_input_embed(const GnnParams& g, const float* lb0, const float* x, const float* ub0, float* mu0, RowMap map, int64_t rows,
                    cudaStream_t st, int64_t* launches);
void tc_input_update(const GnnParams& g, const float* lb0, const float* ub0, const float* nb, float* mu0, RowMap map, int64_t rows,
                     cudaStream_t st, int64_t* launches);
// repack one nn.Linear weight [64][K] (host) into the tensor-core plane layout; returns elements written
int64_t tc_pack_weight(const float* w_host, int K, uint16_t* dst_host);
int64_t tc_packed_elems(int K);
int tc_init();   // opt-in shared memory sizes; returns cudaError_t
bool tc_available();
// tile image (gnnb_umma.cuh: mu = swizzled, nb = piece-major) -> fp32 [rows][64]; debugging snapshots
void tc_unpack_tile_image(const float* img, float* out, RowMap map, int64_t rows, bool piece_major, cudaStream_t st);   // out: node order

// propagation through the verified network and the small kernels (gnnb_prop.cu)
int prop_init(int max_smem_bytes);
void prop_forward(const LayerDev& L, const float* mu_prev, float* nb, int Bc, cudaStream_t st, int64_t* launches);
void prop_backward(const LayerDev& L, const float* mu_next, float* nb, int Bc, bool normalise, cudaStream_t st, int64_t* launches);
void prop_property_backward(const float* wp, const float* mu_out, float* nb, int nL, int Bc, cudaStream_t st, int64_t* launches);
void output_node(const GnnParams& g, const float* wp, const float* bp, const float* mu_L, bool mu_image, int mu_stride, const float* lb_out,
                 const float* ub_out, const float* prim_out, float* mu_out, int nL, int Bc, cudaStream_t st, int64_t* launches);
// best_score / best_idx (both or neither) and / or packed winner records
void masked_argmax(const float* scores, const float* mask, int n_hidden, int Bc, float* best_score, int32_t* best_idx,
                   gnnb_winner* winners, cudaStream_t st, int64_t* launches);
// the k best candidates of every row of scores [Bc, n] (mask [Bc, n] or null = all), 1 <= k <= GNNB_TOPK_MAX, in the order of
// masked_argmax extended to k (NaN first, then descending, ties by ascending index); top_score / top_idx [Bc, k]
void masked_topk(const float* scores, const float* mask, int n, int Bc, int k, float* top_score, int32_t* top_idx, cudaStream_t st,
                 int64_t* launches);
// re-score pass of option "rescore": one launch copies row rows[i] of every array of `tab` (floats per row = per) to row i of
// its destination, i < n; the second writes the results of those n rows back to rows rows[i] of the call's outputs (k best
// scores / indices per row or winner records, and the dense score rows when `scores` is not null) and clears their flags
struct RowGather { const float* src; float* dst; int64_t per; };
// The arrays of a batch of subdomains the GNN reads, device pointers, node order: every field of gnnb_frontier but `mask`
// (run_chunk of gnnb_api.cu, train_backward of gnnb_train.cu).  walk_inputs (gnnb_api.cu) lists them in one fixed order.
struct GnnInputs {
    std::vector<const float*> lb, ub;            // L + 2 arrays [B, n_k]
    std::vector<const float*> dual, pre, post;   // L arrays [B, n_k, 3] / [B, n_k] / [B, n_k], hidden layer k = 1..L
    const float *pout = nullptr, *pin = nullptr, *wp = nullptr, *bp = nullptr;
    explicit GnnInputs(int L) : lb(L + 2), ub(L + 2), dual(L), pre(L), post(L) {}
};
void gather_rows(const RowGather* tab, int n_arrays, const int32_t* rows, int n, cudaStream_t st, int64_t* launches);
void scatter_rescored(const int32_t* rows, int n, int k, const float* sub_best, const int32_t* sub_idx, const float* sub_scores,
                      int n_hidden, float* best_score, int32_t* best_idx, gnnb_winner* winners, float* scores, int32_t* flag,
                      cudaStream_t st, int64_t* launches);

// tensor-core propagation (gnnb_prop_tc.cu): block plans built once per network, gather-GEMM kernel
struct PropPlan;
int prop_tc_init();
PropPlan* prop_plan_build(const LayerDev& L, const float* host_weight, bool backward, bool normalise, const LayerTiling& out,
                          const LayerTiling& in);
void prop_plan_free(PropPlan* p);
double prop_plan_density(const PropPlan* p);
void prop_tc_run(const PropPlan* plan, const float* mu_in, float* nb_img, int Bc, cudaStream_t st, int64_t* launches);
void prop_tc_property_backward(const float* wp, const float* mu_out, float* nb_img, int nL, int nslots, int Bc, cudaStream_t st, int64_t* launches);

// BaBSR / KW heuristic (gnnb_babsr.cu); every pointer is a device pointer; returns -1 when the network does not fit
int babsr_max_layers();
int babsr_run(const LayerDev* d_layers, int L, int n_hidden, int nmax, const float* const* d_lb, const float* const* d_ub,
              const float* wp, const float* mask, const int32_t* d_hidden_off, const int32_t* d_random_order,
              const int32_t* counter_in, int sparsest_layer, float threshold, int32_t* decision, int32_t* counter_out,
              int32_t* kind, float* scores, int B, cudaStream_t st, int64_t* launches);

// device-resident domain queue (gnnb_queue.cu); every data pointer is a device pointer
struct DomainQueue;
int queue_create(int device, const std::vector<int>& n, int n_hidden, int64_t capacity, DomainQueue** out, std::string* err);
void queue_destroy(DomainQueue* q);
const std::string& queue_error(const DomainQueue* q);
int64_t queue_size(const DomainQueue* q);
int64_t queue_capacity(const DomainQueue* q);
int queue_global_lb(DomainQueue* q, float* out, cudaStream_t st);
int queue_add(DomainQueue* q, int B, const float* lower, const float* upper, const float* const* lb, const float* const* ub,
              const int8_t* mask, const int32_t* decision, const uint8_t* keep, int32_t* added, cudaStream_t st, int64_t* launches);
int queue_pick(DomainQueue* q, int max_B, float threshold, bool discard, int32_t* picked, float* lower, float* upper, float* const* lb,
               float* const* ub, int8_t* mask, int32_t* decision, cudaStream_t st, int64_t* launches);
int queue_prune(DomainQueue* q, float threshold, cudaStream_t st, int64_t* launches);
float* queue_stage(DomainQueue* q, size_t bytes);

// batched KW intermediate bounds (gnnb_kw.cu); every pointer is a device pointer.  KwTc (or null): the dense layers' column
// blocks go through the tensor-core propagation kernel — plans[j] = un-normalised transposed plan of layer j + 1 -> j, maps[k] =
// slot order of layer k
struct KwTc { const std::vector<PropPlan*>* plans; const std::vector<RowMap>* maps; };
int kw_init();   // opt-in shared memory size of the cone kernel on the current device; returns cudaError_t
int kw_bounds(const std::vector<LayerDev>& layers, const std::vector<int>& n, int B, const float* x, float eps, const float* wp, const float* bp,
              const float* const* prov_lb, const float* const* prov_ub, float* const* out_lb, float* const* out_ub, const KwTc* tc, float** ws,
              size_t* ws_cap, cudaStream_t st, int64_t* launches, std::string* err);
// bounds part of update_the_model for B children (KW pass with the split, interval pass, second KW pass where needed); iscratch:
// 3 B + 1 int32 of device scratch; synchronises `st` once
int child_bounds(const std::vector<LayerDev>& layers, const std::vector<int>& n, int B, const float* x, float eps, const float* wp, const float* bp,
                 const float* const* parent_lb, const float* const* parent_ub, const int32_t* dec_layer, const int32_t* dec_index,
                 const int32_t* choice, float* const* out_lb, float* const* out_ub, int8_t* const* out_mask, int32_t* second_pass,
                 int32_t* iscratch, const KwTc* tc, float** ws, size_t* ws_cap, cudaStream_t st, int64_t* launches, std::string* err);

// bounds part of build_the_model for B root domains (KW bounds, interval pass from the input box, KW pass where a hidden layer moved)
int root_bounds(const std::vector<LayerDev>& layers, const std::vector<int>& n, int B, const float* x, float eps, const float* wp, const float* bp,
                float* const* out_lb, float* const* out_ub, int8_t* const* out_mask, int32_t* second_pass, int32_t* iscratch, const KwTc* tc,
                float** ws, size_t* ws_cap, cudaStream_t st, int64_t* launches, std::string* err);

// ---- device helpers ---------------------------------------------------------------------------
// compute_ratio of graph_conv.py:499-514 in the reference's operation order (IEEE division, no fast-math)
struct Ratio { float r0, r1, beta, amb; };
__device__ __forceinline__ Ratio compute_ratio(float l, float u) {
    Ratio r;
    float lt = l - fmaxf(l, 0.0f);          // lower - relu(lower)
    float ut = fmaxf(u, 0.0f);
    if (u != u) ut = u;                     // F.relu propagates NaN, fmaxf does not
    if (l != l) lt = l;
    r.r0 = __fdiv_rn(ut, __fsub_rn(ut, lt));
    r.beta = __fmul_rn(__fmul_rn(-1.0f, lt), r.r0);
    r.amb = (r.beta > 0.0f) ? 1.0f : 0.0f;
    r.r1 = __fadd_rn(__fmul_rn(__fsub_rn(1.0f, __fmul_rn(2.0f, __fmul_rn(r.r0, r.amb))), r.amb), r.r0);
    return r;
}

}  // namespace gnnb
