// C ABI of libgnnb.so (include/gnnb.h): context, parameter packing, workspace, and the per-chunk stage schedule.
//
// HBM layout per chunk of Bc subdomains (node-major, 256 bytes of 64 channels per node = global row b * n_k + node):
//   mu[k]      [Bc, n_k, 64]  k = 0 (input pixels) .. L (hidden) .. L+1 (output node)   init_mu, graph_conv.py:487-496
//   nb         [Bc, max_k n_k, 64]   neighbour embeddings of the layer being updated (reused by every stage)
//   relax_f[k], relax_b[k]  [Bc, n_k, 64]  round-independent relaxation features (see gnnb_simt.cu header)
//   scores     [Bc, sum n_k]
// SIMT mode keeps them as plain fp32 rows; the tensor-core mode keeps mu[0..L] and nb as fp16 hi/lo tile images of 128
// rows (32 KB per tile, same 256 bytes per node; formats in gnnb_umma.cuh) and relax' tile-transposed (gnnb_tc.cu).
// Only adjacent layers are live at any time, so a chunk's stage working set is ~3 * Bc * n_k * 256 B.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "gnnb_common.cuh"
#include "gnnb_train.cuh"

using namespace gnnb;

struct gnnb_ctx {
    int device = 0;
    int last_status = 0;
    std::string err;
    int64_t launches = 0;
    // options
    int math = GNNB_MATH_TC_FP16X3;
    int chunk = 0;
    int snapshot = 0;
    int fuse = 1;                   // propagation + node update of a layer in one launch, nb handed over in tensor memory (k_tc_fused); 0 = two launches
    int rescore = 0;                // score the subdomains whose tensor-core pass met a NaN again in exact fp32 (rescore_flagged)
    int64_t rescored = 0;           // subdomains the last scoring call scored again
    // GNN parameters
    bool have_gnn = false;
    float* d_gnn = nullptr;
    uint16_t* d_tc = nullptr;
    GnnParams gp{};
    // online fine-tuning (gnnb_train.cu): master parameters in nn.Linear layout, gradients and Adam moments, one block of
    // 4 * n_params floats [master | grad | exp_avg | exp_avg_sq]; offsets of weight / bias of each linear inside a quarter
    float* d_train = nullptr;
    int64_t n_params = 0;
    size_t po_w[N_LIN] = {0}, po_b[N_LIN] = {0};
    int adam_steps = 0;
    float* train_ws = nullptr;      // gnnb_score_grad(_device): tape of a wave, staged input rows, gather table (grow-only)
    size_t train_ws_cap = 0;
    int grad_chunk = 0;             // subdomains per wave of the gradient pass; 0 = the most whose tape fits GRAD_TAPE_BYTES
    int grad_ws_domains = 0;        // subdomains per wave of the last gradient call
    int64_t grad_bad_terms = 0;     // out-of-range terms of the last gradient call
    float* kw_ws = nullptr;         // column buffers of gnnb_kw_bounds (grow-only)
    size_t kw_ws_cap = 0;
    int32_t* kw_iscratch = nullptr; // per-domain flags of gnnb_child_bounds, named subdomains of gnnb_score_grad_device (grow-only)
    int kw_iscratch_cap = 0;
    // verified network
    bool have_net = false;
    float* d_net = nullptr;
    std::vector<LayerDev> layers;
    std::vector<PropPlan*> plan_fwd, plan_bwd;   // tensor-core propagation plans per layer
    std::vector<PropPlan*> plan_kw_own;          // un-normalised transposed plans of the conv layers k > 0 (bound producer), else null
    std::vector<PropPlan*> plan_kw;              // per layer: plan_kw_own[k] or plan_bwd[k] (already un-normalised: layer 0, linear layers)
    std::vector<int> n;             // n[0] = input nodes, n[1..L] hidden, n[L+1] = 1
    int zero_tap_layer = 0;         // first conv layer j >= 2 (1-based) with an input position no tap reaches, else 0
    // slot order of the tensor-core path (gnnb_common.cuh): tiling and device map of layers 0..L
    std::vector<LayerTiling> tiling;
    std::vector<RowMap> rowmap;
    int32_t* d_maps = nullptr;
    // BaBSR heuristic: device copies of the layer table, hidden offsets, preference order and the per-call pointer tables
    LayerDev* d_layers = nullptr;
    int32_t* d_hidden_off = nullptr;
    int32_t* d_random_order = nullptr;
    const float** d_ptrs = nullptr;   // [2 * (L + 2)] lb pointers then ub pointers
    std::vector<int> hidden_off;    // offset of layer k (1-based) in the flat ReLU index
    int n_hidden = 0;
    std::vector<struct gnnb_queue*> queues;      // live gnnb_queue objects: they were sized for the current network
    // workspace
    int ws_cap = 0;                 // subdomains the workspace can hold
    bool ws_host_staging = false;
    float* d_ws = nullptr;
    std::vector<float*> mu, relax_f, relax_b;
    std::vector<int32_t*> amb_cnt, amb_base, amb_rows;   // compaction of the ambiguous rows of each hidden layer (tensor-core path)
    float* nb = nullptr;
    float* ws_scores = nullptr;
    float* ws_best = nullptr;
    int32_t* ws_idx = nullptr;
    // staged copies of host inputs: two sets, so that the copies of the next chunk (copy stream) overlap the kernels of
    // the current one (caller's stream)
    struct Staging {
        std::vector<float*> inputs;  // the GNN's input arrays of a wave, in the order of walk_inputs
        float* mask = nullptr;
        float* best = nullptr;
        int32_t* idx = nullptr;
        float* scores = nullptr;
    } stg[2];
    float* res_best = nullptr;      // winners of a whole host-buffer call (one device->host copy at the end, so that a
    int32_t* res_idx = nullptr;     // pageable result buffer cannot stall the wave pipeline)
    int64_t res_cap = 0;            // entries (subdomains x k)
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr};
    unsigned long long* d_nan = nullptr;
    // option "rescore": NanDoms of a call, [count | flags [resc_cap] | list [resc_cap]] (grow-only; count and flags are 0 between
    // calls), and the gather table of the re-score pass (grow-only)
    int32_t* d_resc = nullptr;
    int resc_cap = 0;
    RowGather* d_gather = nullptr;
    size_t gather_cap = 0;
    // debugging snapshots
    std::map<std::string, std::pair<float*, int64_t>> snaps;
    // per-kernel-class device timing (option "profile")
    int profile = 0;
    struct Pending { int klass; int64_t rows; cudaEvent_t a, b; };
    std::vector<Pending> pending;
    std::vector<cudaEvent_t> ev_pool;
    double prof_ms[GNNB_K_COUNT] = {0};
    int64_t prof_launches[GNNB_K_COUNT] = {0};
    int64_t prof_rows[GNNB_K_COUNT] = {0};
};

struct gnnb_queue {
    gnnb_ctx* ctx;                  // null once the context has been destroyed (the queue's own device memory stays valid)
    DomainQueue* q;
};

namespace {

int fail(gnnb_ctx* c, int status, const std::string& msg) {
    if (c) { c->last_status = status; c->err = msg; }
    return status;
}

// taps of conv_transpose2d along one axis that reach input position i (the per-axis count of k_div_freq)
int axis_taps(int i, int ksize, int stride, int pad, int n_out) {
    int t = 0;
    for (int k = 0; k < ksize; ++k) {
        const int a = i + pad - k;
        if (a >= 0 && a % stride == 0 && a / stride < n_out) ++t;
    }
    return t;
}

// First conv layer j >= 2 (1-based) with an input position that no tap of conv_transpose2d reaches (stride > kernel), else 0.
// The GNN's backward propagation divides such a position by freq = 0 (graph_conv.py:306-312): 0/0 in the reference.  Layer 1's
// transpose feeds the input nodes and is not normalised, so it may have such positions.
int first_zero_tap_layer(const std::vector<LayerDev>& layers) {
    for (size_t k = 1; k < layers.size(); ++k) {
        const LayerDev& L = layers[k];
        if (L.kind != GNNB_LAYER_CONV) continue;
        for (int y = 0; y < L.h_in; ++y)
            if (axis_taps(y, L.ksize, L.stride, L.pad, L.h_out) == 0) return (int)k + 1;
        for (int x = 0; x < L.w_in; ++x)
            if (axis_taps(x, L.ksize, L.stride, L.pad, L.w_out) == 0) return (int)k + 1;
    }
    return 0;
}

// the GNN scoring entries (score, winners, top-k, score_grad) refuse a network whose normalisation divides by zero
int check_zero_taps(gnnb_ctx* c) {
    if (!c->zero_tap_layer) return GNNB_OK;
    return fail(c, GNNB_ERR_UNSUPPORTED, "layer " + std::to_string(c->zero_tap_layer) +
                " (conv, stride > kernel) has input positions no tap reaches: the GNN's tap-count normalisation divides by zero");
}

// The arrays of a frontier the GNN reads, in one fixed order: lb[k] and ub[k] for k = 0 .. L + 1, then dual, prim_pre and
// prim_post of each hidden layer, then prim_out, primal_input, wp and bp.  Calls f(src, slot, per) for each: src = the
// frontier's array (null also when its per-layer table is null), slot = the matching pointer of `in`, per = floats per subdomain.
// Staging, gathering, copying and checking a frontier all go through this walk, and the staging sets are laid out in its order.
template <class F>
void walk_inputs(const gnnb_frontier& fr, GnnInputs& in, const std::vector<int>& n, F f) {
    const int L = (int)n.size() - 2;
    auto at = [](const float* const* table, int k) { return table ? table[k] : nullptr; };
    for (int k = 0; k <= L + 1; ++k) {
        f(at(fr.lb, k), in.lb[k], (int64_t)n[k]);
        f(at(fr.ub, k), in.ub[k], (int64_t)n[k]);
    }
    for (int k = 0; k < L; ++k) {
        f(at(fr.dual, k), in.dual[k], (int64_t)n[k + 1] * 3);
        f(at(fr.prim_pre, k), in.pre[k], (int64_t)n[k + 1]);
        f(at(fr.prim_post, k), in.post[k], (int64_t)n[k + 1]);
    }
    f(fr.prim_out, in.pout, (int64_t)1);
    f(fr.primal_input, in.pin, (int64_t)n[0]);
    f(fr.wp, in.wp, (int64_t)n[L]);
    f(fr.bp, in.bp, (int64_t)1);
}

// *out = the frontier's arrays the GNN reads; GNNB_ERR_INVALID when one of them, or the mask when `mask`, is null.  Called before
// anything is enqueued, so that an error return never leaves copies in flight.
int frontier_inputs(gnnb_ctx* ctx, const gnnb_frontier* fr, bool mask, GnnInputs* out) {
    bool ok = !mask || fr->mask;
    walk_inputs(*fr, *out, ctx->n, [&](const float* src, const float*& slot, int64_t) { slot = src; ok = ok && src; });
    return ok ? GNNB_OK : fail(ctx, GNNB_ERR_INVALID, "null frontier array");
}

#define CU(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e__ = (call);                                                                         \
        if (e__ != cudaSuccess)                                                                           \
            return fail(ctx, GNNB_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));         \
    } while (0)

size_t align4(size_t x) { return (x + 3) & ~size_t(3); }

void free_workspace(gnnb_ctx* c) {
    if (c->d_ws) cudaFree(c->d_ws);
    c->d_ws = nullptr;
    c->ws_cap = 0;
    for (auto& kv : c->snaps) cudaFree(kv.second.first);
    c->snaps.clear();
}

int ensure_workspace(gnnb_ctx* ctx, int Bc, bool host_staging) {
    if (ctx->d_ws && ctx->ws_cap >= Bc && (ctx->ws_host_staging || !host_staging)) return GNNB_OK;
    free_workspace(ctx);
    const int L = (int)ctx->layers.size();
    int nmax = 0;
    for (int k = 0; k <= L; ++k) nmax = ctx->n[k] > nmax ? ctx->n[k] : nmax;
    size_t total = 0;
    auto take = [&](size_t elems) { size_t off = total; total += (elems + 63) & ~size_t(63); return off; };      // 256-byte aligned (32-byte sector stores, bulk copies)
    std::vector<size_t> o_mu(L + 2), o_rf(L + 1), o_rb(L + 1), o_lb(L + 2), o_ub(L + 2), o_du(L), o_pr(L), o_po(L);
    // mu, nb and relax' are stored per tile of 128 rows by the tensor-core kernels: round the row counts up
    // rows of a layer in the workspace: slots (multiple of 128 per subdomain) >= nodes, so the SIMT path's node-order rows fit too
    auto wrows = [&](int k) { return (size_t)Bc * (k <= L ? (size_t)ctx->rowmap[k].nslots : 128); };
    for (int k = 0; k <= L + 1; ++k) o_mu[k] = take(wrows(k) * P);
    for (int k = 1; k <= L; ++k) { o_rf[k] = take(wrows(k) * P); o_rb[k] = take(wrows(k) * P); }
    std::vector<size_t> o_ac(L + 1), o_ab(L + 1), o_ar(L + 1);
    for (int k = 1; k <= L; ++k) {
        const size_t rows = wrows(k), nt = rows / 128;
        o_ac[k] = take(nt + 1); o_ab[k] = take(nt + 1); o_ar[k] = take(rows);
    }
    size_t nb_rows = 0;
    for (int k = 0; k <= L; ++k) nb_rows = wrows(k) > nb_rows ? wrows(k) : nb_rows;
    const size_t o_nb = take(nb_rows * P);
    const size_t o_sc = take((size_t)Bc * ctx->n_hidden);
    const size_t o_best = take(Bc), o_idx = take(Bc);
    struct StgOff { std::vector<size_t> inputs; size_t mask, best, idx, sc; } so[2];
    if (host_staging) {
        GnnInputs unused(L);
        for (StgOff& o : so) {
            walk_inputs(gnnb_frontier{}, unused, ctx->n, [&](const float*, const float*&, int64_t per) {
                o.inputs.push_back(take((size_t)Bc * per));
            });
            o.mask = take((size_t)Bc * ctx->n_hidden);
            o.best = take((size_t)Bc * GNNB_TOPK_MAX); o.idx = take((size_t)Bc * GNNB_TOPK_MAX);   // k results per row (re-score pass)
            o.sc = take((size_t)Bc * ctx->n_hidden);
        }
    }
    CU(cudaMalloc(&ctx->d_ws, total * sizeof(float)));
    float* base = ctx->d_ws;
    ctx->mu.assign(L + 2, nullptr); ctx->relax_f.assign(L + 1, nullptr); ctx->relax_b.assign(L + 1, nullptr);
    for (int k = 0; k <= L + 1; ++k) ctx->mu[k] = base + o_mu[k];
    for (int k = 1; k <= L; ++k) { ctx->relax_f[k] = base + o_rf[k]; ctx->relax_b[k] = base + o_rb[k]; }
    ctx->amb_cnt.assign(L + 1, nullptr); ctx->amb_base.assign(L + 1, nullptr); ctx->amb_rows.assign(L + 1, nullptr);
    for (int k = 1; k <= L; ++k) {
        ctx->amb_cnt[k] = reinterpret_cast<int32_t*>(base + o_ac[k]);
        ctx->amb_base[k] = reinterpret_cast<int32_t*>(base + o_ab[k]);
        ctx->amb_rows[k] = reinterpret_cast<int32_t*>(base + o_ar[k]);
    }
    ctx->nb = base + o_nb; ctx->ws_scores = base + o_sc; ctx->ws_best = base + o_best;
    ctx->ws_idx = reinterpret_cast<int32_t*>(base + o_idx);
    if (host_staging) {
        for (int i = 0; i < 2; ++i) {
            gnnb_ctx::Staging& g = ctx->stg[i];
            const StgOff& o = so[i];
            g.inputs.clear();
            for (size_t off : o.inputs) g.inputs.push_back(base + off);
            g.mask = base + o.mask;
            g.best = base + o.best; g.idx = reinterpret_cast<int32_t*>(base + o.idx); g.scores = base + o.sc;
        }
        if (!ctx->copy_stream) {
            CU(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
            for (int i = 0; i < 2; ++i) {
                CU(cudaEventCreateWithFlags(&ctx->ev_copied[i], cudaEventDisableTiming));
                CU(cudaEventCreateWithFlags(&ctx->ev_free[i], cudaEventDisableTiming));
            }
        }
    }
    ctx->ws_cap = Bc;
    ctx->ws_host_staging = host_staging;
    return GNNB_OK;
}

#define TRY_(expr) do { int s__ = (expr); if (s__ != GNNB_OK) return s__; } while (0)

int snap(gnnb_ctx* ctx, bool on, const std::string& name, const float* src, int64_t numel, cudaStream_t st) {
    if (!on) return GNNB_OK;
    auto it = ctx->snaps.find(name);
    if (it == ctx->snaps.end() || it->second.second < numel) {
        if (it != ctx->snaps.end()) cudaFree(it->second.first);
        float* p = nullptr;
        CU(cudaMalloc(&p, (size_t)numel * sizeof(float)));
        ctx->snaps[name] = std::make_pair(p, numel);
        it = ctx->snaps.find(name);
    }
    it->second.second = numel;
    CU(cudaMemcpyAsync(it->second.first, src, (size_t)numel * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return GNNB_OK;
}

cudaEvent_t prof_event(gnnb_ctx* ctx) {
    if (!ctx->ev_pool.empty()) { cudaEvent_t e = ctx->ev_pool.back(); ctx->ev_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
}

// brackets one stage launch with events on its stream
struct ProfScope {
    gnnb_ctx* ctx; cudaStream_t st; cudaEvent_t a = nullptr, b = nullptr; int klass; int64_t rows;
    ProfScope(gnnb_ctx* c, int k, int64_t r, cudaStream_t s) : ctx(c), st(s), klass(k), rows(r) {
        if (ctx->profile) { a = prof_event(ctx); b = prof_event(ctx); cudaEventRecord(a, st); }
    }
    ~ProfScope() {
        if (ctx->profile) { cudaEventRecord(b, st); ctx->pending.push_back({klass, rows, a, b}); }
    }
};

int prof_collect(gnnb_ctx* ctx) {
    if (ctx->pending.empty()) return GNNB_OK;
    CU(cudaDeviceSynchronize());
    for (auto& p : ctx->pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
            ctx->prof_ms[p.klass] += ms;
            ctx->prof_launches[p.klass] += 1;
            ctx->prof_rows[p.klass] += p.rows;
        }
        ctx->ev_pool.push_back(p.a);
        ctx->ev_pool.push_back(p.b);
    }
    ctx->pending.clear();
    return GNNB_OK;
}

// mu and nb are fp16 tile images in tensor-core mode (mu swizzled, nb piece-major): unpack them into the snapshot
int snap_img(gnnb_ctx* ctx, bool on, const std::string& name, const float* img, int k, int Bc, bool piece_major, cudaStream_t st) {
    if (!on) return GNNB_OK;
    const int64_t numel = (int64_t)Bc * ctx->n[k] * P;                     // snapshots are in node order in both modes
    if (ctx->math != GNNB_MATH_TC_FP16X3) return snap(ctx, on, name, img, numel, st);
    TRY_(snap(ctx, on, name, img, numel, st));      // allocates / sizes the snapshot buffer
    tc_unpack_tile_image(img, ctx->snaps[name].first, ctx->rowmap[k], (int64_t)Bc * ctx->rowmap[k].nslots, piece_major, st);
    return GNNB_OK;
}

#define TRY(expr) do { int s__ = (expr); if (s__ != GNNB_OK) return s__; } while (0)

// the stage schedule for one chunk in arithmetic `math`; every pointer is a device pointer; nd: where the tensor-core NaN watch
// records the subdomains it flags (nd.flag = null: nowhere); best_score / best_idx: [Bc, k], the k best candidates per subdomain
int run_chunk(gnnb_ctx* ctx, const GnnInputs& in, const float* mask, int Bc, int math, const NanDoms& nd, float* scores, int k,
              float* best_score, int32_t* best_idx, gnnb_winner* winners, cudaStream_t st) {
    const int L = (int)ctx->layers.size();
    const GnnParams& g = ctx->gp;
    const bool tc = math == GNNB_MATH_TC_FP16X3;
    const bool snaps = ctx->snapshot && math == ctx->math;        // an fp32 re-score pass leaves the tensor-core pass's snapshots
    int64_t* lc = &ctx->launches;
    auto name = [](const char* fmt, int a, int b) { char buf[64]; snprintf(buf, sizeof buf, fmt, a, b); return std::string(buf); };

    // rows of layer k in the mode's row order: slots (tensor-core path) or nodes (SIMT path)
    auto R = [&](int k) { return (int64_t)Bc * (tc ? ctx->rowmap[k].nslots : ctx->n[k]); };
    const RowMap nomap{nullptr, 0, 0};
    auto M = [&](int k) { return tc ? ctx->rowmap[k] : nomap; };
    const bool fused = tc && ctx->fuse;

    // ambiguous rows of every hidden layer, compacted (three launches for the wave)
    const bool amb_all = tc && L <= AMB_MAX_LAYERS;
    if (amb_all) {
        ProfScope ps(ctx, GNNB_K_RELAX, 0, st);
        AmbLayers al{};
        al.n = L;
        for (int k = 1; k <= L; ++k) {
            al.lb[k - 1] = in.lb[k]; al.ub[k - 1] = in.ub[k]; al.map[k - 1] = M(k); al.rows[k - 1] = R(k);
            al.cnt[k - 1] = ctx->amb_cnt[k]; al.base[k - 1] = ctx->amb_base[k]; al.out_rows[k - 1] = ctx->amb_rows[k];
        }
        amb_compact_all(al, st, lc);
    }
    // round-independent relaxation features of every hidden layer (tensor-core path: one launch per AMB_MAX_LAYERS layers)
    {
        std::vector<NodeInputs> nis(L + 1);
        for (int k = 1; k <= L; ++k)
            nis[k] = NodeInputs{in.lb[k], in.ub[k], in.dual[k - 1], in.pre[k - 1], in.post[k - 1], ctx->layers[k - 1].bias_node,
                                ctx->n[k], R(k), ctx->amb_rows[k], ctx->amb_base[k], M(k)};
        if (tc) {
            for (int k0 = 1; k0 <= L; k0 += AMB_MAX_LAYERS) {
                const int nl = (L - k0 + 1) < AMB_MAX_LAYERS ? (L - k0 + 1) : AMB_MAX_LAYERS;
                int64_t nodes = 0;
                for (int k = k0; k < k0 + nl; ++k) {
                    nodes += (int64_t)Bc * ctx->n[k];
                    if (!amb_all) amb_compact(in.lb[k], in.ub[k], M(k), nis[k].rows, ctx->amb_cnt[k], ctx->amb_base[k], ctx->amb_rows[k], st, lc);
                }
                ProfScope ps(ctx, GNNB_K_RELAX, nodes, st);
                tc_relax(g, &nis[k0], &ctx->relax_f[k0], &ctx->relax_b[k0], nl, st, lc);
            }
        }
        for (int k = 1; k <= L; ++k) {
            if (!tc) {
                ProfScope ps(ctx, GNNB_K_RELAX, (int64_t)Bc * ctx->n[k], st);
                simt_relax(g, nis[k], ctx->relax_f[k], ctx->relax_b[k], st, lc);
            }
            // tensor-core mode stores relax' (pre-multiplied by fc4 / bc4's relax half, compacted, tile-transposed): not comparable 1:1
            TRY(snap(ctx, snaps, name(tc ? "relaxp_f%d" : "relax_f%d", k, 0), ctx->relax_f[k], (int64_t)Bc * ctx->n[k] * P, st));
            TRY(snap(ctx, snaps, name(tc ? "relaxp_b%d" : "relax_b%d", k, 0), ctx->relax_b[k], (int64_t)Bc * ctx->n[k] * P, st));
        }
    }
    {
        ProfScope ps(ctx, GNNB_K_INPUT_EMBED, (int64_t)Bc * ctx->n[0], st);
        if (tc) tc_input_embed(g, in.lb[0], in.pin, in.ub[0], ctx->mu[0], M(0), R(0), st, lc);
        else simt_input_embed(g, in.lb[0], in.pin, in.ub[0], ctx->mu[0], R(0), st, lc);
    }
    TRY(snap_img(ctx, snaps, "mu0_embed", ctx->mu[0], 0, Bc, false, st));

    for (int t = 0; t < g.T; ++t) {
        const bool last = (t == g.T - 1);
        // forward sweep
        for (int k = 1; k <= L; ++k) {
            const int64_t rows = R(k), nodes = (int64_t)Bc * ctx->n[k];
            if (fused) {
                ProfScope ps(ctx, GNNB_K_LAYER_FWD, nodes, st);
                tc_fused(g, ctx->plan_fwd[k - 1], ctx->mu[k - 1], false, in.lb[k], in.ub[k], ctx->relax_f[k], ctx->amb_base[k],
                         ctx->mu[k], nullptr, M(k), 0, 0, rows, ctx->d_nan, nd, ctx->snapshot ? ctx->nb : nullptr, false, st, lc);
            } else {
                ProfScope ps(ctx, GNNB_K_PROP_FWD, nodes, st);
                if (tc) prop_tc_run(ctx->plan_fwd[k - 1], ctx->mu[k - 1], ctx->nb, Bc, st, lc);
                else prop_forward(ctx->layers[k - 1], ctx->mu[k - 1], ctx->nb, Bc, st, lc);
            }
            TRY(snap_img(ctx, snaps, name("t%d_fwd_nb%d", t, k), ctx->nb, k, Bc, true, st));
            if (!fused) {
                ProfScope ps(ctx, GNNB_K_UPDATE_FWD, nodes, st);
                if (tc) tc_update(g, false, in.lb[k], in.ub[k], ctx->nb, ctx->relax_f[k], ctx->amb_base[k], ctx->mu[k], nullptr, M(k), 0, 0, rows, ctx->d_nan, nd, st, lc);
                else simt_update(g, false, in.lb[k], in.ub[k], ctx->nb, ctx->relax_f[k], ctx->mu[k], nullptr, ctx->n[k], 0, 0, rows, ctx->d_nan, st, lc);
            }
            TRY(snap_img(ctx, snaps, name("t%d_fwd_mu%d", t, k), ctx->mu[k], k, Bc, false, st));
        }
        {
            ProfScope ps(ctx, GNNB_K_OUTPUT, Bc, st);
            output_node(g, in.wp, in.bp, ctx->mu[L], tc, tc ? ctx->rowmap[L].nslots : ctx->n[L], in.lb[L + 1], in.ub[L + 1], in.pout,
                        ctx->mu[L + 1], ctx->n[L], Bc, st, lc);
        }
        TRY(snap(ctx, snaps, name("t%d_mu_out", t, 0), ctx->mu[L + 1], (int64_t)Bc * P, st));
        // backward sweep
        for (int k = L; k >= 1; --k) {
            const int64_t rows = R(k), nodes = (int64_t)Bc * ctx->n[k];
            float* sc = last ? scores : nullptr;
            // the last sweep's embeddings of the first hidden layer feed only the (dead) last input-layer update: not stored
            float* mu_k = (last && k == 1 && tc && !ctx->snapshot) ? nullptr : ctx->mu[k];
            const bool fused_k = fused && k < L;           // the property layer's rank-1 back-propagation is a separate small kernel
            if (fused_k) {
                ProfScope ps(ctx, last ? GNNB_K_LAYER_BWD_SCORE : GNNB_K_LAYER_BWD, nodes, st);
                tc_fused(g, ctx->plan_bwd[k], ctx->mu[k + 1], true, in.lb[k], in.ub[k], ctx->relax_b[k], ctx->amb_base[k],
                         mu_k, sc, M(k), ctx->n_hidden, ctx->hidden_off[k], rows, ctx->d_nan, nd, ctx->snapshot ? ctx->nb : nullptr, false, st, lc);
            } else {
                ProfScope ps(ctx, GNNB_K_PROP_BWD, nodes, st);
                if (k == L && tc) prop_tc_property_backward(in.wp, ctx->mu[L + 1], ctx->nb, ctx->n[L], ctx->rowmap[L].nslots, Bc, st, lc);
                else if (k == L) prop_property_backward(in.wp, ctx->mu[L + 1], ctx->nb, ctx->n[L], Bc, st, lc);
                else if (tc) prop_tc_run(ctx->plan_bwd[k], ctx->mu[k + 1], ctx->nb, Bc, st, lc);
                else prop_backward(ctx->layers[k], ctx->mu[k + 1], ctx->nb, Bc, true, st, lc);
            }
            TRY(snap_img(ctx, snaps, name("t%d_bwd_nb%d", t, k), ctx->nb, k, Bc, true, st));
            if (!fused_k) {
                ProfScope ps(ctx, last ? GNNB_K_UPDATE_BWD_SCORE : GNNB_K_UPDATE_BWD, nodes, st);
                if (tc) tc_update(g, true, in.lb[k], in.ub[k], ctx->nb, ctx->relax_b[k], ctx->amb_base[k], mu_k, sc, M(k), ctx->n_hidden, ctx->hidden_off[k], rows, ctx->d_nan, nd, st, lc);
                else simt_update(g, true, in.lb[k], in.ub[k], ctx->nb, ctx->relax_b[k], ctx->mu[k], sc, ctx->n[k], ctx->n_hidden, ctx->hidden_off[k], rows, ctx->d_nan, st, lc);
            }
            TRY(snap_img(ctx, snaps, name("t%d_bwd_mu%d", t, k), ctx->mu[k], k, Bc, false, st));
        }
        // input layer: feeds the next round only (dead on the last round, SURVEY §8a fact 2)
        if (!last && fused) {
            ProfScope ps(ctx, GNNB_K_INPUT_UPDATE, (int64_t)Bc * ctx->n[0], st);
            tc_fused(g, ctx->plan_bwd[0], ctx->mu[1], true, in.lb[0], in.ub[0], nullptr, nullptr, ctx->mu[0], nullptr, M(0), 0, 0, R(0),
                     ctx->d_nan, nd, nullptr, true, st, lc);
            TRY(snap_img(ctx, snaps, name("t%d_mu0", t, 0), ctx->mu[0], 0, Bc, false, st));
        } else if (!last) {
            {
                ProfScope ps(ctx, GNNB_K_PROP_BWD, (int64_t)Bc * ctx->n[0], st);
                if (tc) prop_tc_run(ctx->plan_bwd[0], ctx->mu[1], ctx->nb, Bc, st, lc);
                else prop_backward(ctx->layers[0], ctx->mu[1], ctx->nb, Bc, false, st, lc);
            }
            {
                ProfScope ps(ctx, GNNB_K_INPUT_UPDATE, (int64_t)Bc * ctx->n[0], st);
                if (tc) tc_input_update(g, in.lb[0], in.ub[0], ctx->nb, ctx->mu[0], M(0), R(0), st, lc);
                else simt_input_update(g, in.lb[0], in.ub[0], ctx->nb, ctx->mu[0], R(0), st, lc);
            }
            TRY(snap_img(ctx, snaps, name("t%d_mu0", t, 0), ctx->mu[0], 0, Bc, false, st));
        }
    }
    {
        ProfScope ps(ctx, GNNB_K_ARGMAX, Bc, st);
        if (k == 1) masked_argmax(scores, mask, ctx->n_hidden, Bc, best_score, best_idx, winners, st, lc);
        else masked_topk(scores, mask, ctx->n_hidden, Bc, k, best_score, best_idx, st, lc);
    }
    CU(cudaGetLastError());
    return GNNB_OK;
}

// grow-only NanDoms buffer of option "rescore" for calls of up to B subdomains (zeroed when it is allocated)
int ensure_nan_doms(gnnb_ctx* ctx, int B) {
    if (ctx->resc_cap >= B) return GNNB_OK;
    if (ctx->d_resc) { cudaFree(ctx->d_resc); ctx->d_resc = nullptr; ctx->resc_cap = 0; }
    CU(cudaMalloc(&ctx->d_resc, (1 + 2 * (size_t)B) * sizeof(int32_t)));
    CU(cudaMemset(ctx->d_resc, 0, (1 + 2 * (size_t)B) * sizeof(int32_t)));
    ctx->resc_cap = B;
    return GNNB_OK;
}

// grow-only per-domain scratch of gnnb_child_bounds / gnnb_root_bounds / gnnb_score_grad_device for B domains (3 B + 2 int32)
int ensure_kw_iscratch(gnnb_ctx* ctx, int B, cudaStream_t st) {
    if (ctx->kw_iscratch_cap >= B) return GNNB_OK;
    if (ctx->kw_iscratch) { CU(cudaStreamSynchronize(st)); cudaFree(ctx->kw_iscratch); ctx->kw_iscratch = nullptr; ctx->kw_iscratch_cap = 0; }
    CU(cudaMalloc(&ctx->kw_iscratch, (3 * (size_t)B + 2) * sizeof(int32_t)));
    ctx->kw_iscratch_cap = B;
    return GNNB_OK;
}

NanDoms nan_doms(gnnb_ctx* ctx) { return NanDoms{ctx->d_resc, ctx->d_resc + 1, ctx->d_resc + 1 + ctx->resc_cap, 0}; }

// after a call that failed part-way: no subdomain may stay flagged for the next call
void reset_nan_doms(gnnb_ctx* ctx, cudaStream_t st) {
    cudaStreamSynchronize(st);
    cudaMemset(ctx->d_resc, 0, (1 + 2 * (size_t)ctx->resc_cap) * sizeof(int32_t));
}

// Option "rescore", after the tensor-core pass of a call: read how many subdomains its NaN watch flagged (one device -> host copy
// and one synchronise of `st`; nothing else when there are none), then score those again with the exact-fp32 schedule, in waves
// of up to `chunk` gathered into staging set 0, and write their results over the tensor-core ones.  best / idx [B, k] or winners:
// device arrays of the whole call; scores: the caller's dense scores (in->mem) or null.  The NaN count is reset first, so that
// afterwards it counts the fp32 pass only.
int rescore_flagged(gnnb_ctx* ctx, const gnnb_frontier* in, int chunk, int k, float* best, int32_t* idx, gnnb_winner* winners,
                    float* scores, cudaStream_t st) {
    const bool host = in->mem == GNNB_MEM_HOST;
    const int nh = ctx->n_hidden;
    const NanDoms nd = nan_doms(ctx);
    int32_t count = 0;
    CU(cudaMemcpyAsync(&count, nd.count, sizeof count, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    ctx->rescored = count;
    if (count == 0) return GNNB_OK;
    std::vector<int32_t> rows;                    // host frontier: the flagged rows are copied from the caller's arrays one by one
    if (host) {
        rows.resize(count);
        CU(cudaMemcpyAsync(rows.data(), nd.list, (size_t)count * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    CU(cudaMemsetAsync(nd.count, 0, sizeof(int32_t), st));             // the scatter kernel clears the flags
    CU(cudaMemsetAsync(ctx->d_nan, 0, sizeof(unsigned long long), st));
    gnnb_ctx::Staging& sg = ctx->stg[0];
    std::vector<RowGather> tab;
    GnnInputs cp((int)ctx->layers.size());
    walk_inputs(*in, cp, ctx->n, [&](const float* src, const float*& slot, int64_t per) {
        float* dst = sg.inputs[tab.size()];
        tab.push_back(RowGather{src, dst, per});
        slot = dst;
    });
    tab.push_back(RowGather{in->mask, sg.mask, nh});
    if (!host) {
        if (ctx->gather_cap < tab.size()) {
            if (ctx->d_gather) cudaFree(ctx->d_gather);
            ctx->d_gather = nullptr; ctx->gather_cap = 0;
            CU(cudaMalloc(&ctx->d_gather, tab.size() * sizeof(RowGather)));
            ctx->gather_cap = tab.size();
        }
        // a stream-ordered copy from pageable memory returns after the source has been read: `tab` may go out of scope
        CU(cudaMemcpyAsync(ctx->d_gather, tab.data(), tab.size() * sizeof(RowGather), cudaMemcpyHostToDevice, st));
    }
    for (int s0 = 0, Bs = 0; s0 < count; s0 += Bs) {
        Bs = (count - s0) < chunk ? (count - s0) : chunk;
        if (host) {
            for (int i = 0; i < Bs; ++i)
                for (const RowGather& t : tab)
                    CU(cudaMemcpyAsync(t.dst + i * t.per, t.src + rows[s0 + i] * t.per, t.per * sizeof(float), cudaMemcpyHostToDevice, st));
        } else {
            gather_rows(ctx->d_gather, (int)tab.size(), nd.list + s0, Bs, st, &ctx->launches);
        }
        TRY(run_chunk(ctx, cp, sg.mask, Bs, GNNB_MATH_SIMT_FP32, NanDoms{nullptr, nullptr, nullptr, 0}, sg.scores, k, sg.best, sg.idx, nullptr, st));
        scatter_rescored(nd.list + s0, Bs, k, sg.best, sg.idx, sg.scores, nh, best, idx, winners, host ? nullptr : scores, nd.flag, st,
                         &ctx->launches);
        if (host && scores)
            for (int i = 0; i < Bs; ++i)
                CU(cudaMemcpyAsync(scores + (size_t)rows[s0 + i] * nh, sg.scores + (size_t)i * nh, (size_t)nh * sizeof(float),
                                   cudaMemcpyDeviceToHost, st));
    }
    CU(cudaEventRecord(ctx->ev_free[0], st));       // the next host-buffer wave that stages into set 0 waits for this pass
    CU(cudaGetLastError());
    return GNNB_OK;
}

// upload the 52 host tensors in every form the kernels read: transposed fp32, composed linears, tensor-core planes, and
// the nn.Linear-layout master copy of the fine-tuning path (its gradient and Adam buffers are kept when they exist)
int upload_gnn(gnnb_ctx* ctx, const float* const* tensors, int T) {
    // fp32 blob: transposed weights + biases
    std::vector<size_t> o_w(N_LIN), o_b(N_LIN);
    size_t total = 0;
    for (int l = 0; l < N_LIN; ++l) {
        o_w[l] = total; total += align4((size_t)lin_in(l) * lin_out(l));
        o_b[l] = total; total += align4(lin_out(l));
    }
    std::vector<float> blob(total, 0.f);
    for (int l = 0; l < N_LIN; ++l) {
        const int K = lin_in(l), N = lin_out(l);
        const float* W = tensors[2 * l];
        for (int nn = 0; nn < N; ++nn)
            for (int k = 0; k < K; ++k) blob[o_w[l] + (size_t)k * N + nn] = W[(size_t)nn * K + k];
        memcpy(&blob[o_b[l]], tensors[2 * l + 1], sizeof(float) * N);
    }
    // composed linears of the tensor-core path (gnnb_tc.cu header), formed in double
    std::vector<float> cw((size_t)N_TCLIN * P * P, 0.f), cb((size_t)N_TCLIN * P, 0.f);
    auto compose = [&](int id, int outer, int half, int inner, bool add_outer_bias) {
        // W = outer[:, half*64 : half*64+64] * inner (or the slice itself when inner < 0);  b = [b_outer +] slice * b_inner
        const float* Wo = tensors[2 * outer];
        const float* bo = tensors[2 * outer + 1];
        const int Ko = lin_in(outer);
        for (int nn = 0; nn < P; ++nn) {
            double bacc = add_outer_bias ? (double)bo[nn] : 0.0;
            for (int k = 0; k < P; ++k) {
                double acc = 0.0;
                if (inner < 0) acc = Wo[(size_t)nn * Ko + half * P + k];
                else
                    for (int j = 0; j < P; ++j) acc += (double)Wo[(size_t)nn * Ko + half * P + j] * (double)tensors[2 * inner][(size_t)j * P + k];
                cw[((size_t)id * P + nn) * P + k] = (float)acc;
            }
            if (inner >= 0)
                for (int j = 0; j < P; ++j) bacc += (double)Wo[(size_t)nn * Ko + half * P + j] * (double)tensors[2 * inner + 1][j];
            cb[(size_t)id * P + nn] = (float)bacc;
        }
    };
    compose(T_FWD_R, FC4, 0, FC1_1, false);
    compose(T_FWD_C, FC4, 1, FC3_2, true);
    compose(T_BWD_R, BC4, 0, BC2_1, false);
    compose(T_BWD_C, BC4, 1, BC3_1, true);
    compose(T_INP_C, INP_B2, 0, INP_B_1, true);
    compose(T_INP_NB, INP_B2, 1, -1, false);
    // tensor-core planes for the K >= 64 linears
    std::vector<size_t> o_tc(N_LIN, 0);
    size_t tc_total = 0;
    for (int l = 0; l < N_LIN; ++l)
        if (lin_in(l) >= P && lin_out(l) == P) { o_tc[l] = tc_total; tc_total += (size_t)tc_packed_elems(lin_in(l)); }
    std::vector<size_t> o_tcx(N_TCLIN, 0);
    for (int i = 0; i < N_TCLIN; ++i) { o_tcx[i] = tc_total; tc_total += (size_t)tc_packed_elems(P); }
    std::vector<uint16_t> tcblob(tc_total ? tc_total : 1, 0);
    for (int l = 0; l < N_LIN; ++l)
        if (lin_in(l) >= P && lin_out(l) == P) tc_pack_weight(tensors[2 * l], lin_in(l), &tcblob[o_tc[l]]);
    for (int i = 0; i < N_TCLIN; ++i) tc_pack_weight(&cw[(size_t)i * P * P], P, &tcblob[o_tcx[i]]);
    const size_t o_cb = total;            // composed biases ride at the end of the fp32 blob
    total += cb.size();
    blob.resize(total, 0.f);
    memcpy(&blob[o_cb], cb.data(), cb.size() * sizeof(float));
    // the blobs have fixed sizes (p = 64): allocated once, overwritten by later uploads (an Adam step re-uploads every time);
    // no kernel of an earlier call may still be reading them
    CU(cudaDeviceSynchronize());
    if (!ctx->d_gnn) CU(cudaMalloc(&ctx->d_gnn, total * sizeof(float)));
    if (!ctx->d_tc) CU(cudaMalloc(&ctx->d_tc, tcblob.size() * sizeof(uint16_t)));
    CU(cudaMemcpy(ctx->d_gnn, blob.data(), total * sizeof(float), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(ctx->d_tc, tcblob.data(), tcblob.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
    for (int l = 0; l < N_LIN; ++l) {
        ctx->gp.wt[l] = ctx->d_gnn + o_w[l];
        ctx->gp.bias[l] = ctx->d_gnn + o_b[l];
        ctx->gp.tc[l] = (lin_in(l) >= P && lin_out(l) == P) ? ctx->d_tc + o_tc[l] : nullptr;
    }
    for (int i = 0; i < N_TCLIN; ++i) {
        ctx->gp.tcx_w[i] = ctx->d_tc + o_tcx[i];
        ctx->gp.tcx_b[i] = ctx->d_gnn + o_cb + (size_t)i * P;
    }
    ctx->gp.T = T;
    // master copy (nn.Linear layout, state_dict order); the gradient / Adam quarters survive a re-upload
    if (!ctx->d_train) {
        size_t np = 0;
        for (int l = 0; l < N_LIN; ++l) {
            ctx->po_w[l] = np; np += align4((size_t)lin_in(l) * lin_out(l));
            ctx->po_b[l] = np; np += align4(lin_out(l));
        }
        ctx->n_params = (int64_t)np;
        CU(cudaMalloc(&ctx->d_train, 4 * np * sizeof(float)));
        CU(cudaMemset(ctx->d_train, 0, 4 * np * sizeof(float)));
        ctx->adam_steps = 0;
    }
    {
        std::vector<float> master((size_t)ctx->n_params, 0.f);
        for (int l = 0; l < N_LIN; ++l) {
            memcpy(&master[ctx->po_w[l]], tensors[2 * l], sizeof(float) * lin_in(l) * lin_out(l));
            memcpy(&master[ctx->po_b[l]], tensors[2 * l + 1], sizeof(float) * lin_out(l));
        }
        CU(cudaMemcpy(ctx->d_train, master.data(), master.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    ctx->have_gnn = true;
    return GNNB_OK;
}

TrainParams train_params(gnnb_ctx* ctx) {
    TrainParams tp;
    float* grad = ctx->d_train + ctx->n_params;
    for (int l = 0; l < N_LIN; ++l) {
        tp.w[l] = ctx->d_train + ctx->po_w[l]; tp.b[l] = ctx->d_train + ctx->po_b[l];
        tp.dw[l] = grad + ctx->po_w[l]; tp.db[l] = grad + ctx->po_b[l];
    }
    return tp;
}

// copy one quarter of the training block (0 = parameters, 1 = gradients) to 52 host tensors in state_dict order
int download_quarter(gnnb_ctx* ctx, int quarter, float* const* tensors, const int64_t* numels, int n_tensors) {
    if (!ctx || !tensors || !numels) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    if (!ctx->have_gnn) return fail(ctx, GNNB_ERR_STATE, "gnnb_set_gnn_weights must be called first");
    if (n_tensors != 2 * N_LIN) return fail(ctx, GNNB_ERR_INVALID, "expected 52 tensors (weight, bias of 26 linears)");
    for (int l = 0; l < N_LIN; ++l)
        if (numels[2 * l] != (int64_t)lin_in(l) * lin_out(l) || numels[2 * l + 1] != lin_out(l))
            return fail(ctx, GNNB_ERR_INVALID, "tensor " + std::to_string(2 * l) + " has the wrong number of elements");
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    // host or device destinations: the direction follows from the pointer (unified addressing)
    const float* src = ctx->d_train + (size_t)quarter * ctx->n_params;
    for (int l = 0; l < N_LIN; ++l) {
        CU(cudaMemcpy(tensors[2 * l], src + ctx->po_w[l], sizeof(float) * lin_in(l) * lin_out(l), cudaMemcpyDefault));
        CU(cudaMemcpy(tensors[2 * l + 1], src + ctx->po_b[l], sizeof(float) * lin_out(l), cudaMemcpyDefault));
    }
    return GNNB_OK;
}

}  // namespace

extern "C" {

int gnnb_abi_version(void) { return 1; }

int gnnb_create(gnnb_ctx** out, int device) {
    if (!out) return GNNB_ERR_INVALID;
    *out = nullptr;
    gnnb_ctx* ctx = new gnnb_ctx();
    ctx->device = device;
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) { delete ctx; return GNNB_ERR_CUDA; }
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) { delete ctx; return GNNB_ERR_CUDA; }
    if (prop.major != 10) {   // sm_100a cubins only; there is no other code path
        fprintf(stderr, "libgnnb: device %d is sm_%d%d; this library is built for sm_100a (B200) only\n", device, prop.major, prop.minor);
        delete ctx;
        return GNNB_ERR_UNSUPPORTED;
    }
    if (cudaMalloc(&ctx->d_nan, sizeof(unsigned long long)) != cudaSuccess ||
        cudaMemset(ctx->d_nan, 0, sizeof(unsigned long long)) != cudaSuccess ||
        simt_init() != 0 || prop_init(64 * 1024) != 0 || tc_init() != 0 || prop_tc_init() != 0 || kw_init() != 0 || train_init() != 0) {
        fprintf(stderr, "libgnnb: initialisation failed: %s\n", cudaGetErrorString(cudaGetLastError()));
        if (ctx->d_nan) cudaFree(ctx->d_nan);
        delete ctx;
        return GNNB_ERR_CUDA;
    }
    *out = ctx;
    return GNNB_OK;
}

void gnnb_destroy(gnnb_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    free_workspace(ctx);
    if (ctx->d_gnn) cudaFree(ctx->d_gnn);
    if (ctx->d_tc) cudaFree(ctx->d_tc);
    if (ctx->d_train) cudaFree(ctx->d_train);
    if (ctx->train_ws) cudaFree(ctx->train_ws);
    if (ctx->kw_ws) cudaFree(ctx->kw_ws);
    if (ctx->kw_iscratch) cudaFree(ctx->kw_iscratch);
    if (ctx->d_net) cudaFree(ctx->d_net);
    if (ctx->d_maps) cudaFree(ctx->d_maps);
    if (ctx->d_layers) cudaFree(ctx->d_layers);
    if (ctx->d_hidden_off) cudaFree(ctx->d_hidden_off);
    if (ctx->d_random_order) cudaFree(ctx->d_random_order);
    if (ctx->d_ptrs) cudaFree(ctx->d_ptrs);
    if (ctx->d_nan) cudaFree(ctx->d_nan);
    if (ctx->d_resc) cudaFree(ctx->d_resc);
    if (ctx->d_gather) cudaFree(ctx->d_gather);
    for (PropPlan* p : ctx->plan_fwd) prop_plan_free(p);
    for (PropPlan* p : ctx->plan_bwd) prop_plan_free(p);
    for (PropPlan* p : ctx->plan_kw_own) prop_plan_free(p);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->res_best) cudaFree(ctx->res_best);
    if (ctx->res_idx) cudaFree(ctx->res_idx);
    for (int i = 0; i < 2; ++i) { if (ctx->ev_copied[i]) cudaEventDestroy(ctx->ev_copied[i]); if (ctx->ev_free[i]) cudaEventDestroy(ctx->ev_free[i]); }
    for (auto& p : ctx->pending) { cudaEventDestroy(p.a); cudaEventDestroy(p.b); }
    for (auto e : ctx->ev_pool) cudaEventDestroy(e);
    for (gnnb_queue* q : ctx->queues) q->ctx = nullptr;
    delete ctx;
}

int gnnb_set_gnn_weights(gnnb_ctx* ctx, const float* const* tensors, const int64_t* numels, int n_tensors, int T, int p) {
    if (!ctx || !tensors || !numels) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    if (p != P) return fail(ctx, GNNB_ERR_UNSUPPORTED, "embedding size p must be 64");
    if (T < 1) return fail(ctx, GNNB_ERR_INVALID, "T must be >= 1");
    if (n_tensors != 2 * N_LIN) return fail(ctx, GNNB_ERR_INVALID, "expected 52 tensors (weight, bias of 26 linears)");
    for (int l = 0; l < N_LIN; ++l) {
        if (numels[2 * l] != (int64_t)lin_in(l) * lin_out(l) || numels[2 * l + 1] != lin_out(l))
            return fail(ctx, GNNB_ERR_INVALID, "tensor " + std::to_string(2 * l) + " has the wrong number of elements");
    }
    CU(cudaSetDevice(ctx->device));
    return upload_gnn(ctx, tensors, T);
}

int gnnb_set_network(gnnb_ctx* ctx, const gnnb_layer_desc* layers, int n_layers, int c0, int h0, int w0) {
    if (!ctx || !layers || n_layers < 1) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    if (!ctx->queues.empty()) return fail(ctx, GNNB_ERR_STATE, "gnnb_set_network while domain queues of the previous network exist");
    CU(cudaSetDevice(ctx->device));
    std::vector<LayerDev> devs(n_layers);
    std::vector<int> n(n_layers + 2);
    n[0] = c0 * h0 * w0;
    int pc = c0, ph = h0, pw = w0;
    bool flat = false;
    size_t total = 0;
    std::vector<size_t> o_w(n_layers), o_b(n_layers);
    for (int k = 0; k < n_layers; ++k) {
        const gnnb_layer_desc& d = layers[k];
        LayerDev& L = devs[k];
        L.kind = d.kind;
        L.c_in = d.c_in; L.h_in = d.h_in; L.w_in = d.w_in; L.c_out = d.c_out; L.h_out = d.h_out; L.w_out = d.w_out;
        L.ksize = d.ksize; L.stride = d.stride; L.pad = d.pad;
        L.n_in = d.c_in * d.h_in * d.w_in;
        L.n_out = d.c_out * d.h_out * d.w_out;
        if (!d.weight || !d.bias) return fail(ctx, GNNB_ERR_INVALID, "layer weight/bias is null");
        if (L.n_in != n[k]) return fail(ctx, GNNB_ERR_INVALID, "layer " + std::to_string(k) + ": input size does not match the previous layer");
        size_t wn;
        if (d.kind == GNNB_LAYER_CONV) {
            if (flat || d.c_in != pc || d.h_in != ph || d.w_in != pw) return fail(ctx, GNNB_ERR_INVALID, "conv layer input shape mismatch");
            if (d.ksize < 1 || d.stride < 1 || d.pad < 0) return fail(ctx, GNNB_ERR_INVALID, "bad conv geometry");
            if (d.h_out != (d.h_in + 2 * d.pad - d.ksize) / d.stride + 1 || d.w_out != (d.w_in + 2 * d.pad - d.ksize) / d.stride + 1)
                return fail(ctx, GNNB_ERR_INVALID, "conv output shape mismatch");
            // conv_transpose2d must land exactly on the input grid (no output_padding in the reference call)
            if ((d.h_out - 1) * d.stride - 2 * d.pad + d.ksize != d.h_in || (d.w_out - 1) * d.stride - 2 * d.pad + d.ksize != d.w_in)
                return fail(ctx, GNNB_ERR_UNSUPPORTED, "conv geometry needs output_padding in the backward pass");
            if ((size_t)d.c_in * d.ksize * d.ksize * d.c_out * sizeof(float) > 64 * 1024)
                return fail(ctx, GNNB_ERR_UNSUPPORTED, "conv weights exceed the 64 KB shared-memory staging buffer");
            wn = (size_t)d.c_out * d.c_in * d.ksize * d.ksize;
            pc = d.c_out; ph = d.h_out; pw = d.w_out;
        } else if (d.kind == GNNB_LAYER_LINEAR) {
            if (d.h_in != 1 || d.w_in != 1 || d.h_out != 1 || d.w_out != 1) return fail(ctx, GNNB_ERR_INVALID, "linear layers use c_in/c_out only");
            wn = (size_t)L.n_out * L.n_in;
            flat = true;
        } else {
            return fail(ctx, GNNB_ERR_INVALID, "unknown layer kind");
        }
        n[k + 1] = L.n_out;
        o_w[k] = total; total += align4(wn);
        o_b[k] = total; total += align4(L.n_out);
    }
    n[n_layers + 1] = 1;
    std::vector<float> blob(total, 0.f);
    for (int k = 0; k < n_layers; ++k) {
        const gnnb_layer_desc& d = layers[k];
        const LayerDev& L = devs[k];
        const size_t wn = d.kind == GNNB_LAYER_CONV ? (size_t)d.c_out * d.c_in * d.ksize * d.ksize : (size_t)L.n_out * L.n_in;
        memcpy(&blob[o_w[k]], d.weight, wn * sizeof(float));
        const int per = d.kind == GNNB_LAYER_CONV ? d.h_out * d.w_out : 1;     // graph_conv.py:122-124
        for (int j = 0; j < L.n_out; ++j) blob[o_b[k] + j] = d.bias[j / per];
    }
    // Transactional: everything the new network needs is built into locals first; the context is only touched once every
    // allocation, copy and plan has succeeded, so a failure leaves the previous network (if any) fully usable.
    struct Staged {
        float* d_net = nullptr;
        int32_t* d_maps = nullptr;
        LayerDev* d_layers = nullptr;
        int32_t *d_hidden_off = nullptr, *d_random_order = nullptr;
        const float** d_ptrs = nullptr;
        std::vector<PropPlan*> plan_fwd, plan_bwd, plan_kw_own;
        bool keep = false;
        ~Staged() {
            if (keep) return;
            if (d_net) cudaFree(d_net);
            if (d_maps) cudaFree(d_maps);
            if (d_layers) cudaFree(d_layers);
            if (d_hidden_off) cudaFree(d_hidden_off);
            if (d_random_order) cudaFree(d_random_order);
            if (d_ptrs) cudaFree(d_ptrs);
            for (PropPlan* p : plan_fwd) prop_plan_free(p);
            for (PropPlan* p : plan_bwd) prop_plan_free(p);
            for (PropPlan* p : plan_kw_own) prop_plan_free(p);
        }
    } sg;
    CU(cudaMalloc(&sg.d_net, total * sizeof(float)));
    CU(cudaMemcpy(sg.d_net, blob.data(), total * sizeof(float), cudaMemcpyHostToDevice));
    for (int k = 0; k < n_layers; ++k) { devs[k].weight = sg.d_net + o_w[k]; devs[k].bias_node = sg.d_net + o_b[k]; }
    sg.plan_fwd.assign(n_layers, nullptr);
    sg.plan_bwd.assign(n_layers, nullptr);
    sg.plan_kw_own.assign(n_layers, nullptr);
    // slot order of layers 0..L (gnnb_common.cuh) and the device copies of the slot -> node maps
    std::vector<LayerTiling> tiling(n_layers + 1);
    std::vector<RowMap> rowmap(n_layers + 1, RowMap{nullptr, 0, 0});
    tiling[0] = make_tiling(c0, h0, w0);
    for (int k = 0; k < n_layers; ++k)
        tiling[k + 1] = devs[k].kind == GNNB_LAYER_CONV ? make_tiling(devs[k].c_out, devs[k].h_out, devs[k].w_out)
                                                       : make_tiling(devs[k].n_out, 1, 1);
    {
        size_t total_slots = 0;
        for (const LayerTiling& t : tiling) total_slots += t.node_of_slot.size();
        CU(cudaMalloc(&sg.d_maps, total_slots * sizeof(int32_t)));
        size_t off = 0;
        for (int k = 0; k <= n_layers; ++k) {
            const LayerTiling& t = tiling[k];
            CU(cudaMemcpy(sg.d_maps + off, t.node_of_slot.data(), t.node_of_slot.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
            rowmap[k] = RowMap{sg.d_maps + off, n[k], (int)t.node_of_slot.size()};
            off += t.node_of_slot.size();
        }
    }
    for (int k = 0; k < n_layers; ++k) {
        // layer 0's transpose feeds the input nodes and is not normalised (graph_conv.py:361-372); the others are (:299-318)
        sg.plan_fwd[k] = prop_plan_build(devs[k], layers[k].weight, false, false, tiling[k + 1], tiling[k]);
        sg.plan_bwd[k] = prop_plan_build(devs[k], layers[k].weight, true, k > 0, tiling[k], tiling[k + 1]);
        if (!sg.plan_fwd[k] || !sg.plan_bwd[k]) return fail(ctx, GNNB_ERR_CUDA, "building the propagation plans failed");
        // the bound producer's dense recursion needs A_{k+1}^T without the tap-count normalisation (gnnb_kw.cu)
        if (k > 0 && devs[k].kind == GNNB_LAYER_CONV) {
            sg.plan_kw_own[k] = prop_plan_build(devs[k], layers[k].weight, true, false, tiling[k], tiling[k + 1]);
            if (!sg.plan_kw_own[k]) return fail(ctx, GNNB_ERR_CUDA, "building the propagation plans failed");
        }
    }
    std::vector<int> hidden_off(n_layers + 2, 0);
    int n_hidden = 0;
    for (int k = 1; k <= n_layers; ++k) { hidden_off[k] = n_hidden; n_hidden += n[k]; }
    // tables of the BaBSR kernel
    CU(cudaMalloc(&sg.d_layers, n_layers * sizeof(LayerDev)));
    CU(cudaMemcpy(sg.d_layers, devs.data(), n_layers * sizeof(LayerDev), cudaMemcpyHostToDevice));
    CU(cudaMalloc(&sg.d_hidden_off, (n_layers + 1) * sizeof(int32_t)));
    CU(cudaMemcpy(sg.d_hidden_off, hidden_off.data() + 1, (n_layers + 1) * sizeof(int32_t), cudaMemcpyHostToDevice));
    CU(cudaMalloc(&sg.d_random_order, n_layers * sizeof(int32_t)));
    CU(cudaMalloc(&sg.d_ptrs, 2 * (n_layers + 2) * sizeof(float*)));
    // ---- commit: nothing below can fail ----
    CU(cudaDeviceSynchronize());                 // no kernel of an earlier call may still read the old tables
    ctx->have_net = false;
    free_workspace(ctx);
    if (ctx->d_net) cudaFree(ctx->d_net);
    if (ctx->d_maps) cudaFree(ctx->d_maps);
    if (ctx->d_layers) cudaFree(ctx->d_layers);
    if (ctx->d_hidden_off) cudaFree(ctx->d_hidden_off);
    if (ctx->d_random_order) cudaFree(ctx->d_random_order);
    if (ctx->d_ptrs) cudaFree(ctx->d_ptrs);
    for (PropPlan* p : ctx->plan_fwd) prop_plan_free(p);
    for (PropPlan* p : ctx->plan_bwd) prop_plan_free(p);
    for (PropPlan* p : ctx->plan_kw_own) prop_plan_free(p);
    sg.keep = true;
    ctx->d_net = sg.d_net; ctx->d_maps = sg.d_maps; ctx->d_layers = sg.d_layers; ctx->d_hidden_off = sg.d_hidden_off;
    ctx->d_random_order = sg.d_random_order; ctx->d_ptrs = sg.d_ptrs;
    ctx->plan_fwd = sg.plan_fwd; ctx->plan_bwd = sg.plan_bwd; ctx->plan_kw_own = sg.plan_kw_own;
    ctx->plan_kw.assign(n_layers, nullptr);
    for (int k = 0; k < n_layers; ++k) ctx->plan_kw[k] = sg.plan_kw_own[k] ? sg.plan_kw_own[k] : sg.plan_bwd[k];
    ctx->tiling = tiling; ctx->rowmap = rowmap;
    ctx->layers = devs;
    ctx->n = n;
    ctx->zero_tap_layer = first_zero_tap_layer(devs);
    ctx->hidden_off = hidden_off;
    ctx->n_hidden = n_hidden;
    ctx->have_net = true;
    return GNNB_OK;
}

int gnnb_set_option(gnnb_ctx* ctx, const char* key, int64_t value) {
    if (!ctx || !key) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    const std::string k(key);
    if (k == "math") {
        if (value != GNNB_MATH_TC_FP16X3 && value != GNNB_MATH_SIMT_FP32) return fail(ctx, GNNB_ERR_INVALID, "unknown math mode");
        if (value == GNNB_MATH_TC_FP16X3 && !tc_available()) return fail(ctx, GNNB_ERR_UNSUPPORTED, "tensor-core path not built");
        ctx->math = (int)value;
    } else if (k == "chunk") {
        if (value < 0) return fail(ctx, GNNB_ERR_INVALID, "chunk must be >= 0");
        ctx->chunk = (int)value;
    } else if (k == "fuse") {
        ctx->fuse = value ? 1 : 0;
    } else if (k == "snapshot") {
        ctx->snapshot = value ? 1 : 0;
    } else if (k == "profile") {
        ctx->profile = value ? 1 : 0;
    } else if (k == "rescore") {
        ctx->rescore = value ? 1 : 0;
    } else if (k == "grad_chunk") {
        if (value < 0 || value > 0x7fffffff) return fail(ctx, GNNB_ERR_INVALID, "grad_chunk must be in [0, 2^31)");
        ctx->grad_chunk = (int)value;
    } else {
        return fail(ctx, GNNB_ERR_INVALID, "unknown option " + k);
    }
    return GNNB_OK;
}

int64_t gnnb_get_option(gnnb_ctx* ctx, const char* key) {
    if (!ctx || !key) return -1;
    const std::string k(key);
    if (k == "math") return ctx->math;
    if (k == "chunk") return ctx->chunk;
    if (k == "snapshot") return ctx->snapshot;
    if (k == "fuse") return ctx->fuse;
    if (k == "profile") return ctx->profile;
    if (k == "rescore") return ctx->rescore;
    if (k == "rescored") return ctx->rescored;
    if (k == "grad_chunk") return ctx->grad_chunk;
    if (k == "grad_workspace_domains") return ctx->grad_ws_domains;
    if (k == "grad_bad_terms") return ctx->grad_bad_terms;
    if (k == "n_hidden") return ctx->n_hidden;
    if (k == "workspace_domains") return ctx->ws_cap;
    if (k.rfind("plan_density_pct_", 0) == 0) {      // e.g. plan_density_pct_f0 / plan_density_pct_b1
        const bool bwd = k[17] == 'b';
        const size_t i = (size_t)atoi(k.c_str() + 18);
        const auto& v = bwd ? ctx->plan_bwd : ctx->plan_fwd;
        return i < v.size() ? (int64_t)(100.0 * prop_plan_density(v[i])) : -1;
    }
    return -1;
}

// best_score / best_idx: [B, k] (k = 1: gnnb_score), or winner records (k = 1)
static int score_impl(gnnb_ctx* ctx, const gnnb_frontier* in, int k, float* best_score, int32_t* best_idx, gnnb_winner* winners,
                      float* scores, void* stream) {
    if (!ctx || !in || ((!best_score || !best_idx) && !winners)) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    if (!ctx->have_gnn || !ctx->have_net) return fail(ctx, GNNB_ERR_STATE, "gnnb_set_gnn_weights and gnnb_set_network must be called first");
    if (in->B < 0) return fail(ctx, GNNB_ERR_INVALID, "negative batch");
    ctx->rescored = 0;
    TRY(check_zero_taps(ctx));
    if (in->B == 0) return GNNB_OK;
    GnnInputs cp((int)ctx->layers.size());         // the arrays of each wave, staged or in place
    TRY(frontier_inputs(ctx, in, true, &cp));
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const bool host = in->mem == GNNB_MEM_HOST;
    // subdomains per wave: large waves amortise launches and tails; with host buffers smaller waves let the copies of
    // wave i + 1 (copy stream, second staging set) run under the kernels of wave i
    int chunk = ctx->chunk > 0 ? ctx->chunk : 1024;
    if (chunk > in->B) chunk = in->B;
    const bool resc = ctx->rescore && ctx->math == GNNB_MATH_TC_FP16X3;
    TRY(ensure_workspace(ctx, chunk, host || resc));        // the re-score pass gathers its sub-frontier into a staging set
    NanDoms nd{nullptr, nullptr, nullptr, 0};
    if (resc) {
        TRY(ensure_nan_doms(ctx, in->B));
        nd = nan_doms(ctx);
    }
    const int64_t n_res = (int64_t)in->B * k;
    if (host && !winners && ctx->res_cap < n_res) {
        if (ctx->res_best) cudaFree(ctx->res_best);
        if (ctx->res_idx) cudaFree(ctx->res_idx);
        ctx->res_best = nullptr; ctx->res_idx = nullptr; ctx->res_cap = 0;
        CU(cudaMalloc(&ctx->res_best, (size_t)n_res * sizeof(float)));
        CU(cudaMalloc(&ctx->res_idx, (size_t)n_res * sizeof(int32_t)));
        ctx->res_cap = n_res;
    }

    // host buffers: the first wave is small so that the kernels start after a short copy; a later wave's copy (copy stream, the
    // other staging set) hides behind the kernels of the wave before it only if it is not much larger than that wave — the copy
    // engine moves a subdomain's inputs 1.3x (base) - 1.6x (wide) faster than the kernels score it — so the wave size grows by
    // 1.5x: 128, 192, 288, 432, ... up to `chunk`.  (A fixed ~0.2 ms of launch fill and drain per wave is the price of many
    // waves; a simulation of the two streams over start sizes 32 - 128 and growth factors 1 - 4 puts this schedule within 1 %
    // of the best for 1 024 - 8 192 subdomains; the earlier 64, 256, 1 024 left the GPU idle for 1 ms of a 5.7 ms call.)
    int wave = 0, ramp = host ? (chunk < 128 ? chunk : 128) : chunk;
    for (int c0 = 0, Bc = 0; c0 < in->B; c0 += Bc, ++wave) {
        Bc = (in->B - c0) < ramp ? (in->B - c0) : ramp;
        ramp = ramp + ramp / 2 > chunk ? chunk : ramp + ramp / 2;
        gnnb_ctx::Staging& sg = ctx->stg[wave & 1];
        cudaStream_t cs = host ? ctx->copy_stream : st;
        // this staging set's previous user (an earlier wave of this call, or the last waves of an earlier call — possibly on
        // another stream, or one that ended in an error) is done; an event that was never recorded is a no-op
        if (host) CU(cudaStreamWaitEvent(cs, ctx->ev_free[wave & 1], 0));
        auto stage = [&](const float* src, float* dst, size_t per_domain) -> const float* {
            const float* p = src + (size_t)c0 * per_domain;
            if (!host) return p;
            cudaMemcpyAsync(dst, p, (size_t)Bc * per_domain * sizeof(float), cudaMemcpyHostToDevice, cs);
            return dst;
        };
        size_t a = 0;
        walk_inputs(*in, cp, ctx->n, [&](const float* src, const float*& slot, int64_t per) {
            slot = stage(src, host ? sg.inputs[a++] : nullptr, per);
        });
        const float* mask = stage(in->mask, sg.mask, ctx->n_hidden);
        CU(cudaGetLastError());
        if (host) {
            CU(cudaEventRecord(ctx->ev_copied[wave & 1], cs));
            CU(cudaStreamWaitEvent(st, ctx->ev_copied[wave & 1], 0));
        }

        float* d_scores = host ? sg.scores : (scores ? scores + (size_t)c0 * ctx->n_hidden : ctx->ws_scores);
        float* d_best = winners ? nullptr : (host ? ctx->res_best : best_score) + (size_t)c0 * k;
        int32_t* d_idx = winners ? nullptr : (host ? ctx->res_idx : best_idx) + (size_t)c0 * k;
        {
            nd.dom0 = c0;
            const int rc = run_chunk(ctx, cp, mask, Bc, ctx->math, nd, d_scores, k, d_best, d_idx, winners ? winners + c0 : nullptr, st);
            if (rc != GNNB_OK) {      // nothing of this call may still be touching the caller's buffers or the staging sets
                if (host) cudaStreamSynchronize(ctx->copy_stream);
                cudaStreamSynchronize(st);
                if (resc) reset_nan_doms(ctx, st);
                return rc;
            }
        }
        if (host) {
            if (scores)
                CU(cudaMemcpyAsync(scores + (size_t)c0 * ctx->n_hidden, d_scores, (size_t)Bc * ctx->n_hidden * sizeof(float),
                                   cudaMemcpyDeviceToHost, st));
            CU(cudaEventRecord(ctx->ev_free[wave & 1], st));
        }
    }
    if (resc) {
        const int rc = rescore_flagged(ctx, in, chunk, k, winners ? nullptr : (host ? ctx->res_best : best_score),
                                       winners ? nullptr : (host ? ctx->res_idx : best_idx), winners, scores, st);
        if (rc != GNNB_OK) {
            reset_nan_doms(ctx, st);
            return rc;
        }
    }
    if (host) {
        if (!winners) {
            CU(cudaMemcpyAsync(best_score, ctx->res_best, (size_t)n_res * sizeof(float), cudaMemcpyDeviceToHost, st));
            CU(cudaMemcpyAsync(best_idx, ctx->res_idx, (size_t)n_res * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        }
        return gnnb_check(ctx, stream, nullptr);
    }
    return GNNB_OK;
}

int gnnb_score(gnnb_ctx* ctx, const gnnb_frontier* in, float* best_score, int32_t* best_idx, float* scores, void* stream) {
    if (!best_score || !best_idx) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    return score_impl(ctx, in, 1, best_score, best_idx, nullptr, scores, stream);
}

int gnnb_score_winners(gnnb_ctx* ctx, const gnnb_frontier* in, gnnb_winner* winners, float* scores, void* stream) {
    if (!winners) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    if (in && in->mem == GNNB_MEM_HOST && scores) return fail(ctx, GNNB_ERR_INVALID, "dense scores of a HOST frontier: use gnnb_score");
    return score_impl(ctx, in, 1, nullptr, nullptr, winners, scores, stream);
}

int gnnb_score_topk(gnnb_ctx* ctx, const gnnb_frontier* in, int32_t k, float* top_score, int32_t* top_idx, float* scores, void* stream) {
    if (k < 1 || k > GNNB_TOPK_MAX) return fail(ctx, GNNB_ERR_INVALID, "k must be in [1, GNNB_TOPK_MAX]");
    if (!top_score || !top_idx) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    return score_impl(ctx, in, k, top_score, top_idx, nullptr, scores, stream);
}

int gnnb_topk(gnnb_ctx* ctx, int32_t B, int32_t n, const float* scores, const float* mask, int32_t k, float* top_score,
              int32_t* top_idx, void* stream) {
    if (!ctx) return GNNB_ERR_INVALID;
    if (k < 1 || k > GNNB_TOPK_MAX) return fail(ctx, GNNB_ERR_INVALID, "k must be in [1, GNNB_TOPK_MAX]");
    if (!scores || !top_score || !top_idx) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    if (B < 0 || n < 0) return fail(ctx, GNNB_ERR_INVALID, "negative size");
    if (B == 0) return GNNB_OK;
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    {
        ProfScope ps(ctx, GNNB_K_ARGMAX, B, st);
        masked_topk(scores, mask, n, B, k, top_score, top_idx, st, &ctx->launches);
    }
    CU(cudaGetLastError());
    return GNNB_OK;
}

int gnnb_babsr(gnnb_ctx* ctx, const gnnb_frontier* in, int32_t sparsest_layer, float decision_threshold,
               const int32_t* random_order, const int32_t* icp_counter_in, int32_t* decision, int32_t* icp_counter_out,
               int32_t* kind, float* scores, void* stream) {
    if (!ctx || !in || !random_order || !decision || !icp_counter_out) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    if (!ctx->have_net) return fail(ctx, GNNB_ERR_STATE, "gnnb_set_network must be called first");
    if (in->B < 0) return fail(ctx, GNNB_ERR_INVALID, "negative batch");
    if (in->B == 0) return GNNB_OK;
    if (!in->lb || !in->ub || !in->wp || !in->mask) return fail(ctx, GNNB_ERR_INVALID, "null frontier field");
    const int L = (int)ctx->layers.size(), B = in->B;
    if (L > babsr_max_layers()) return fail(ctx, GNNB_ERR_UNSUPPORTED, "too many layers for the BaBSR kernel");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const bool host = in->mem == GNNB_MEM_HOST;
    const std::vector<int>& n = ctx->n;
    int nmax = 0;
    for (int k = 0; k <= L; ++k) nmax = n[k] > nmax ? n[k] : nmax;
    // host buffers: one temporary device block for the inputs and results of this call (this entry is not the hot path)
    float* tmp = nullptr;
    std::vector<const float*> ptrs(2 * (L + 2), nullptr);
    const float *d_wp = in->wp, *d_mask = in->mask;
    const int32_t* d_cin = icp_counter_in;
    int32_t *d_dec = decision, *d_cout = icp_counter_out, *d_kind = kind;
    float* d_scores = scores;
    if (host) {
        size_t total = 0;
        auto take = [&](size_t elems) { size_t o = total; total += align4(elems); return o; };
        std::vector<size_t> o_lb(L + 2), o_ub(L + 2);
        for (int k = 1; k <= L; ++k) { o_lb[k] = take((size_t)B * n[k]); o_ub[k] = take((size_t)B * n[k]); }
        const size_t o_wp = take((size_t)B * n[L]), o_mask = take((size_t)B * ctx->n_hidden), o_cin = take(B), o_dec = take(2 * (size_t)B),
                     o_cout = take(B), o_kind = take(B), o_sc = take(scores ? (size_t)B * ctx->n_hidden : 0);
        CU(cudaMalloc(&tmp, total * sizeof(float)));
        auto up = [&](size_t off, const void* src, size_t elems) {
            cudaMemcpyAsync(tmp + off, src, elems * sizeof(float), cudaMemcpyHostToDevice, st);
            return tmp + off;
        };
        for (int k = 1; k <= L; ++k) {
            if (!in->lb[k] || !in->ub[k]) { cudaFree(tmp); return fail(ctx, GNNB_ERR_INVALID, "null bound array"); }
            ptrs[k] = up(o_lb[k], in->lb[k], (size_t)B * n[k]);
            ptrs[L + 2 + k] = up(o_ub[k], in->ub[k], (size_t)B * n[k]);
        }
        d_wp = up(o_wp, in->wp, (size_t)B * n[L]);
        d_mask = up(o_mask, in->mask, (size_t)B * ctx->n_hidden);
        d_cin = icp_counter_in ? reinterpret_cast<const int32_t*>(up(o_cin, icp_counter_in, B)) : nullptr;
        d_dec = reinterpret_cast<int32_t*>(tmp + o_dec); d_cout = reinterpret_cast<int32_t*>(tmp + o_cout);
        d_kind = kind ? reinterpret_cast<int32_t*>(tmp + o_kind) : nullptr;
        d_scores = scores ? tmp + o_sc : nullptr;
    } else {
        for (int k = 1; k <= L; ++k) {
            if (!in->lb[k] || !in->ub[k]) return fail(ctx, GNNB_ERR_INVALID, "null bound array");
            ptrs[k] = in->lb[k];
            ptrs[L + 2 + k] = in->ub[k];
        }
    }
    // the pointer table and the preference order change per call: stream-ordered copies from pageable memory return
    // after the source has been read, so the local vectors may go out of scope
    cudaError_t e = cudaMemcpyAsync(ctx->d_ptrs, ptrs.data(), ptrs.size() * sizeof(float*), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->d_random_order, random_order, L * sizeof(int32_t), cudaMemcpyHostToDevice, st);
    int rc = 0;
    if (e == cudaSuccess)
        rc = babsr_run(ctx->d_layers, L, ctx->n_hidden, nmax, ctx->d_ptrs, ctx->d_ptrs + (L + 2), d_wp, d_mask, ctx->d_hidden_off,
                       ctx->d_random_order, d_cin, sparsest_layer, decision_threshold, d_dec, d_cout, d_kind, d_scores, B, st,
                       &ctx->launches);
    if (e == cudaSuccess && rc == 0 && host) {
        cudaMemcpyAsync(decision, d_dec, 2 * (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, st);
        cudaMemcpyAsync(icp_counter_out, d_cout, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, st);
        if (kind) cudaMemcpyAsync(kind, d_kind, (size_t)B * sizeof(int32_t), cudaMemcpyDeviceToHost, st);
        if (scores) cudaMemcpyAsync(scores, d_scores, (size_t)B * ctx->n_hidden * sizeof(float), cudaMemcpyDeviceToHost, st);
        e = cudaStreamSynchronize(st);
    }
    if (tmp) { cudaStreamSynchronize(st); cudaFree(tmp); }
    if (e != cudaSuccess) return fail(ctx, GNNB_ERR_CUDA, std::string("gnnb_babsr: ") + cudaGetErrorString(e));
    if (rc != 0) return fail(ctx, GNNB_ERR_UNSUPPORTED, "a layer is too large for the BaBSR kernel's shared-memory buffers");
    CU(cudaGetLastError());
    return GNNB_OK;
}

// tape of one wave of the gradient pass with option grad_chunk = 0 (about 25 MB per base subdomain: ~170 per wave)
static const size_t GRAD_TAPE_BYTES = size_t(4) << 30;

// argument checks of gnnb_score_grad(_device) that need no term values; *ti = the frontier's arrays
static int grad_args(gnnb_ctx* ctx, const gnnb_frontier* in, int32_t n_terms, GnnInputs* ti) {
    if (!ctx->have_gnn || !ctx->have_net) return fail(ctx, GNNB_ERR_STATE, "gnnb_set_gnn_weights and gnnb_set_network must be called first");
    if (in->B < 1 || n_terms < 1) return fail(ctx, GNNB_ERR_INVALID, "need at least one subdomain and one term");
    TRY(check_zero_taps(ctx));
    return frontier_inputs(ctx, in, false, ti);
}

// host frontier: copy its arrays into one temporary device block *tmp (the caller frees it after synchronising `st`) and point
// *ti at them
static int stage_grad_frontier(gnnb_ctx* ctx, const gnnb_frontier* in, GnnInputs* ti, float** tmp, cudaStream_t st) {
    const int B = in->B;
    size_t total = 0;
    walk_inputs(*in, *ti, ctx->n, [&](const float*, const float*&, int64_t per) { total += align4((size_t)B * per); });
    CU(cudaMalloc(tmp, total * sizeof(float)));
    float* dst = *tmp;
    walk_inputs(*in, *ti, ctx->n, [&](const float* src, const float*& slot, int64_t per) {
        cudaMemcpyAsync(dst, src, (size_t)B * per * sizeof(float), cudaMemcpyHostToDevice, st);
        slot = dst;
        dst += align4((size_t)B * per);
    });
    CU(cudaGetLastError());
    return GNNB_OK;
}

// The gradient pass over device terms.  in: device arrays of the frontier's B subdomains.  The subdomains some active term
// names are listed on the device; the count is read back (one synchronise of `st`), and those subdomains run through the
// taped forward and the backward in waves of at most W, each gathered into staging rows of the arena first.
static int score_grad_impl(gnnb_ctx* ctx, GnnInputs& in, int B, int n_terms, const int32_t* term_domain, const int32_t* term_index,
                           const float* term_coeff, float* term_scores, cudaStream_t st) {
    const int L = (int)ctx->layers.size();
    TRY(ensure_kw_iscratch(ctx, B, st));
    int32_t* cnt = ctx->kw_iscratch;                     // [named, bad | flag [B] | list [B] | row_of [B]]
    int32_t *flag = cnt + 2, *list = flag + B, *row_of = list + B;
    CU(cudaMemsetAsync(cnt, 0, (2 + (size_t)B) * sizeof(int32_t), st));
    // optimizer.zero_grad() (graph_score_online.py:73), then loss.backward()
    CU(cudaMemsetAsync(ctx->d_train + ctx->n_params, 0, (size_t)ctx->n_params * sizeof(float), st));
    name_terms(term_domain, term_index, n_terms, B, ctx->n_hidden, term_scores, cnt, flag, list, row_of, st, &ctx->launches);
    int32_t hc[2] = {0, 0};
    CU(cudaMemcpyAsync(hc, cnt, sizeof hc, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const int named = hc[0];
    ctx->grad_bad_terms = hc[1];
    ctx->grad_ws_domains = 0;
    if (named == 0) return GNNB_OK;
    size_t W = (size_t)ctx->grad_chunk;
    if (W == 0) W = std::max<size_t>(1, GRAD_TAPE_BYTES / (sizeof(float) * train_tape_floats(ctx->n, ctx->gp.T, 1)));
    W = std::min<size_t>(W, (size_t)named);
    // arena: tape of a wave | the wave's input rows, in walk_inputs order | their gather table
    auto align64 = [](size_t x) { return (x + 63) & ~size_t(63); };
    size_t total = align64(train_tape_floats(ctx->n, ctx->gp.T, (int)W));
    std::vector<RowGather> tab;
    std::vector<size_t> off;
    walk_inputs(gnnb_frontier{}, in, ctx->n, [&](const float*, const float*& src, int64_t per) {
        tab.push_back(RowGather{src, nullptr, per});
        off.push_back(total);
        total += align64(W * per);
    });
    const size_t o_tab = total;
    total += align64((tab.size() * sizeof(RowGather) + sizeof(float) - 1) / sizeof(float));
    if (ctx->train_ws_cap < total) {
        if (ctx->train_ws) { CU(cudaStreamSynchronize(st)); cudaFree(ctx->train_ws); }
        ctx->train_ws = nullptr; ctx->train_ws_cap = 0;
        CU(cudaMalloc(&ctx->train_ws, total * sizeof(float)));
        ctx->train_ws_cap = total;
    }
    GnnInputs cp(L);
    size_t i = 0;
    walk_inputs(gnnb_frontier{}, cp, ctx->n, [&](const float*, const float*& slot, int64_t) {
        tab[i].dst = ctx->train_ws + off[i];
        slot = tab[i++].dst;
    });
    RowGather* d_tab = reinterpret_cast<RowGather*>(ctx->train_ws + o_tab);
    // a stream-ordered copy from pageable memory returns after the source has been read: `tab` may go out of scope
    CU(cudaMemcpyAsync(d_tab, tab.data(), tab.size() * sizeof(RowGather), cudaMemcpyHostToDevice, st));
    const TrainParams tp = train_params(ctx);
    for (int row0 = 0, Bw = 0; row0 < named; row0 += Bw) {
        Bw = std::min((int)W, named - row0);
        gather_rows(d_tab, (int)tab.size(), list + row0, Bw, st, &ctx->launches);
        const WaveTerms wt{term_domain, term_index, term_coeff, row_of, n_terms, B, ctx->n_hidden, row0, term_scores};
        const int e = train_wave(ctx->gp, tp, ctx->layers, ctx->n, ctx->hidden_off, cp, (int)W, Bw, wt, ctx->train_ws, st,
                                 &ctx->launches);
        if (e != cudaSuccess) return fail(ctx, GNNB_ERR_CUDA, std::string("gradient pass: ") + cudaGetErrorString((cudaError_t)e));
    }
    ctx->grad_ws_domains = (int)W;
    return GNNB_OK;
}

int gnnb_score_grad_device(gnnb_ctx* ctx, const gnnb_frontier* in, int32_t n_terms, const int32_t* term_domain,
                           const int32_t* term_index, const float* term_coeff, float* term_scores, void* stream) {
    if (!ctx || !in || !term_domain || !term_index || !term_coeff || !term_scores) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    GnnInputs ti((int)ctx->layers.size());
    TRY(grad_args(ctx, in, n_terms, &ti));
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    float* tmp = nullptr;
    int rc = in->mem == GNNB_MEM_HOST ? stage_grad_frontier(ctx, in, &ti, &tmp, st) : GNNB_OK;
    if (rc == GNNB_OK) rc = score_grad_impl(ctx, ti, in->B, n_terms, term_domain, term_index, term_coeff, term_scores, st);
    if (tmp) { cudaStreamSynchronize(st); cudaFree(tmp); }
    return rc;
}

int gnnb_score_grad(gnnb_ctx* ctx, const gnnb_frontier* in, int32_t n_terms, const int32_t* term_domain, const int32_t* term_index,
                    const float* term_coeff, float* term_scores, void* stream) {
    if (!ctx || !in || !term_domain || !term_index || !term_coeff) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    GnnInputs ti((int)ctx->layers.size());
    TRY(grad_args(ctx, in, n_terms, &ti));
    for (int i = 0; i < n_terms; ++i)
        if (term_domain[i] < 0 || term_domain[i] >= in->B || term_index[i] < 0 || term_index[i] >= ctx->n_hidden)
            return fail(ctx, GNNB_ERR_INVALID, "term " + std::to_string(i) + " is out of range");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    // the terms in, their scores out: one temporary device block [domain | index | coeff | scores] (this entry is not the hot path)
    const size_t nt = (size_t)n_terms;
    int32_t* d_terms = nullptr;
    CU(cudaMalloc(&d_terms, 4 * nt * sizeof(int32_t)));
    float* d_coeff = reinterpret_cast<float*>(d_terms + 2 * nt);
    float* d_scores = d_coeff + nt;
    float* tmp = nullptr;
    cudaError_t e = cudaMemcpyAsync(d_terms, term_domain, nt * sizeof(int32_t), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_terms + nt, term_index, nt * sizeof(int32_t), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_coeff, term_coeff, nt * sizeof(float), cudaMemcpyHostToDevice, st);
    int rc = e == cudaSuccess ? GNNB_OK : fail(ctx, GNNB_ERR_CUDA, std::string("copying the terms: ") + cudaGetErrorString(e));
    if (rc == GNNB_OK && in->mem == GNNB_MEM_HOST) rc = stage_grad_frontier(ctx, in, &ti, &tmp, st);
    if (rc == GNNB_OK) rc = score_grad_impl(ctx, ti, in->B, n_terms, d_terms, d_terms + nt, d_coeff, d_scores, st);
    if (rc == GNNB_OK && term_scores) {
        e = cudaMemcpyAsync(term_scores, d_scores, nt * sizeof(float), cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) rc = fail(ctx, GNNB_ERR_CUDA, std::string("copying the term scores: ") + cudaGetErrorString(e));
    }
    e = cudaStreamSynchronize(st);          // returns after the gradients are complete
    if (rc == GNNB_OK && e != cudaSuccess) rc = fail(ctx, GNNB_ERR_CUDA, std::string("gradient pass: ") + cudaGetErrorString(e));
    if (tmp) cudaFree(tmp);
    cudaFree(d_terms);
    return rc;
}

int gnnb_get_gradients(gnnb_ctx* ctx, float* const* tensors, const int64_t* numels, int n_tensors) {
    return download_quarter(ctx, 1, tensors, numels, n_tensors);
}

int gnnb_get_gnn_weights(gnnb_ctx* ctx, float* const* tensors, const int64_t* numels, int n_tensors) {
    return download_quarter(ctx, 0, tensors, numels, n_tensors);
}

int gnnb_adam_step(gnnb_ctx* ctx, float lr, float beta1, float beta2, float eps, float weight_decay, void* stream) {
    if (!ctx) return GNNB_ERR_INVALID;
    if (!ctx->have_gnn) return fail(ctx, GNNB_ERR_STATE, "gnnb_set_gnn_weights must be called first");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t np = (size_t)ctx->n_params;
    ++ctx->adam_steps;
    adam_step(ctx->d_train, ctx->d_train + np, ctx->d_train + 2 * np, ctx->d_train + 3 * np, ctx->n_params, lr, beta1, beta2, eps,
              weight_decay, ctx->adam_steps, st, &ctx->launches);
    // every derived form of the parameters (transposed, composed, tensor-core planes) is rebuilt from the new master copy
    std::vector<float> host(np);
    CU(cudaMemcpyAsync(host.data(), ctx->d_train, np * sizeof(float), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    std::vector<const float*> tensors(2 * N_LIN);
    for (int l = 0; l < N_LIN; ++l) { tensors[2 * l] = &host[ctx->po_w[l]]; tensors[2 * l + 1] = &host[ctx->po_b[l]]; }
    return upload_gnn(ctx, tensors.data(), ctx->gp.T);
}

int gnnb_adam_reset(gnnb_ctx* ctx) {
    if (!ctx) return GNNB_ERR_INVALID;
    ctx->adam_steps = 0;
    if (ctx->d_train) {
        CU(cudaSetDevice(ctx->device));
        CU(cudaMemset(ctx->d_train + 2 * (size_t)ctx->n_params, 0, 2 * (size_t)ctx->n_params * sizeof(float)));
    }
    return GNNB_OK;
}


int gnnb_queue_create(gnnb_ctx* ctx, int64_t capacity, gnnb_queue** out) {
    if (!ctx || !out || capacity < 1) return fail(ctx, GNNB_ERR_INVALID, "bad argument");
    *out = nullptr;
    if (!ctx->have_net) return fail(ctx, GNNB_ERR_STATE, "gnnb_set_network must be called first");
    if (capacity > 0x7fffffff) return fail(ctx, GNNB_ERR_INVALID, "capacity must fit 31 bits");
    std::string err;
    DomainQueue* q = nullptr;
    const int rc = queue_create(ctx->device, ctx->n, ctx->n_hidden, capacity, &q, &err);
    if (rc != GNNB_OK) return fail(ctx, rc, err);
    *out = new gnnb_queue{ctx, q};
    ctx->queues.push_back(*out);
    return GNNB_OK;
}

void gnnb_queue_destroy(gnnb_queue* q) {
    if (!q) return;
    queue_destroy(q->q);
    if (q->ctx) {
        auto& v = q->ctx->queues;
        for (size_t i = 0; i < v.size(); ++i) if (v[i] == q) { v.erase(v.begin() + i); break; }
    }
    delete q;
}

namespace {
// device views of a gnnb_domains batch: the caller's pointers (DEVICE) or a staged copy (HOST; `to_device` copies in)
struct DomView {
    std::vector<float*> lb, ub;
    float *lower = nullptr, *upper = nullptr;
    int8_t* mask = nullptr;
    int32_t* dec = nullptr;
    uint8_t* keep = nullptr;
};
int view_domains(gnnb_queue* q, const gnnb_domains* d, const uint8_t* keep, bool to_device, DomView* v, cudaStream_t st) {
    gnnb_ctx* ctx = q->ctx;
    const int L = (int)ctx->layers.size(), B = d->B;
    v->lb.assign(L + 2, nullptr); v->ub.assign(L + 2, nullptr);
    if (d->mem != GNNB_MEM_HOST) {
        for (int k = 0; k <= L + 1; ++k) { v->lb[k] = d->lb ? d->lb[k] : nullptr; v->ub[k] = d->ub ? d->ub[k] : nullptr; }
        v->lower = d->lower_bound; v->upper = d->upper_bound; v->mask = d->mask; v->dec = d->decision; v->keep = const_cast<uint8_t*>(keep);
        return GNNB_OK;
    }
    size_t floats = 0;
    for (int k = 0; k <= L + 1; ++k) floats += 2 * align4((size_t)B * ctx->n[k]);
    floats += 2 * align4(B) + align4(2 * (size_t)B) + align4(((size_t)B * ctx->n_hidden + 3) / 4) + align4(((size_t)B + 3) / 4);
    float* base = queue_stage(q->q, floats * sizeof(float));
    if (!base) return fail(ctx, GNNB_ERR_CUDA, queue_error(q->q));
    size_t o = 0;
    auto take = [&](size_t elems) { float* p = base + o; o += align4(elems); return p; };
    auto up = [&](void* dst, const void* src, size_t bytes) { if (to_device && src) cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st); };
    for (int k = 0; k <= L + 1; ++k) {
        v->lb[k] = take((size_t)B * ctx->n[k]); v->ub[k] = take((size_t)B * ctx->n[k]);
        up(v->lb[k], d->lb ? d->lb[k] : nullptr, (size_t)B * ctx->n[k] * sizeof(float));
        up(v->ub[k], d->ub ? d->ub[k] : nullptr, (size_t)B * ctx->n[k] * sizeof(float));
    }
    v->lower = take(B); v->upper = take(B);
    up(v->lower, d->lower_bound, B * sizeof(float)); up(v->upper, d->upper_bound, B * sizeof(float));
    v->dec = reinterpret_cast<int32_t*>(take(2 * (size_t)B));
    if (to_device && !d->decision) v->dec = nullptr; else up(v->dec, d->decision, 2 * (size_t)B * sizeof(int32_t));
    v->mask = reinterpret_cast<int8_t*>(take(((size_t)B * ctx->n_hidden + 3) / 4));
    up(v->mask, d->mask, (size_t)B * ctx->n_hidden);
    v->keep = nullptr;
    if (keep) { v->keep = reinterpret_cast<uint8_t*>(take(((size_t)B + 3) / 4)); up(v->keep, keep, B); }
    return GNNB_OK;
}
}  // namespace

int gnnb_queue_add(gnnb_queue* q, const gnnb_domains* d, const uint8_t* keep, int32_t* added, void* stream) {
    if (!q || !d || !added || !q->ctx) return GNNB_ERR_INVALID;
    gnnb_ctx* ctx = q->ctx;
    *added = 0;
    if (d->B < 0) return fail(ctx, GNNB_ERR_INVALID, "negative batch");
    if (d->B == 0) return GNNB_OK;
    if (!d->lower_bound || !d->upper_bound || !d->lb || !d->ub || !d->mask) return fail(ctx, GNNB_ERR_INVALID, "null domain field");
    const int L = (int)ctx->layers.size();
    for (int k = 0; k <= L + 1; ++k) if (!d->lb[k] || !d->ub[k]) return fail(ctx, GNNB_ERR_INVALID, "null bound array");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    DomView v;
    TRY(view_domains(q, d, keep, true, &v, st));
    const int rc = queue_add(q->q, d->B, v.lower, v.upper, v.lb.data(), v.ub.data(), v.mask, v.dec, v.keep, added, st, &ctx->launches);
    if (rc != GNNB_OK) return fail(ctx, rc, queue_error(q->q));
    if (d->mem == GNNB_MEM_HOST) CU(cudaStreamSynchronize(st));      // the staging block is reused by the next call
    return GNNB_OK;
}

int gnnb_queue_pick(gnnb_queue* q, float threshold, int32_t discard_rest, gnnb_domains* out, int32_t* picked, void* stream) {
    if (!q || !out || !picked || !q->ctx) return GNNB_ERR_INVALID;
    gnnb_ctx* ctx = q->ctx;
    *picked = 0;
    if (out->B < 0) return fail(ctx, GNNB_ERR_INVALID, "negative batch");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    const int L = (int)ctx->layers.size();
    DomView v;
    TRY(view_domains(q, out, nullptr, false, &v, st));
    const bool host = out->mem == GNNB_MEM_HOST;
    if (host) {      // only the fields the caller asked for
        if (!out->lower_bound) v.lower = nullptr;
        if (!out->upper_bound) v.upper = nullptr;
        if (!out->mask) v.mask = nullptr;
        if (!out->decision) v.dec = nullptr;
        for (int k = 0; k <= L + 1; ++k) { if (!out->lb || !out->lb[k]) v.lb[k] = nullptr; if (!out->ub || !out->ub[k]) v.ub[k] = nullptr; }
    }
    const int rc = queue_pick(q->q, out->B, threshold, discard_rest != 0, picked, v.lower, v.upper, v.lb.data(), v.ub.data(), v.mask, v.dec, st,
                              &ctx->launches);
    if (rc != GNNB_OK) return fail(ctx, rc, queue_error(q->q));
    if (host && *picked > 0) {
        const size_t n = (size_t)*picked;
        auto down = [&](void* dst, const void* src, size_t bytes) { if (dst && src) cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st); };
        for (int k = 0; k <= L + 1; ++k) {
            down(out->lb ? out->lb[k] : nullptr, v.lb[k], n * ctx->n[k] * sizeof(float));
            down(out->ub ? out->ub[k] : nullptr, v.ub[k], n * ctx->n[k] * sizeof(float));
        }
        down(out->lower_bound, v.lower, n * sizeof(float)); down(out->upper_bound, v.upper, n * sizeof(float));
        down(out->mask, v.mask, n * ctx->n_hidden); down(out->decision, v.dec, 2 * n * sizeof(int32_t));
        CU(cudaStreamSynchronize(st));
    }
    return GNNB_OK;
}

int gnnb_queue_prune(gnnb_queue* q, float threshold, void* stream) {
    if (!q || !q->ctx) return GNNB_ERR_INVALID;
    gnnb_ctx* ctx = q->ctx;
    CU(cudaSetDevice(ctx->device));
    const int rc = queue_prune(q->q, threshold, (cudaStream_t)stream, &ctx->launches);
    if (rc != GNNB_OK) return fail(ctx, rc, queue_error(q->q));
    return GNNB_OK;
}

int gnnb_queue_stats(gnnb_queue* q, int64_t* size, float* global_lb, void* stream) {
    if (!q || !q->ctx) return GNNB_ERR_INVALID;
    gnnb_ctx* ctx = q->ctx;
    if (size) *size = queue_size(q->q);
    if (global_lb && queue_size(q->q) > 0) {
        CU(cudaSetDevice(ctx->device));
        const int rc = queue_global_lb(q->q, global_lb, (cudaStream_t)stream);
        if (rc != GNNB_OK) return fail(ctx, rc, queue_error(q->q));
    }
    return GNNB_OK;
}

int gnnb_kw_bounds(gnnb_ctx* ctx, int32_t B, const float* x, float eps, const float* wp, const float* bp, const float* const* provided_lb,
                   const float* const* provided_ub, float* const* out_lb, float* const* out_ub, void* stream) {
    if (!ctx || !x || !wp || !bp || !out_lb || !out_ub) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    if (!ctx->have_net) return fail(ctx, GNNB_ERR_STATE, "gnnb_set_network must be called first");
    if (B < 1) return fail(ctx, GNNB_ERR_INVALID, "need at least one domain");
    if ((provided_lb == nullptr) != (provided_ub == nullptr)) return fail(ctx, GNNB_ERR_INVALID, "provide both lower and upper bounds or neither");
    const int L = (int)ctx->layers.size();
    for (int k = 0; k <= L + 1; ++k) if (!out_lb[k] || !out_ub[k]) return fail(ctx, GNNB_ERR_INVALID, "null output array");
    if (provided_lb)
        for (int k = 0; k < L; ++k) if (!provided_lb[k] || !provided_ub[k]) return fail(ctx, GNNB_ERR_INVALID, "null provided-bounds array");
    CU(cudaSetDevice(ctx->device));
    std::string err;
    const KwTc tc{&ctx->plan_kw, &ctx->rowmap};
    const int rc = kw_bounds(ctx->layers, ctx->n, B, x, eps, wp, bp, provided_lb, provided_ub, out_lb, out_ub,
                             ctx->math == GNNB_MATH_TC_FP16X3 ? &tc : nullptr, &ctx->kw_ws, &ctx->kw_ws_cap, (cudaStream_t)stream, &ctx->launches, &err);
    if (rc != GNNB_OK) return fail(ctx, rc, err);
    return GNNB_OK;
}

int gnnb_child_bounds(gnnb_ctx* ctx, int32_t B, const float* x, float eps, const float* wp, const float* bp, const float* const* parent_lb,
                      const float* const* parent_ub, const int32_t* dec_layer, const int32_t* dec_index, const int32_t* choice,
                      float* const* out_lb, float* const* out_ub, int8_t* const* out_mask, int32_t* second_pass, void* stream) {
    if (!ctx || !x || !wp || !bp || !parent_lb || !parent_ub || !dec_layer || !dec_index || !choice || !out_lb || !out_ub)
        return fail(ctx, GNNB_ERR_INVALID, "null argument");
    if (!ctx->have_net) return fail(ctx, GNNB_ERR_STATE, "gnnb_set_network must be called first");
    if (B < 1) return fail(ctx, GNNB_ERR_INVALID, "need at least one domain");
    const int L = (int)ctx->layers.size();
    for (int k = 0; k <= L + 1; ++k)
        if (!out_lb[k] || !out_ub[k] || !parent_lb[k] || !parent_ub[k]) return fail(ctx, GNNB_ERR_INVALID, "null bounds array");
    if (out_mask)
        for (int k = 0; k < L; ++k) if (!out_mask[k]) return fail(ctx, GNNB_ERR_INVALID, "null mask array");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    TRY(ensure_kw_iscratch(ctx, B, st));
    std::string err;
    const KwTc tc{&ctx->plan_kw, &ctx->rowmap};
    const int rc = child_bounds(ctx->layers, ctx->n, B, x, eps, wp, bp, parent_lb, parent_ub, dec_layer, dec_index, choice, out_lb, out_ub, out_mask,
                                second_pass, ctx->kw_iscratch, ctx->math == GNNB_MATH_TC_FP16X3 ? &tc : nullptr, &ctx->kw_ws, &ctx->kw_ws_cap, st,
                                &ctx->launches, &err);
    if (rc != GNNB_OK) return fail(ctx, rc, err);
    return GNNB_OK;
}

int gnnb_root_bounds(gnnb_ctx* ctx, int32_t B, const float* x, float eps, const float* wp, const float* bp, float* const* out_lb,
                     float* const* out_ub, int8_t* const* out_mask, int32_t* second_pass, void* stream) {
    if (!ctx || !x || !wp || !bp || !out_lb || !out_ub) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    if (!ctx->have_net) return fail(ctx, GNNB_ERR_STATE, "gnnb_set_network must be called first");
    if (B < 1) return fail(ctx, GNNB_ERR_INVALID, "need at least one domain");
    const int L = (int)ctx->layers.size();
    for (int k = 0; k <= L + 1; ++k) if (!out_lb[k] || !out_ub[k]) return fail(ctx, GNNB_ERR_INVALID, "null bounds array");
    if (out_mask)
        for (int k = 0; k < L; ++k) if (!out_mask[k]) return fail(ctx, GNNB_ERR_INVALID, "null mask array");
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    TRY(ensure_kw_iscratch(ctx, B, st));
    std::string err;
    const KwTc tc{&ctx->plan_kw, &ctx->rowmap};
    const int rc = root_bounds(ctx->layers, ctx->n, B, x, eps, wp, bp, out_lb, out_ub, out_mask, second_pass, ctx->kw_iscratch,
                               ctx->math == GNNB_MATH_TC_FP16X3 ? &tc : nullptr, &ctx->kw_ws, &ctx->kw_ws_cap, st, &ctx->launches, &err);
    if (rc != GNNB_OK) return fail(ctx, rc, err);
    return GNNB_OK;
}

int gnnb_check(gnnb_ctx* ctx, void* stream, int64_t* nan_count) {
    if (!ctx) return GNNB_ERR_INVALID;
    CU(cudaSetDevice(ctx->device));
    cudaStream_t st = (cudaStream_t)stream;
    unsigned long long h = 0;
    CU(cudaMemcpyAsync(&h, ctx->d_nan, sizeof h, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (nan_count) *nan_count = (int64_t)h;
    if (h != 0) {
        CU(cudaMemsetAsync(ctx->d_nan, 0, sizeof h, st));
        return fail(ctx, GNNB_ERR_NAN, "mu contains nan (" + std::to_string(h) + " tiles)");
    }
    return GNNB_OK;
}

int64_t gnnb_launch_count(gnnb_ctx* ctx) { return ctx ? ctx->launches : -1; }

int gnnb_last_error(gnnb_ctx* ctx, char* buf, int n) {
    if (!ctx) return GNNB_ERR_INVALID;
    if (buf && n > 0) {
        strncpy(buf, ctx->err.c_str(), (size_t)n - 1);
        buf[n - 1] = 0;
    }
    return ctx->last_status;
}

int gnnb_profile_read(gnnb_ctx* ctx, int klass, double* ms, int64_t* launches, int64_t* rows) {
    if (!ctx || klass < 0 || klass >= GNNB_K_COUNT) return fail(ctx, GNNB_ERR_INVALID, "bad kernel class");
    CU(cudaSetDevice(ctx->device));
    TRY(prof_collect(ctx));
    if (ms) *ms = ctx->prof_ms[klass];
    if (launches) *launches = ctx->prof_launches[klass];
    if (rows) *rows = ctx->prof_rows[klass];
    return GNNB_OK;
}

int gnnb_profile_reset(gnnb_ctx* ctx) {
    if (!ctx) return GNNB_ERR_INVALID;
    CU(cudaSetDevice(ctx->device));
    TRY(prof_collect(ctx));
    for (int k = 0; k < GNNB_K_COUNT; ++k) { ctx->prof_ms[k] = 0; ctx->prof_launches[k] = 0; ctx->prof_rows[k] = 0; }
    return GNNB_OK;
}

int gnnb_debug_snapshot(gnnb_ctx* ctx, const char* name, float* dst, int64_t max_numel, int64_t* numel) {
    if (!ctx || !name) return fail(ctx, GNNB_ERR_INVALID, "null argument");
    auto it = ctx->snaps.find(name);
    if (it == ctx->snaps.end()) return fail(ctx, GNNB_ERR_INVALID, std::string("no snapshot named ") + name);
    if (numel) *numel = it->second.second;
    if (!dst) return GNNB_OK;
    if (max_numel < it->second.second) return fail(ctx, GNNB_ERR_INVALID, "snapshot buffer too small");
    CU(cudaSetDevice(ctx->device));
    CU(cudaDeviceSynchronize());
    CU(cudaMemcpy(dst, it->second.first, (size_t)it->second.second * sizeof(float), cudaMemcpyDeviceToHost));
    return GNNB_OK;
}

}  // extern "C"
