/*
 * gnnb.h — C ABI of libgnnb.so: B200-native batched GNN branching scores.
 *
 * Drop-in boundary for the GNN ReLU-scoring hot path of oval-group/GNN_branching.  The reference has no
 * FFI layer; its boundary is the Python class API (graphnet/graph_conv.py:473-483 GraphNet,
 * graphnet/graph_score.py:8-56 GraphChoice).  Each entry point below names the reference interface it
 * replaces; gnn_branching_b200/graph_conv.py and graph_score.py bind them with ctypes and keep the
 * reference's Python signatures.  See INTEGRATION.md for the binding a reference maintainer would add.
 *
 * Conventions: plain pointers and sizes only; every function returns a status (0 = ok) and never throws;
 * the context is bound to one CUDA device and is not re-entrant; all fp32, indices int32.
 */
#ifndef GNNB_H
#define GNNB_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct gnnb_ctx gnnb_ctx;

enum gnnb_status {
    GNNB_OK = 0,
    GNNB_ERR_INVALID = 1,      /* bad argument / shape mismatch */
    GNNB_ERR_CUDA = 2,         /* a CUDA runtime call failed (message in gnnb_last_error) */
    GNNB_ERR_STATE = 3,        /* weights or network not set */
    GNNB_ERR_NAN = 4,          /* NaN appeared in an embedding: the reference stops in pdb here
                                  (graphnet/graph_conv.py:184-186, 339-341); outputs are still written.  In tensor-core mode
                                  this includes activations beyond the fp16 operand range (|x| >= 524 288), unless option
                                  "rescore" scores those subdomains again in exact fp32 */
    GNNB_ERR_UNSUPPORTED = 5
};

enum gnnb_layer_kind { GNNB_LAYER_CONV = 0, GNNB_LAYER_LINEAR = 1 };
enum gnnb_mem_kind { GNNB_MEM_DEVICE = 0, GNNB_MEM_HOST = 1 };

/* Arithmetic of the per-node MLP GEMMs.  Both are sm_100a CUDA; TC is the product path, SIMT the
 * exact-fp32 validation path used by the tests to localise tensor-path errors. */
enum gnnb_math_mode {
    GNNB_MATH_TC_FP16X3 = 0,   /* tcgen05.mma kind::f16, fp16 hi/lo split, 3 MMAs, fp32 accumulate in TMEM */
    GNNB_MATH_SIMT_FP32 = 1    /* fp32 FMA on CUDA cores */
};

/* Kernel classes of the stage schedule, for gnnb_profile_read. */
enum gnnb_kernel_class {
    GNNB_K_RELAX = 0,          /* round-independent relaxation-feature MLPs of a hidden layer */
    GNNB_K_UPDATE_FWD,         /* forward-sweep node update (fc3, fc3_2, fc4, fc4_2) */
    GNNB_K_UPDATE_BWD,         /* backward-sweep node update (bc3, bc3_1, bc4, bc4_1) */
    GNNB_K_UPDATE_BWD_SCORE,   /* last backward sweep: node update + score head (fnode, fscore) */
    GNNB_K_INPUT_EMBED,        /* input-node embedding, round 0 */
    GNNB_K_INPUT_UPDATE,       /* input-node backward update, rounds < T-1 */
    GNNB_K_PROP_FWD,           /* embeddings through A_k (conv / linear) */
    GNNB_K_PROP_BWD,           /* embeddings through A_k^T (transposed conv / linear / property rank-1) */
    GNNB_K_OUTPUT,             /* output node */
    GNNB_K_ARGMAX,             /* masked argmax per subdomain */
    GNNB_K_LAYER_FWD,          /* fused launch: propagation through A_k + forward node update (option "fuse") */
    GNNB_K_LAYER_BWD,          /* fused launch: propagation through A_{k+1}^T + backward node update */
    GNNB_K_LAYER_BWD_SCORE,    /* the same on the last backward sweep, with the score head */
    GNNB_K_COUNT
};

/* One edge set A_k of the graph = one conv / linear layer of the verified network followed by a ReLU
 * (reference: layers['fixed_layers'], graphnet/graph_conv.py:107-137).  Weight and bias are HOST pointers,
 * copied (and repacked) by gnnb_set_network. */
typedef struct {
    int32_t kind;                        /* gnnb_layer_kind */
    int32_t c_in, h_in, w_in;            /* conv input shape (linear: c_in = n_in, h_in = w_in = 1) */
    int32_t c_out, h_out, w_out;         /* conv output shape (linear: c_out = n_out, 1, 1) */
    int32_t ksize, stride, pad;          /* conv only (square kernels) */
    const float* weight;                 /* conv [c_out, c_in, k, k]; linear [n_out, n_in] (nn.Linear layout) */
    const float* bias;                   /* [c_out] */
} gnnb_layer_desc;

/* A frontier of B subdomains, struct-of-arrays, node index within a layer = PyTorch NCHW flatten
 * (reference: the argument lists of GraphNet.forward, graphnet/graph_conv.py:479; SURVEY §8a row a1).
 * All pointers live in the memory space named by `mem` (device, or host — pinned for full copy speed). */
typedef struct {
    int32_t B;
    int32_t mem;                         /* gnnb_mem_kind of every pointer below AND of gnnb_score's outputs */
    const float* const* lb;              /* L+2 arrays [B, n_k]: k = 0 input, 1..L hidden pre-ReLU, L+1 output */
    const float* const* ub;              /* L+2 arrays [B, n_k] */
    const float* const* dual;            /* L arrays [B, n_k, 3]   (dual_vars) */
    const float* const* prim_pre;        /* L arrays [B, n_k]      (primals[i_k]) */
    const float* const* prim_post;       /* L arrays [B, n_k]      (primals[i_k + 1]) */
    const float* prim_out;               /* [B]                    (primals[-1]) */
    const float* primal_input;           /* [B, n_0]               (primal_inputs) */
    const float* wp;                     /* [B, n_L] property layer weights (layers['prop_layers'][b].weight) */
    const float* bp;                     /* [B]      property layer biases */
    const float* mask;                   /* [B, sum n_k] 0/1, 1 = branching candidate (masks) */
} gnnb_frontier;

/* Create a context on CUDA device `device`.  Replaces GraphChoice.__init__'s `.cuda()` (graph_score.py:13). */
int gnnb_create(gnnb_ctx** out, int device);
void gnnb_destroy(gnnb_ctx* ctx);

/* Load the GNN parameters: 52 HOST fp32 tensors in state_dict order — for each of
 * inp_f, inp_f_1, inp_b, inp_b_1, inp_b2, inp_b2_2, fc1, fc1_1, fc3, fc3_2, fc4, fc4_2, out1, out2, out3,
 * bc1, bc1_1, bc1_2, bc2, bc2_1, bc3, bc3_1, bc4, bc4_1 (EmbedUpdates.update.*), fnode, fscore
 * (ComputeFinalScore.*): weight [out, in] then bias [out].  Replaces model.load_state_dict
 * (graph_score.py:11); T, p are GraphNet's constructor arguments (graph_conv.py:474); p must be 64. */
int gnnb_set_gnn_weights(gnnb_ctx* ctx, const float* const* tensors, const int64_t* numels, int n_tensors,
                         int T, int p);

/* Describe the verified network (the graph).  Replaces the per-call walk over layers['fixed_layers']
 * (graph_conv.py:107-137, 222-249).  Conv layers: conv_transpose2d must land on the input grid (no output_padding) and the
 * weights must fit 64 KB, else GNNB_ERR_UNSUPPORTED.  A conv layer j >= 2 with stride > kernel may leave input positions
 * that no tap reaches; the GNN's backward propagation divides those by a tap count of 0 (0/0 in the reference).  Such a
 * network is accepted, and the KW bounds, BaBSR and the domain queue work on it, but gnnb_score, gnnb_score_winners,
 * gnnb_score_topk and gnnb_score_grad return GNNB_ERR_UNSUPPORTED before enqueuing anything (the message names the layer).
 * Layer 1 may have such positions: its transpose feeds the input nodes and is not normalised. */
int gnnb_set_network(gnnb_ctx* ctx, const gnnb_layer_desc* layers, int n_layers, int c0, int h0, int w0);

/* Options: "math" (gnnb_math_mode), "chunk" (subdomains per wave; 0 = auto), "fuse" (0/1, default 1: propagation and
 * node update of a layer in one launch, tensor-core mode; 0 = two launches), "snapshot" (0/1: keep per-stage copies
 * for gnnb_debug_snapshot; debugging only), "profile" (0/1: time every stage launch with CUDA events for
 * gnnb_profile_read), "rescore" (0/1, default 0; see below).  Any other key of gnnb_set_option fails with GNNB_ERR_INVALID.
 * "rescore" = 1, tensor-core mode: gnnb_score, gnnb_score_winners and gnnb_score_topk record every subdomain in which the
 * tensor-core pass met a NaN (activations beyond the fp16 operand range, |x| >= 524 288), score those subdomains again with the
 * exact-fp32 SIMT schedule on the same GPU and write their results (best score and index, the k best, or winner record, dense
 * scores) over the tensor-core
 * ones; every other subdomain keeps its tensor-core result bit for bit.  Cost on a frontier without such subdomains: one 4-byte
 * device -> host copy and one synchronise of `stream` per call, also with DEVICE buffers (no extra launch or allocation).
 * The NaN count is reset before the fp32 pass, so GNNB_ERR_NAN (returned for HOST calls, through gnnb_check for DEVICE calls)
 * then reports only NaN that exact fp32 gives too.  The option does nothing in SIMT mode; snapshots keep the tensor-core pass.
 * "grad_chunk" (>= 0, default 0): subdomains per wave of gnnb_score_grad(_device); 0 = the most whose activation tape fits
 * 4 GiB.
 * gnnb_get_option also reads these, "rescored" (subdomains the last scoring call scored again), and "n_hidden" (hidden ReLUs of
 * the network), "workspace_domains" (subdomains the
 * workspace holds), "grad_workspace_domains" (subdomains per wave of the last gnnb_score_grad(_device): the tape arena holds
 * at least that many; 0 when no term was active), "grad_bad_terms" (out-of-range terms of the last gnnb_score_grad_device) and "plan_density_pct_f<k>" / "plan_density_pct_b<k>" (percentage of the MACs issued by forward /
 * backward propagation plan k that are useful); it returns -1 for an unknown key. */
int gnnb_set_option(gnnb_ctx* ctx, const char* key, int64_t value);
int64_t gnnb_get_option(gnnb_ctx* ctx, const char* key);

/* Score a frontier.  Replaces GraphNet.forward (graph_conv.py:479-483) + the argmax / index mapping of
 * GraphChoice.decision (graph_score.py:41-47) for B subdomains at once.
 *   best_score [B]   score of the winning ReLU (-inf when the domain has no candidate)
 *   best_idx   [B]   its flat index into the concatenated hidden layers, lowest index on ties, -1 when none
 *   scores     [B, sum n_k] or NULL: dense scores of every hidden ReLU (only rows with mask != 0 are
 *                    what the reference returns)
 * Work is enqueued on `stream` (a cudaStream_t, NULL = default stream).  With mem = HOST the call copies
 * inputs in and results out on that stream and returns after they have landed; with mem = DEVICE it
 * returns without synchronising and GNNB_ERR_NAN is reported by gnnb_check. */
int gnnb_score(gnnb_ctx* ctx, const gnnb_frontier* in, float* best_score, int32_t* best_idx, float* scores,
               void* stream);

/* The same scoring pass with the winners written as packed 8-byte records straight into a buffer a collective can send:
 * the multi-GPU frontier (one context per GPU, contiguous shards) all-gathers exactly these records over NCCL / NVLink
 * (SURVEY 8e), so no pack / pad / concatenate pass runs between the argmax kernel and the collective.
 *   winners    [B] DEVICE records (score, index) — always device memory, also when `in->mem` is HOST (inputs are then
 *              staged host -> device inside the call as in gnnb_score, the records stay on the GPU that scored them)
 * Replaces the same reference lines as gnnb_score (graph_score.py:32-56).  Returns without synchronising when
 * `in->mem` is DEVICE; with HOST inputs it returns after the staged copies and kernels have completed. */
typedef struct gnnb_winner {
    float score;                         /* -inf when the subdomain has no candidate */
    int32_t index;                       /* flat index into the concatenated hidden layers, -1 when none */
} gnnb_winner;
int gnnb_score_winners(gnnb_ctx* ctx, const gnnb_frontier* in, gnnb_winner* winners, float* scores, void* stream);

/* The k best branching candidates per subdomain instead of the best one: what strong branching over the GNN's top candidates
 * (and a caller-side top-k) needs, without the dense [B, sum n_k] scores.  Order, per subdomain: the candidates are the
 * entries with mask != 0 (a -inf score is still a candidate); NaN scores come first in ascending index, then the others by
 * score, descending, equal scores (-0.0 == +0.0) by ascending index; top_score[b, j] is the bit pattern of the score of
 * top_idx[b, j]; slots past the last candidate hold (-inf, -1).  Entry 0 is gnnb_score's (best_score, best_idx) bit for bit.
 * A k outside [1, GNNB_TOPK_MAX], a null output or a negative B fails with GNNB_ERR_INVALID before anything is enqueued. */
#define GNNB_TOPK_MAX 64
/* gnnb_score with the k best candidates per subdomain instead of the best one; order contract above.
 * top_score [B, k] f32, top_idx [B, k] i32 in in->mem (HOST: returns after they have landed);
 * scores [B, sum n_k] or NULL as in gnnb_score.  Same launches as gnnb_score (the last one per wave is the top-k kernel,
 * profiled as GNNB_K_ARGMAX; k = 1 runs the argmax kernel itself); option "rescore" applies as in gnnb_score. */
int gnnb_score_topk(gnnb_ctx* ctx, const gnnb_frontier* in, int32_t k, float* top_score, int32_t* top_idx,
                    float* scores, void* stream);
/* The same selection over caller-provided DEVICE arrays: scores [B, n], mask [B, n] or NULL (= every entry is a
 * candidate).  Enqueues one launch on `stream`; needs no weights or network. */
int gnnb_topk(gnnb_ctx* ctx, int32_t B, int32_t n, const float* scores, const float* mask, int32_t k,
              float* top_score, int32_t* top_idx, void* stream);

/* BaBSR / KW branching heuristic for B subdomains at once.  Replaces choose_node_conv (plnn/kw_score_conv.py:41-156),
 * the hand-written score the reference falls back to when the GNN decision did not improve the bound
 * (plnn/relu_conv_gnnkwthreshold.py:155-157).  Uses `in->lb`, `in->ub` (hidden layers), `in->wp`, `in->mask` and
 * `in->mem`; the other frontier fields may be NULL.
 *   random_order      [L] HOST: layer preference of the last fallback, most preferred last (relu_conv_gnnkwthreshold.py:98-101)
 *   icp_counter_in    [B] or NULL (= zeros): the caller's icp_score_counter per subdomain
 *   decision          [B, 2] (layer, index within the layer); (-1, -1) when the subdomain has no candidate
 *   icp_counter_out   [B] updated counters
 *   kind              [B] or NULL: 0 = score decision, 1 = intercept score, 2 = preference order, -1 = no candidate
 *   scores            [B, sum n_k] or NULL: the masked |score| of every hidden ReLU (the reference's gt=True output)
 * Arrays other than random_order live in the memory space `in->mem`; with HOST buffers the call returns after the
 * results have landed, with DEVICE buffers it only enqueues on `stream`. */
int gnnb_babsr(gnnb_ctx* ctx, const gnnb_frontier* in, int32_t sparsest_layer, float decision_threshold,
               const int32_t* random_order, const int32_t* icp_counter_in, int32_t* decision, int32_t* icp_counter_out,
               int32_t* kind, float* scores, void* stream);

/* ---- online fine-tuning (the reference's `--bab_online` variant) ------------------------------------------------------
 * Replaces loss.backward() + optimizer.step() of GraphChoice.online_learning (graphnet/graph_score_online.py:62-77, called
 * from plnn/relu_conv_online.py:198-211): the reference differentiates `gnn_score - kw_score + improvement` through
 * GraphNet.forward with PyTorch autograd and applies torch.optim.Adam(lr, weight_decay) (graph_score_online.py:15).
 *
 * gnnb_score_grad: zeroes the gradient buffers (optimizer.zero_grad, :73), runs an exact-fp32 forward pass of the
 * subdomains of `in` that keeps the activations, and back-propagates
 *     loss = sum_i term_coeff[i] * score[term_domain[i]][term_index[i]]
 * (term_index = flat index into the concatenated hidden layers) into d loss / d parameter for all 52 tensors.  The
 * reference's loss is the two terms (+1, argmax index), (-1, index of the KW decision); `improvement` is a constant and
 * has no gradient.  term_* are HOST arrays, checked on the host (a term out of range fails with GNNB_ERR_INVALID);
 * term_scores [n_terms] (HOST, may be NULL) receives the terms' fp32 scores.  Frontier pointers live in `in->mem`; `in->mask`
 * is not read.  Copies the terms in and runs gnnb_score_grad_device; returns after the gradients are complete. */
int gnnb_score_grad(gnnb_ctx* ctx, const gnnb_frontier* in, int32_t n_terms, const int32_t* term_domain,
                    const int32_t* term_index, const float* term_coeff, float* term_scores, void* stream);

/* The same gradient with the terms on the device, for a branch-and-bound loop whose terms are computed on the GPU.
 * term_domain, term_index, term_coeff and term_scores [n_terms] are DEVICE arrays; frontier pointers live in `in->mem`.
 *   - A term with term_domain < 0 is inactive: it adds nothing, so a caller can pass a fixed-size list without reading a count.
 *   - A term with term_domain >= B or term_index outside [0, n_hidden) is never dereferenced: it is treated as inactive and
 *     counted, gnnb_get_option("grad_bad_terms").
 *   - term_scores of an inactive or out-of-range term is NaN.
 * Only the subdomains that carry an active term are run: they are listed on the device, and their count is read back (one
 * 8-byte device -> host copy and one synchronise of `stream`).  Forward with tape and backward then run over that list in
 * waves of at most option "grad_chunk" subdomains, each gathered into staging rows first; the gradients of the waves add up.
 * Everything after the read-back is only enqueued on `stream` (HOST frontiers: the call returns after the pass).  Argument
 * errors (null pointers, B < 1, n_terms < 1, weights or network not set, a network with zero-tap positions) are reported
 * before anything is enqueued, as in gnnb_score_grad. */
int gnnb_score_grad_device(gnnb_ctx* ctx, const gnnb_frontier* in, int32_t n_terms, const int32_t* term_domain,
                           const int32_t* term_index, const float* term_coeff, float* term_scores, void* stream);

/* Copy the gradients of the last gnnb_score_grad (the reference's `p.grad`) / the current parameters (the reference's
 * `model.state_dict()`) into 52 tensors in the order of gnnb_set_gnn_weights, HOST or DEVICE memory (each pointer's memory
 * space is taken from its address).  Synchronises the device. */
int gnnb_get_gradients(gnnb_ctx* ctx, float* const* tensors, const int64_t* numels, int n_tensors);
int gnnb_get_gnn_weights(gnnb_ctx* ctx, float* const* tensors, const int64_t* numels, int n_tensors);

/* One torch.optim.Adam step (amsgrad off) on all 52 tensors with the gradients of the last gnnb_score_grad:
 * g += weight_decay * p; m = lerp(m, g, 1 - beta1); v = beta2 v + (1 - beta2) g^2;
 * p -= lr / (1 - beta1^t) * m / (sqrt(v) / sqrt(1 - beta2^t) + eps).  The moments and the step count t live in the context
 * (they survive gnnb_set_gnn_weights, as the reference's optimizer survives load_state_dict) until gnnb_adam_reset.
 * Every packed form of the parameters used by gnnb_score is rebuilt before the call returns. */
int gnnb_adam_step(gnnb_ctx* ctx, float lr, float beta1, float beta2, float eps, float weight_decay, void* stream);
int gnnb_adam_reset(gnnb_ctx* ctx);

/* ---- device-resident domain queue of the branch-and-bound loop -------------------------------------------------------
 * Replaces the sorted Python list `domains` of ReLUDomain objects (plnn/relu_conv_gnnkwthreshold.py:20-53: mask, lower /
 * upper bound, every layer's bounds, the stored GNN decision) and the functions that work on it:
 *   add_domain(candidate, domains)      bisect.insort_left by lower bound          plnn/branch_and_bound.py:159-164
 *   pick_out(domains, threshold)        pop the front until lower_bound < threshold                          :167-184
 *   prune_domains(domains, threshold)   keep the prefix with lower_bound < threshold                         :264-281
 *   len(domains), domains[0].lower_bound                              plnn/relu_conv_gnnkwthreshold.py:236-244
 * A domain's payload (bounds of layers 0..L+1 in the gnnb_frontier layout, mask, bounds, decision) stays in a device pool;
 * the order is a sorted (key, slot) array on the device.  Equal lower bounds: the newest domain first (insort_left). */
typedef struct gnnb_queue gnnb_queue;

typedef struct {
    int32_t B;                           /* domains in this batch (capacity of the arrays for gnnb_queue_pick) */
    int32_t mem;                         /* gnnb_mem_kind of every pointer below */
    float* lower_bound;                  /* [B]  ReLUDomain.lower_bound (the sort key) */
    float* upper_bound;                  /* [B]  ReLUDomain.upper_bound */
    float* const* lb;                    /* L+2 arrays [B, n_k]: ReLUDomain.lower_all at the layers the GNN reads */
    float* const* ub;                    /* L+2 arrays [B, n_k]: ReLUDomain.upper_all */
    int8_t* mask;                        /* [B, sum n_k]  -1 undecided, 0 / 1 fixed (ReLUDomain.mask, concatenated) */
    int32_t* decision;                   /* [B, 2] (layer, index) or NULL: ReLUDomain.gnn_decision */
} gnnb_domains;

/* A queue for the network of `ctx` (gnnb_set_network first) with room for `capacity` domains. */
int gnnb_queue_create(gnnb_ctx* ctx, int64_t capacity, gnnb_queue** out);
void gnnb_queue_destroy(gnnb_queue* q);

/* add_domain for every domain b of `d` with keep[b] != 0 (keep: [B] bytes in d->mem, NULL = all; the reference adds a child
 * only when its lower bound is below the decision bound, relu_conv_gnnkwthreshold.py:217, 226).  *added = how many. */
int gnnb_queue_add(gnnb_queue* q, const gnnb_domains* d, const uint8_t* keep, int32_t* added, void* stream);

/* pick_out(domains, threshold) repeated until out->B domains are picked or the front of the queue is not below the
 * threshold; the picked domains are written to `out` in pick order (fields may be NULL) and leave the queue.
 * discard_rest != 0 mirrors the reference exactly: a pick_out that finds no domain below the threshold has popped (dropped)
 * every remaining domain; 0 keeps them for gnnb_queue_prune.  *picked = how many (HOST). */
int gnnb_queue_pick(gnnb_queue* q, float threshold, int32_t discard_rest, gnnb_domains* out, int32_t* picked, void* stream);

/* prune_domains(domains, threshold). */
int gnnb_queue_prune(gnnb_queue* q, float threshold, void* stream);

/* len(domains) and domains[0].lower_bound (global_lb is written only when the queue is not empty; either may be NULL). */
int gnnb_queue_stats(gnnb_queue* q, int64_t* size, float* global_lb, void* stream);

/* ---- batched KW intermediate bounds (the bound producer in front of the scoring path) ---------------------------------
 * Replaces DualNetwork(net, x, eps, bounded_input=False[, provided_zl, provided_zu]) of the reference's vendored
 * convex_adversarial as called by init_kw_bounds (plnn/dual_network_linear_approximation.py:205-288) for B domains at once:
 * pre-ReLU bounds of the L hidden layers (DualReLU.zl / zu), each intersected with the provided bounds when given (the
 * parent's bounds with one ReLU fixed, :313-319), the input box, and the bounds of the property output (dual(+-1)).
 * Every pointer is a DEVICE pointer: x [B, n_0], wp [B, n_L], bp [B]; provided_lb / provided_ub: L arrays [B, n_k],
 * k = 1..L, or both NULL; out_lb / out_ub: L + 2 arrays [B, n_k], k = 0..L+1.  Work is enqueued on `stream`. */
int gnnb_kw_bounds(gnnb_ctx* ctx, int32_t B, const float* x, float eps, const float* wp, const float* bp,
                   const float* const* provided_lb, const float* const* provided_ub, float* const* out_lb,
                   float* const* out_ub, void* stream);

/* Bounds of B root domains: the bounds part of KWConvGen.build_the_model(input_domain, x, ball_eps, bounded)
 * (plnn/conv_kwinter_gen.py:199-270) — init_kw_bounds, intersected layer by layer with interval bounds (the first layer from
 * the input box x -+ eps), and, for the domains where a hidden layer moved by more than 1e-4, update_kw_bounds from the first
 * such layer (:262-267).  Arrays as in gnnb_child_bounds (DEVICE pointers; out_mask and second_pass may be NULL).
 * Synchronises `stream` once. */
int gnnb_root_bounds(gnnb_ctx* ctx, int32_t B, const float* x, float eps, const float* wp, const float* bp,
                     float* const* out_lb, float* const* out_ub, int8_t* const* out_mask, int32_t* second_pass,
                     void* stream);

/* Bounds of B child domains: the bounds part of KWConvGen.update_the_model(relu_mask, pre_lb_all, pre_ub_all, decision,
 * choice) (plnn/conv_kwinter_gen.py:558-660), i.e. update_kw_bounds (plnn/dual_network_linear_approximation.py:296-439) with
 * the decided ReLU fixed — layers up to the split keep the parent's bounds, later layers get KW bounds intersected with the
 * parent's —, interval bounds of the layers behind the split intersected with them (:594-651), and a second KW pass for the
 * domains where the interval bounds tightened a hidden layer (:652-656).  The LP that follows in the reference (Gurobi) is
 * out of scope; the property-output bounds returned here are the KW / interval ones.
 * Every pointer is a DEVICE pointer.  parent_lb / parent_ub, out_lb / out_ub: L + 2 arrays [B, n_k], k = 0..L+1 (input box,
 * pre-ReLU bounds, property output; out may alias parent); dec_layer (0-based hidden layer) / dec_index / choice (0: blocked,
 * u = 0; 1: passing, l = 0): [B] int32; out_mask: L arrays [B, n_k] int8 in the BaB convention (1 passing, 0 blocked,
 * -1 ambiguous; :696-713) or NULL; second_pass: [B] int32 (1 where the second KW pass ran) or NULL.
 * Synchronises `stream` once (the number of domains that need the second pass). */
int gnnb_child_bounds(gnnb_ctx* ctx, int32_t B, const float* x, float eps, const float* wp, const float* bp,
                      const float* const* parent_lb, const float* const* parent_ub, const int32_t* dec_layer,
                      const int32_t* dec_index, const int32_t* choice, float* const* out_lb, float* const* out_ub,
                      int8_t* const* out_mask, int32_t* second_pass, void* stream);

/* Synchronise `stream` and report sticky device-side errors of earlier gnnb_score calls
 * (GNNB_ERR_NAN with the NaN count in *nan_count, may be NULL).  Clears the flag. */
int gnnb_check(gnnb_ctx* ctx, void* stream, int64_t* nan_count);

/* Kernel launches issued by this context since creation (bench.py's gpu_launches). */
int64_t gnnb_launch_count(gnnb_ctx* ctx);

/* Device time per kernel class, measured with CUDA events on the launching stream while option "profile" = 1.
 * Synchronises the device.  ms = summed duration, launches = launch count, rows = summed rows (nodes, or
 * subdomains for OUTPUT / ARGMAX) since the last gnnb_profile_reset. */
int gnnb_profile_read(gnnb_ctx* ctx, int klass, double* ms, int64_t* launches, int64_t* rows);
int gnnb_profile_reset(gnnb_ctx* ctx);

/* Copy the last error message into buf (NUL-terminated, truncated to n). Returns the last status. */
int gnnb_last_error(gnnb_ctx* ctx, char* buf, int n);

/* Debugging: copy a per-stage snapshot (names follow the oracle's `stages` keys, e.g. "t0_fwd_mu1") of
 * the LAST chunk processed to a HOST buffer; returns the element count through *numel. */
int gnnb_debug_snapshot(gnnb_ctx* ctx, const char* name, float* dst, int64_t max_numel, int64_t* numel);

/* ABI version of this header. */
int gnnb_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* GNNB_H */
