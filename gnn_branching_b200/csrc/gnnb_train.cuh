// Online fine-tuning (gnnb_train.cu): gradients of selected scores w.r.t. the GNN parameters and the Adam step.
#pragma once

#include <string>
#include <vector>

#include "gnnb_common.cuh"

namespace gnnb {

// master parameters and their gradients on the device, nn.Linear layout (weight [out][in], bias [out])
struct TrainParams {
    const float* w[N_LIN];
    const float* b[N_LIN];
    float* dw[N_LIN];
    float* db[N_LIN];
};

int train_init();   // opt-in shared memory sizes; returns cudaError_t

// Hidden layer k of a wave's tape as the score head reads it: mu (after the last backward sweep) and its gradient, [rows][64]
// with row = b * n + node; off = the layer's first flat index.
struct TermLayer { const float* mu; float* dmu; int off; int n; };

// The loss terms of one wave (device arrays of the caller's n_terms terms).  A term belongs to the wave when its domain d is in
// [0, B), its index in [0, n_hidden), and row_of[d] - row0 is in [0, rows of the wave).
struct WaveTerms {
    const int32_t *domain, *index;
    const float* coeff;
    const int32_t* row_of;
    int n_terms, B, n_hidden, row0;
    float* scores;            // [n_terms] the wave writes the scores of its terms
};

// Enqueues the naming pass of gnnb_score_grad_device (two launches): scores[t] = NaN for every term; flag[d] = 1 for each domain
// an active term (domain >= 0) names; cnt[1] += 1 for each active term whose domain or index is out of range; the flagged
// domains in ascending order -> list, their positions -> row_of, their count -> cnt[0].  flag and cnt[0..1] must be zero.
void name_terms(const int32_t* domain, const int32_t* index, int n_terms, int B, int n_hidden, float* scores, int32_t* cnt,
                int32_t* flag, int32_t* list, int32_t* row_of, cudaStream_t st, int64_t* launches);

// Floats of the tape of waves of up to Bcap subdomains (activations, gradient temporaries, the score head's layer table).
size_t train_tape_floats(const std::vector<int>& n, int T, int Bcap);

// One wave of B <= Bcap subdomains (`in`: their arrays, node order): exact-fp32 forward with the tape in `arena` (laid out
// for Bcap, train_tape_floats floats), then d(sum of the wave's terms coeff * score) / d(parameters) ADDED to tp.dw / tp.db and
// the wave's term scores written.  Enqueues on `st` without synchronising; returns the cudaError_t of the launches.
int train_wave(const GnnParams& g, const TrainParams& tp, const std::vector<LayerDev>& layers, const std::vector<int>& n,
               const std::vector<int>& hidden_off, const GnnInputs& in, int Bcap, int B, const WaveTerms& wt, float* arena,
               cudaStream_t st, int64_t* launches);

void adam_step(float* p, const float* grad, float* m, float* v, int64_t numel, float lr, float b1, float b2, float eps, float wd,
               int step, cudaStream_t st, int64_t* launches);

}  // namespace gnnb
