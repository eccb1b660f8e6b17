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

// d(sum_i coeff_i * score[domain_i][index_i]) / d(parameters) is ADDED to tp.dw / tp.db; the terms' scores are written to
// term_scores_host (may be null).  term_* are host arrays.  *arena / *arena_cap (floats): the caller-kept tape arena, grown when
// too small.  Synchronises `st` before returning.
int train_backward(const GnnParams& g, const TrainParams& tp, const std::vector<LayerDev>& layers, const std::vector<int>& n,
                   const std::vector<int>& hidden_off, const GnnInputs& in, int B, int n_terms, const int32_t* term_domain,
                   const int32_t* term_index, const float* term_coeff, float* term_scores_host, float** arena, size_t* arena_cap,
                   cudaStream_t st, int64_t* launches, std::string* err);

void adam_step(float* p, const float* grad, float* m, float* v, int64_t numel, float lr, float b1, float b2, float eps, float wd,
               int step, cudaStream_t st, int64_t* launches);

}  // namespace gnnb
