// Device-resident optimiser state of one L-BFGS problem (torch/optim/lbfgs.py:359-385,528-535).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "isx_kernels.h"

namespace isx {

static constexpr int kMaxSlots = 104;  // history_size (<= 100, torch default) + 1 candidate slot, padded

struct LbfgsConfig {
  int epochs;      // closure evaluations requested (pipelines.py:16,79)
  int max_iter;    // 20
  int max_eval;    // 25 = max_iter * 5 // 4
  int history;     // 100
  double lr;
  double tolerance_grad;    // 1e-7
  double tolerance_change;  // 1e-9
  double c_weight, s_weight;  // alpha, beta (pipelines.py:89)
};

struct LbfgsState {
  int n_iter;         // state["n_iter"]
  int func_evals;     // state["func_evals"] == current_epoch[0] of pipelines.py:97
  int phase;          // 0: next evaluation opens an optimizer.step(); 1: re-evaluation inside its loop
  int n_iter_step;    // n_iter local to the current step (1..max_iter)
  int current_evals;
  int hist_count, hist_head, cand_slot;  // ring of (y, s) pairs + the slot the candidate pair lives in
  int done;           // pipelines.py:79 loop finished for this problem
  int compute_d, apply;  // orders for pass 2 of this tick
  unsigned int max_td_bits;  // max |t d| of the last update (float bits; lbfgs.py:522)
  double loss, prev_loss, t, H_diag;
  double last_c, last_s;
  double ro[kMaxSlots];
  float coef_s[kMaxSlots], coef_y[kMaxSlots];
  float coef_g;
  float pad_;
};

int lbfgs_nblk(long N);
int lbfgs_init(LbfgsState* states, int P, cudaStream_t s);
int clamp01(float* x, long n, cudaStream_t s);
int lbfgs_tick(float* x, const float* g, float* g_prev, void* S, void* Y, int history_bf16, LbfgsState* states,
               double* mats,
               float* part, float* ext, double* dots, const double* loss_c, const double* loss_s, int images_per_problem, int P,
               long N, const LbfgsConfig& cfg, double* hist_c, double* hist_s, int tick, cudaStream_t s,
               const double* c_w = nullptr, const double* s_w = nullptr,   // per-problem alpha / beta (device [P]) or cfg's
               const ProblemRanges* pr = nullptr);   // with c_w: the problems' slices (N = floats of the largest problem)

}  // namespace isx
