// Stochastic mapping of event classes (event_mapping.cu), shared with the engine's bppgpu_expected_events (engine.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <vector>

namespace bppgpu {

constexpr int kMaxEventTypes = 8;

// Tallies of one simulation, resident on the device, one row per distinct length in increasing order:
//   count [U][S][S]     paths from a in state j at that length
//   sum   [U][S][S][T]  their total number of class-T events
struct EventTallies {
  int S = 0, T = 0, U = 0;
  std::vector<int> row_of;                  // [n_lengths] row of each input length
  unsigned long long *count = nullptr, *sum = nullptr;
  ~EventTallies() {
    cudaFree(count);
    cudaFree(sum);
  }
};

// Validates the inputs (BPPGPU_E_INVALID), simulates paths first .. first + n_sims - 1 from every start state and leaves the
// tallies in `out`.  type_rates [T][S][S] and lengths may be host, pinned or device memory.  *ms = device time of the
// simulation and the prefix pass (CUDA events on `st`).
int event_tallies(int device, cudaStream_t st, int S, int T, const double* type_rates, int64_t n_lengths, const double* lengths,
                  int64_t first, int64_t n_sims, uint64_t seed, EventTallies& out, double* ms);

// For each branch g < n_branches (device arrays): out[out_row[g]][0 .. T-1] = E_T and out[out_row[g]][T] = the unreached mass,
// from the tallies' row rows[g], the branch's joint posterior joint[g] [N][S][S] (node state x, father state y) and the pattern
// weights w [N]; one CTA per branch, enqueued on `st`
cudaError_t event_combine(cudaStream_t st, const EventTallies& t, int n_branches, const int* rows, const double* joint, const double* w,
                          long long N, const int* out_row, double* out);

// device milliseconds of the calling thread's last bppgpu_simulate_event_counts / bppgpu_expected_events: simulation, combination
double* event_timing();

}  // namespace bppgpu
