// Wide-span engine (spans kMaxSpan < W <= kWideSpan, modes 0 and 1 of prib_acc_params): FP64, span-scaled,
// range-checked.  See acc_wide.cu and DESIGN.md §2.9.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "acc_exact.h"  // ExactBatch: the wide engine takes the same batch description

namespace prib {

struct WideEngine;  // opaque: device tables and the scan rings

// Band state of one column: the arrays of acc_core.h (rows as in the FP64 tile engine) and the two outer logs.
long long wide_state_bytes_per_column(int W);
// Builds the span-scaled tables for W and each minimum accessible length (increasing) and uploads them.  klog2:
// kappa = 2^-klog2 (default_scale_wide()).  Returns nullptr and sets err on failure.
WideEngine *wide_create(int W, const std::vector<int> &lengths, double klog2, std::string &err);
void wide_destroy(WideEngine *e);
// All kernels of one batch on `stream`; d_state must hold wide_state_bytes_per_column(W) * NC bytes.  flags[k] is
// set to a non-zero value when a stored value of sequence k left the engine's range (the caller re-runs it in the
// exact engine; its outputs are not written); *bad counts non-finite outputs of the other sequences.  The inside,
// scan and outside passes run once; the strand and finalize kernels once per length (phase events as exact_run's).
// Returns a cudaError_t (0 = ok); *launches receives the number of kernel launches.
int wide_run(WideEngine *e, const ExactBatch &b, int32_t *flags, int32_t *bad, char *d_state, cudaStream_t stream,
             cudaEvent_t *phase_events, int *launches);

}  // namespace prib
