// Exact engine (mode 2 of prib_acc_params): the reference's own arithmetic on the GPU.
//
// The fast engines (acc_tile.h) re-formulate the recurrences in the linear domain; their results agree with
// the reference to ~1e-5 kcal/mol, which is the reference's OWN noise (float-table log inside every
// logsumexp, raccess.cpp:414-419), so the last printed digit of a `ris` energy can differ.  This engine
// instead evaluates, per DP cell and per sequence position, the very same chain of
//     max + (double)fmath::log((float)(fmath::expd(min - max) + 1.0))
// operations in the very same order as raccess.cpp, on bit-exact device copies of fmath's two tables, in
// IEEE double/float without FMA contraction (the TU is compiled with -fmad=false).  Cells of one span are
// independent (SURVEY §8a: every dependency lies at a smaller span (inside) or a larger one (outside)), so a
// span wavefront with one thread per cell gives the reference's bits; the accessibility sums are re-enumerated
// per position in the reference's loop order.  Result: `.acc` records byte-identical to the reference built
// without FMA contraction (-O3, SURVEY Q6), hence a byte-identical database and `ris` output.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

namespace prib {

struct ExactBatch {
  long long NC;            // padded columns of the batch (layout of acc_tables.h: column = seq_off + left index)
  int n;                   // sequences
  const uint8_t *S;        // base code per column (0 = unknown / padding / left index 0)
  const int32_t *col_seq;  // sequence id per column, -1 padding
  const int32_t *seq_len;
  const long long *seq_off;
  const long long *acc_off, *cond_off;  // float offsets into out
  float *out;              // output image of the first minimum accessible length
  long long out_stride;    // floats from the output image of one length to that of the next
};

struct ExactEngine;  // opaque: device tables

long long exact_state_bytes_per_column(int W);
// Builds the scaled energy tables (raccess.hpp:105-158) and the two fmath tables from the host libm, exactly
// as the reference does at static-init time, and uploads them.  lengths: the minimum accessible lengths, increasing.
// Returns nullptr and sets err on failure.
ExactEngine *exact_create(int W, const std::vector<int> &lengths, std::string &err);
void exact_destroy(ExactEngine *e);
// All kernels of one batch on `stream`; d_state must hold exact_state_bytes_per_column(W) * NC bytes.  The inside,
// outer and outside passes run once; the hairpin, loop and finalize kernels once per length.  phase_events: 8 events
// for one length, 3 more per further length (the last three phases of each length).
// Returns a cudaError_t (0 = ok); *launches receives the number of kernel launches.
int exact_run(ExactEngine *e, const ExactBatch &b, char *d_state, cudaStream_t stream, cudaEvent_t *phase_events,
              int *launches);

}  // namespace prib
