/* priblast_acc.h — C ABI of the B200 accessibility library (libpriblast_acc.so).
 *
 * This is the drop-in boundary for pRIblast's database-construction hot path.  It replaces the
 * per-sequence use of `class Raccess` (reference: raccess.hpp:37-62) made by
 * `DbConstruction::CalculateAccessibility` (reference: db_construction.cpp:170-229): instead of one
 * thread-private `Raccess` object and one `Run` call per sequence inside an OpenMP loop, the caller
 * hands the whole list of sequences to ONE call and gets every sequence's accessibility and
 * conditional-accessibility vectors back.  INTEGRATION.md shows the reference-side binding.
 *
 * Plain C types only (no CUDA, torch or C++ types).  All functions return 0 on success and a negative
 * PRIB_E* code on failure; prib_last_error() gives the thread-local message.  The library never calls
 * exit() (the reference does: raccess.hpp:42-50) and has NO CPU fallback: without a usable CUDA device
 * prib_acc_create fails with PRIB_ECUDA.
 */
#ifndef PRIBLAST_ACC_H
#define PRIBLAST_ACC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PRIB_OK 0
#define PRIB_EINVAL (-1)  /* bad argument (reference: "-d option must be greater than 1", raccess.hpp:47-50) */
#define PRIB_ECUDA (-2)   /* CUDA runtime/driver error, no device, or out of device memory */
#define PRIB_ESTATE (-3)  /* call order violated (e.g. compute before stage) */
#define PRIB_ENOMEM (-4)  /* host allocation failed */
#define PRIB_ENUMERIC (-5) /* an output value is not finite (partition function out of the double range); the
                              reference's log-domain sums cannot do this, so the result is refused, not returned */

typedef struct prib_ctx prib_ctx;

/* Constructor arguments of `Raccess(db_name, w, delta, path)` (raccess.hpp:39-58) that matter to the
 * computation, plus device selection. */
typedef struct prib_acc_params {
  int32_t maximal_span;          /* W: reference `-w`, default 70 (db_construction_parameters.hpp:48);
                                    1..1000 (above 200: the wide-span FP64 engine in modes 0 and 1)   */
  int32_t min_accessible_length; /* delta: reference `-d`, default 5; must be > 1 (raccess.hpp:47);
                                    2..1000, and may exceed W                                         */
  int32_t device;                /* CUDA device ordinal                                               */
  int32_t mode;                  /* 0 = auto: FP32 span-scaled engine with on-GPU FP64 re-run of
                                    range-flagged sequences; 1 = FP64 engine only (modes 0 and 1 at
                                    W > 200: FP64 span-scaled wide-span engine with on-GPU exact re-run
                                    of range-flagged sequences); 2 = exact: the
                                    reference's own log-domain arithmetic (float-table logsumexp,
                                    raccess.cpp:414-419, in its summation order) on the GPU: results are
                                    bit-identical to the reference built without FMA contraction     */
  int64_t max_batch_bytes;       /* device-memory budget for DP state; 0 = 60 % of free memory        */
} prib_acc_params;

/* device-time phases of one batch, in launch order */
#define PRIB_NUM_PHASES 7
#define PRIB_PHASE_NAMES {"memset", "inside", "outer_scans", "outside", "biloop_left", "biloop_right", "hairpin_finalize"}

typedef struct prib_acc_counters {
  int64_t sequences;     /* sequences processed since create */
  int64_t nucleotides;   /* sum of their lengths */
  int64_t batches;       /* device batches */
  int64_t kernel_launches;
  double kernel_ms;      /* device time of the DP + accessibility kernels (CUDA events) */
  double h2d_ms, d2h_ms; /* device time of the copies */
  int64_t h2d_bytes, d2h_bytes;
  int64_t dp_state_bytes; /* size of the DP scratch allocation */
  int64_t dp_state_bytes_used; /* part of it the largest batch so far used */
  double phase_ms[PRIB_NUM_PHASES]; /* device time per phase, summed over batches */
  int64_t fp64_rerun_sequences;  /* sequences the FP32 engine flagged and the FP64 engine recomputed */
  int64_t fp32_flagged[4];       /* sequences whose FIRST FP32 pass left the safe range: [0] inside values too
                                    large, [1] inside too small, [2] outside too large, [3] outside too small */
  int64_t exact_rerun_sequences; /* sequences the wide-span engine (W > 200) flagged and the exact engine
                                    recomputed */
} prib_acc_counters;

/* Replaces the `Raccess` constructor.  One context per GPU; not re-entrant per context.
 * Same as prib_acc_create_lengths(out, params, 1, &params->min_accessible_length). */
int prib_acc_create(prib_ctx **out, const prib_acc_params *params);

#define PRIB_MAX_LENGTHS 32

/* A context that computes accessibility for n_lengths minimum accessible lengths in each call: the inside pass, the
 * outer scans and the outside pass run once per batch, the strand weights and the finalize once per length.  Every
 * output float equals that of a context created with prib_acc_create for that length alone.
 *   lengths        : 1 <= n_lengths <= PRIB_MAX_LENGTHS entries, strictly increasing, each checked like
 *                    min_accessible_length (which is not read); a bad entry is PRIB_EINVAL, named in the message.
 *   acc_off/cond_off of prib_acc_run and prib_acc_fetch then have n_lengths * n entries: [l * n + k] is sequence k at
 *                    lengths[l].  With the packed layout of each length back to back, fetch copies the device image
 *                    straight into a page-locked `out`.
 * Counters: sequences, nucleotides and the re-run counts count each sequence once (a flagged sequence is re-run once
 * for all lengths); the last three phase_ms entries sum over the lengths. */
int prib_acc_create_lengths(prib_ctx **out, const prib_acc_params *params, int32_t n_lengths, const int32_t *lengths);
void prib_acc_destroy(prib_ctx *ctx);

/* Replaces the loop of `Raccess::Run(seq, acc, cond)` calls (raccess.cpp:42-50) over n sequences.
 *   seq[k], len[k] : bases as given in the FASTA record (A/C/G/T/U any case; anything else = unknown,
 *                    raccess.cpp:55-68); need not be NUL-terminated.
 *   out            : caller-owned host buffer (pinned memory from prib_host_alloc is fastest).
 *   acc_off[k]     : float offset in `out` of the len[k] accessibility values of sequence k
 *                    (entries len-delta+1 .. len-1 are 0, as in raccess.cpp:487,510-517).
 *   cond_off[k]    : float offset of the len[k] conditional-accessibility values
 *                    (entries 0 .. delta-1 are 0, raccess.cpp:488,519-527).
 * Blocking.  Results do not depend on batching or on the number of GPUs used by the caller.  The call pipelines
 * its own stages: the bases are copied (once) into a page-locked arena batch by batch and each batch is launched as
 * soon as it is staged, so the host copy of one batch runs under the kernels of the previous one; seq[] must stay
 * valid until the call returns.  `h2d_ms` is not accumulated for this call (copies and kernels interleave). */
int prib_acc_run(prib_ctx *ctx, int32_t n, const char *const *seq, const int32_t *len, float *out,
                 const int64_t *acc_off, const int64_t *cond_off);

/* The same work split in three so a caller (or a benchmark) can keep inputs resident in device memory:
 * stage = sort/partition into device batches + upload; compute = all kernels, asynchronous on the
 * context's stream; fetch = download + scatter into `out` (blocks until compute has finished). */
int prib_acc_stage(prib_ctx *ctx, int32_t n, const char *const *seq, const int32_t *len);
int prib_acc_compute(prib_ctx *ctx);
int prib_acc_fetch(prib_ctx *ctx, float *out, const int64_t *acc_off, const int64_t *cond_off);
int prib_acc_sync(prib_ctx *ctx);

/* Use an existing CUDA stream (a `cudaStream_t` passed as void*) for all work of this context, so a
 * caller can bracket the work with its own events.  NULL restores the context's own stream. */
int prib_acc_set_stream(prib_ctx *ctx, void *cuda_stream);

int prib_acc_get_counters(prib_ctx *ctx, prib_acc_counters *out);

/* Measured instruction-issue peaks of one device, in 1e9 lane-operations per second: MUFU ex2.approx,
 * FP32 FMA and FP64 FMA.  These are the roofline denominators of SURVEY §8d (MEASURED_PEAKS.json holds
 * only copy bandwidth and bf16 GEMM throughput). */
int prib_peak_probe(int32_t device, double *mufu_gops, double *ffma_gops, double *dfma_gops);

/* Number of CUDA devices visible to the process (0 if none / no driver). */
int prib_device_count(void);

/* Pinned host memory for `out` (optional). */
void *prib_host_alloc(size_t bytes);
void prib_host_free(void *p);

const char *prib_last_error(void);
const char *prib_version(void);

/* Byte image of one sequence's record in `<db>.acc` exactly as the reference writes it
 * (raccess.cpp:447-481): int32 n1 = L-delta+1, n1 floats, int32 L, L floats.  Pure host helper used by
 * the `db` front-end; returns the number of bytes written (8 + 4*(2L-delta+1)) or a negative code. */
int64_t prib_acc_record_bytes(int32_t len, int32_t delta);
int64_t prib_acc_write_record(const float *acc, const float *cond, int32_t len, int32_t delta, void *dst);

/* Suffix array of one encoded database page on the GPU.  Replaces `sais(T, SA, n)` (sais.cpp:656) as called
 * by DbConstruction::ConstructSuffixArray (db_construction.cpp:330-335): text = the reversed, encoded,
 * sentinel-terminated sequences of the page (symbols 0..9, encoder.hpp:36-78), sa = n int32 in host memory.
 * The suffix array of a text is unique, so the bytes equal the reference's.  Blocking; uses `device`. */
int prib_suffix_array(const unsigned char *text, int32_t n, int32_t *sa, int32_t device);

#ifdef __cplusplus
}
#endif
#endif /* PRIBLAST_ACC_H */
