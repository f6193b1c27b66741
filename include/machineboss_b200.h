/* machineboss_b200.h -- C ABI of the B200-native Forward / Backward / Viterbi engine.
 *
 * The reference (evoldoers/machineboss) has no FFI for this path: its boundary is the C++ class
 * surface  EvaluatedMachine / SeqPair(List) / ForwardMatrix / BackwardMatrix / ViterbiMatrix /
 * MachineCounts  (SURVEY.md section 8b).  This header is the C-ABI layer underneath a host-side
 * mirror of those classes (machineboss_b200/host/boss_b200.h); every entry point names the
 * reference interface it replaces.  Plain pointers and sizes only; the caller owns every host
 * buffer; handles own device memory.  All functions return 0 on success, non-zero on error, with
 * the message available from mb_last_error().  There is no CPU fallback: without a CUDA device
 * every compute call fails.
 *
 * Conventions shared with the reference:
 *   - states 0..nStates-1; start state 0, end state nStates-1          (src/eval.cpp:76-84)
 *   - token 0 is epsilon; input tokens 1..nInTok, output tokens 1..nOutTok, numbered in
 *     alphabetical order of the alphabets                              (src/eval.h:11-25, machine.cpp:175-191)
 *   - transitions are listed in the reference's enumeration order: source state ascending, then
 *     position in the source's TransList, so global id = transOffset[src] + transIndex
 *                                                                      (src/eval.cpp:49-69)
 *   - log-weights are natural-log doubles, -inf allowed                (src/eval.cpp:58)
 */
#ifndef MACHINEBOSS_B200_H
#define MACHINEBOSS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mb_machine mb_machine;
typedef struct mb_batch mb_batch;

/* ---- library state: everything here is PER HOST THREAD, so that a host thread per GPU can drive its own
 * device without locking (the reference has no threads; its only global state is its logger and caches) ---- */
const char* mb_last_error (void);                 /* message of the last failing call on this thread */
int mb_version (void);

/* A directory where the library keeps the modules it compiles at run time for a machine's structure (NVRTC, sm_100a), keyed by a
 * hash of the generated source: a later process that creates a machine of the same structure loads the module instead of
 * compiling it (seconds per machine).  NULL or "": no cache (the default).  Process-wide; the directory must exist. */
int mb_set_kernel_cache_dir (const char* dir);
int mb_device_count (int* count);                  /* cudaGetDeviceCount */
int mb_set_device (int device);                    /* device used by handles this thread creates afterwards (default 0) */
/* Tuning / diagnostic knobs (integers; MB_OPTION_UNSET restores the built-in choice).  mb_set_option sets the
 * calling thread's defaults, copied into every machine it creates afterwards; mb_machine_set_option changes one
 * machine.  Names: see kOptionNames in csrc/mb_api.cu ("verbose", "jit_narrow", "lane_r", "no_big", ...).
 * The compute path never reads the environment. */
#define MB_OPTION_UNSET (-2147483647 - 1)
int mb_set_option (const char* name, int32_t value);

/* ---- EvaluatedMachine (src/eval.h:59-98, src/eval.cpp:42-70) ----
 * Flattens what EvaluatedMachine::init builds: per transition its source, destination, input
 * token, output token and log-weight, in enumeration order.  Fails, like the reference's
 * Assert(isAdvancingMachine) (eval.cpp:44, machine.cpp:758-764), if a silent transition from a
 * state s >= 1 goes to a state <= s. */
int mb_machine_create (mb_machine** out, int32_t nStates, int32_t nInTok, int32_t nOutTok, int64_t nTrans,
                       const int32_t* src, const int32_t* dst, const int32_t* inTok, const int32_t* outTok,
                       const double* logWeight);
/* New log-weights for the same structure: what re-running EvaluatedMachine(machine, params) does
 * once per EM iteration (src/fitter.cpp:29). */
int mb_machine_update_weights (mb_machine* m, const double* logWeight);
int mb_machine_info (const mb_machine* m, int32_t* nStates, int64_t* nTrans, int32_t* engine /* MB_ENGINE_* */);
int mb_machine_set_option (mb_machine* m, const char* name, int32_t value);
void mb_machine_destroy (mb_machine* m);

#define MB_ENGINE_GENERIC 0   /* anti-diagonal wavefront over the CSR machine, any size */
#define MB_ENGINE_JIT     1   /* machine-specialised strip kernel compiled with NVRTC, small machines */
#define MB_ENGINE_WIDE    2   /* Forward and Viterbi of mid-size and large machines (their Backward and counts run on the generic
                                 engine), by whichever sweep fits the call: a generated thread-per-cell kernel for full matrices
                                 of machines of up to ~1000 states, a read per lane for batches without input sequences (profile
                                 HMMs of any size), a table-driven strip kernel over shared-memory transition tables otherwise
                                 (envelopes, log-domain re-runs) */
/* Force an engine for machines this thread creates afterwards (-1 = choose automatically, the default). */
int mb_set_engine (int engine);

/* ---- SeqPairList (src/seqpair.h:18-73,115-121), already tokenised (DPMatrix ctor, dpmatrix.defs.h:6-7) ----
 * Pair k has input tokens inTokens[inOff[k] .. inOff[k+1]) and output tokens
 * outTokens[outOff[k] .. outOff[k+1]).  Tokens are 1-based (0 never appears in data).  The batch is
 * copied to the device with full envelopes (a SeqPair without an alignment, seqpair.cpp:104-110). */
int mb_batch_create (mb_batch** out, int64_t nPairs,
                     const uint8_t* inTokens, const int64_t* inOff,
                     const uint8_t* outTokens, const int64_t* outOff);
void mb_batch_destroy (mb_batch* b);
/* ---- Envelope (src/seqpair.h:75-113, seqpair.cpp:104-152; DPMatrix cell access dpmatrix.h:128-146) ----
 * Restricts pair k's matrices to inStart[r] <= inPos < inEnd[r] on output row o, r = rowOff[k] + o.
 * A pair has either outLen+1 rows or none (rowOff[k+1] == rowOff[k]: the full matrix).  This is what
 * the reference does to every matrix of a SeqPair that carries an alignment (Envelope::initPath).
 * Fails like DPMatrix::alloc (dpmatrix.defs.h:31-32) if an envelope does not fit its pair or is
 * not connected.  rowOff == NULL removes all envelopes.  Batches with envelopes run on the
 * wide engine's table-driven sweep (Forward, Viterbi) and on the generic engine (Backward, counts). */
int mb_batch_set_envelopes (mb_batch* b, const int64_t* rowOff, const int64_t* inStart, const int64_t* inEnd);
/* Gives the scratch the engine keeps attached to the batch between calls (back-pointers, stored
 * Forward values, strip boundaries) back to the device; results already fetched stay valid. */
int mb_batch_trim (mb_batch* b);

/* ---- RollingOutputForwardMatrix::logLike / ForwardMatrix::logLike (src/forward.defs.h:22-55) ----
 * loglike[k] = log-sum over all paths of pair k, -inf if none. */
int mb_forward (mb_machine* m, mb_batch* b, double* loglike);

/* ---- BackwardMatrix::logLike (src/backward.cpp:18-50) ---- */
int mb_backward (mb_machine* m, mb_batch* b, double* loglike);

/* ---- ViterbiMatrix::logLike + ViterbiMatrix::path (src/viterbi.cpp:18-51, dpmatrix.defs.h:82-110) ----
 * score[k] = best path log-weight.  If pathLen != NULL the traceback is run too and pathLen[k]
 * receives the number of transitions on pair k's path (0 when score[k] is -inf, as boss.cpp:831
 * skips those).  The tie-break is the reference's: candidates in the order match, delete, insert,
 * silent, each by ascending source state then transition index; the first maximum wins. */
int mb_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen);
/* Copies the paths of the last mb_viterbi on this batch: pair k's global transition ids, start ->
 * end, go to pathTrans[pathOff[k] .. pathOff[k] + pathLen[k]). */
int mb_viterbi_paths (mb_batch* b, int32_t* pathTrans, const int64_t* pathOff);

/* The same paths with ids narrowed to bytesPerId = 1 or 2 bytes (4: as mb_viterbi_paths), for machines with at
 * most 256 / 65 536 transitions: the paths of 10 000 dnapsw pairs of 1 kb are 150 MB as int32 and 37 MB as
 * bytes, and the copy to the host is what an end-to-end call waits for last.  Pair k's ids go to elements
 * pathOff[k] .. pathOff[k] + pathLen[k]. */
int mb_viterbi_paths_narrow (mb_batch* b, void* pathTrans, int32_t bytesPerId, const int64_t* pathOff);

/* The same copy without waiting for it: the ids are narrowed on the batch's stream and handed to the copy engine;
 * the call returns at once, later calls on the batch (an mb_forward of the same pairs, say) run while the paths
 * travel, and mb_batch_wait returns when they have arrived.  pathTrans should be page-locked host memory (with
 * pageable memory the call simply blocks); it must not be read before mb_batch_wait.  Offsets that are not the
 * packed order of the batch (pathOff[k+1] - pathOff[k] == pathLen[k]) take the blocking path. */
int mb_viterbi_paths_start (mb_batch* b, void* pathTrans, int32_t bytesPerId, const int64_t* pathOff);
int mb_batch_wait (mb_batch* b);

/* ---- MachineCounts over a list (src/counts.cpp:37-64, src/backward.cpp:62-87) ----
 * counts[t] (t < nTrans, may be NULL) receives the expected number of uses of transition t summed
 * over all pairs; loglike[k] (may be NULL) the Forward log-likelihood of pair k.  Pairs whose
 * log-likelihood is -inf contribute nothing. */
int mb_counts (mb_machine* m, mb_batch* b, double* counts, double* loglike);

/* ---- MachineCounts of each pair on its own (src/counts.cpp:37-64 over a list of one) ----
 * Posterior counts of each pair: row k of counts ([nPairs][nTrans], row-major) is what mb_counts gives for a
 * batch holding only pair k; loglike[k] (may be NULL) as mb_counts.  An impossible pair gets a zero row and -inf.
 * Per pair: expected substitutions and gaps, use of a profile's states by each read, weighted EM, and the
 * gradient of pair k's log-likelihood with respect to the log-weights (row k).  counts must not be NULL
 * (mb_counts gives the log-likelihoods alone).  Same engines as mb_counts; the device holds the rows of one
 * chunk of pairs at a time. */
int mb_pair_counts (mb_machine* m, mb_batch* b, double* counts, double* loglike);

/* ---- DPMatrix::cell of a ForwardMatrix / BackwardMatrix / ViterbiMatrix (src/dpmatrix.h:128-146) ----
 * The whole log-domain matrix of ONE pair of the batch, as the reference stores it (dpmatrix.h:86-95):
 * cells[((o * (inLen + 1)) + i) * nStates + s], state fastest; -inf outside the pair's envelope.  It is what
 * the reference's consumers of a stored matrix read: ForwardMatrix::samplePath (forward.cpp:17-23,
 * dpmatrix.defs.h:176-186), postTransQueue / traceFrom (backward.cpp:52-56,89-108).  The caller provides
 * (inLen + 1) * (outLen + 1) * nStates doubles.  Sums use the reference's log-sum-exp cut-off
 * (logsumexp.h:52), so cells track the reference's to its table's interpolation error. */
#define MB_MATRIX_FORWARD  0
#define MB_MATRIX_BACKWARD 1
#define MB_MATRIX_VITERBI  2
int mb_matrix (mb_machine* m, mb_batch* b, int64_t pair, int32_t kind, double* cells);

/* ---- ForwardMatrix::samplePath (src/forward.cpp:17-23) for every pair of the batch, nSamples paths each, drawn on the device ----
 * Path j of pair k has length pathLen[k * nSamples + j] (0 when loglike[k] is -inf); loglike (may be NULL) receives the
 * Forward log-likelihoods of the stored matrices (the generic engine's values).  Draws are keyed by (seed, k, j): the same
 * triple gives the same path on any device and under any chunking.  Each step draws a candidate in proportion to
 * exp (F(previous cell) + log-weight), shifted by the step's largest candidate so that long pairs do not underflow, with
 * Philox4x32-10 (key = seed, counter = { step, j, k & 0xffffffff, k >> 32 }).  The reference's mt19937 stream is not
 * reproduced (ForwardMatrix::samplePath in the host mirror does that).  The paths are kept apart from mb_viterbi's: neither
 * call overwrites the other's.  A failed call leaves no samples stored. */
int mb_sample_paths (mb_machine* m, mb_batch* b, int32_t nSamples, uint64_t seed, double* loglike, int64_t* pathLen);
/* The ids of the last mb_sample_paths on this batch, narrowed to bytesPerId = 1, 2 or 4 as in mb_viterbi_paths_narrow:
 * path r = k * nSamples + j goes to elements pathOff[r] .. pathOff[r] + pathLen[r]. */
int mb_sampled_paths (mb_batch* b, void* pathTrans, int32_t bytesPerId, const int64_t* pathOff);

/* ---- posterior decoding (BackwardMatrix::postTransQueue / traceFrom, src/backward.cpp:52-56,89-108, for a whole batch) ----
 * A step of a path takes transition t from cell (i, o), state src, to cell (i + di, o + do), state dst.  Its posterior
 * probability, the probability that a path drawn from the posterior takes t from that cell, is
 *     gamma = exp ((F(i, o)[src] - ll) + (B(i + di, o + do)[dst] + w_t))
 * over the generic engine's log-domain Forward and Backward matrices, ll = B(0, 0)[0] the Backward log-likelihood; bit for bit
 * the term mb_pair_counts adds to the pair's row (backward.cpp:66); 0 when ll is -inf.  A step is admissible when
 * F(i, o)[src] + w_t + B(i + di, o + do)[dst] is finite (it lies on a complete path of finite weight).  The gain of a path is the
 * sum over its steps of c(t) * gamma, c(t) the number of tokens t consumes (2 match, 1 insert or delete, 0 silent): the expected
 * number of the pair's tokens that a posterior path consumes with the same transition from the same cell, in [0, inLen + outLen].
 * The maximum expected accuracy (MEA) path is the admissible path from (0, 0, state 0) to (inLen, outLen, end state) of largest
 * gain: A(0, 0)[0] = 0, A(cell)[s] = max over admissible candidates of A(source cell)[src] + c(t) * gamma, candidates in the
 * traceback's order (match, delete, insert, silent; each by source state then transition index), the first maximum winning;
 * cells outside the envelope are -inf.
 *
 * mb_mea: the MEA path of every pair.  gain[k] its gain (-inf for an impossible pair, whose path has length 0), loglike[k]
 * (may be NULL) the Forward log-likelihood, pathLen[k] (may be NULL) its number of steps.  Runs on the generic engine, three
 * full matrices per pair.  The paths are kept apart from mb_viterbi's and mb_sample_paths'; a failed call leaves none stored. */
int mb_mea (mb_machine* m, mb_batch* b, double* gain, double* loglike, int64_t* pathLen);
/* The ids of the last mb_mea on this batch, narrowed to bytesPerId = 1, 2 or 4 as in mb_sampled_paths: pair k's path goes to
 * pathTrans[pathOff[k] .. pathOff[k] + pathLen[k]); stepPost (may be NULL) receives gamma of each step at the same offsets. */
int mb_mea_paths (mb_batch* b, void* pathTrans, int32_t bytesPerId, const int64_t* pathOff, double* stepPost);
/* gamma of each step of caller-supplied paths: path r belongs to pair pairOfPath[r] and holds pathTrans[pathOff[r] ..
 * pathOff[r] + pathLen[r]); stepPost uses the same offsets.  A path must be a path of its pair: each step leaves the state the
 * path is in and reads the pair's next tokens, stays in the envelope, and the path ends at (inLen, outLen, end state); the
 * first path that is not fails the call with a message naming the path and the step.  Runs on the generic engine. */
int mb_path_posteriors (mb_machine* m, mb_batch* b, int64_t nPaths, const int64_t* pairOfPath,
                        const int32_t* pathTrans, const int64_t* pathOff, const int64_t* pathLen, double* stepPost);

/* ---- one list of pairs over several GPUs of a box (SURVEY.md 8e) ----
 * Replaces the reference's single-core loops over a SeqPairList: MachineCounts (counts.cpp:37-43) inside
 * MachineFitter::fit (fitter.cpp:23-47), and the -L / -A loops of the CLI (boss.cpp:796,826).  The pairs are
 * dealt to the devices longest-processing-time first by cell count (Li+1)(Lo+1); the machine is replicated; one
 * host thread per device drives that device's share.  Forward / Viterbi / per-pair counts: no communication, results gathered by
 * pair index.  Counts: ncclAllReduce (sum, ncclDouble) of nTrans + 1 values over NVLink (libnccl.so.2, resolved
 * at run time; one device, or no NCCL: added on the host -- mb_group_info says which).  Results are those of
 * the single-device calls: identical for Forward and Viterbi, equal up to the order of summation for counts. */
typedef struct mb_group mb_group;
typedef struct mb_gmachine mb_gmachine;
typedef struct mb_gbatch mb_gbatch;
/* shardOfPair[k] = shard (0 .. nShards-1) of pair k under that deal; deterministic; pure host code */
int mb_shard_pairs (int64_t nPairs, const int64_t* inOff, const int64_t* outOff, int32_t nShards, int32_t* shardOfPair);
int mb_group_create (mb_group** out, const int32_t* devices, int32_t nDevices);      /* nDevices <= 0: every visible device */
int mb_group_info (const mb_group* g, int32_t* nDevices, int32_t* devices, int32_t* usesNccl);
void mb_group_destroy (mb_group* g);
int mb_group_machine_create (mb_group* g, mb_gmachine** out, int32_t nStates, int32_t nInTok, int32_t nOutTok, int64_t nTrans,
                             const int32_t* src, const int32_t* dst, const int32_t* inTok, const int32_t* outTok, const double* logWeight);
int mb_group_machine_update_weights (mb_gmachine* m, const double* logWeight);
int mb_group_machine_set_option (mb_gmachine* m, const char* name, int32_t value);
int mb_group_machine_info (const mb_gmachine* m, int32_t* nStates, int64_t* nTrans, int32_t* engine);
void mb_group_machine_destroy (mb_gmachine* m);
int mb_group_batch_create (mb_group* g, mb_gbatch** out, int64_t nPairs, const uint8_t* inTokens, const int64_t* inOff,
                           const uint8_t* outTokens, const int64_t* outOff);
int mb_group_batch_set_envelopes (mb_gbatch* b, const int64_t* rowOff, const int64_t* inStart, const int64_t* inEnd);
int mb_group_batch_shard (const mb_gbatch* b, int32_t* deviceOfPair /* [nPairs], may be NULL */, double* cellsPerDevice /* [nDevices], may be NULL */);
void mb_group_batch_destroy (mb_gbatch* b);
int mb_group_forward (mb_gmachine* m, mb_gbatch* b, double* loglike);
int mb_group_backward (mb_gmachine* m, mb_gbatch* b, double* loglike);
int mb_group_viterbi (mb_gmachine* m, mb_gbatch* b, double* score, int64_t* pathLen);
int mb_group_viterbi_paths (mb_gbatch* b, int32_t* pathTrans, const int64_t* pathOff);
int mb_group_viterbi_paths_narrow (mb_gbatch* b, void* pathTrans, int32_t bytesPerId, const int64_t* pathOff);
int mb_group_counts (mb_gmachine* m, mb_gbatch* b, double* counts, double* loglike);
/* mb_pair_counts over the group: each device computes the rows of its pairs, the host places them in list order
 * (no all-reduce; mb_group_last_loglike is left as it was) */
int mb_group_pair_counts (mb_gmachine* m, mb_gbatch* b, double* counts, double* loglike);
int mb_group_last_loglike (const mb_gmachine* m, double* total);      /* summed over all pairs by the last mb_group_counts' all-reduce */
int mb_group_last_kernel_ms (const mb_gbatch* b, double* maxMs, int64_t* nLaunches);      /* slowest device, launches of all */

/* ---- diagnostics (not part of the reference surface) ----
 * Generates the machine-specialised kernels for this machine structure and compiles them with
 * NVRTC for sm_100a WITHOUT touching a device (so it also runs where there is no GPU: the build
 * check and the CPU tests use it).  The compiler log (register / spill report) is copied into
 * log[0..logCap). */
int mb_jit_compile_check (int32_t nStates, int32_t nInTok, int32_t nOutTok, int64_t nTrans,
                          const int32_t* src, const int32_t* dst, const int32_t* inTok, const int32_t* outTok,
                          char* log, int64_t logCap);

/* The tables the generated score kernels of a small machine read, as the host prepares them for these weights
 * (no device needed; the CPU tests drive the generated cell functions with them).  which: 0 forward log weights
 * in row layout, 1 / 2 forward / backward normalised linear weights in row layout, 3 the silent log-weights,
 * 4 the normalised silent weights followed by { originF, originB, resLogF, resLogB }, 5 { normalisation usable,
 * no positive log-weight }.  *n receives the number of doubles; at most cap are copied to out. */
int mb_jit_host_tables (int32_t nStates, int32_t nInTok, int32_t nOutTok, int64_t nTrans,
                        const int32_t* src, const int32_t* dst, const int32_t* inTok, const int32_t* outTok, const double* logWeight,
                        int32_t which, double* out, int64_t cap, int64_t* n);

/* The lane engine's windowed program for a machine without input alphabet, built and EXECUTED ON THE HOST for one read
 * (no device needed: the CPU tests check the program's construction -- window, ring, hubs, push-form sums -- against
 * the oracle).  op: 0 scaled linear sums, 1 max-plus (Viterbi), 2 log-sum-exp.  info[8] = { usable, window states, ring
 * slots, hub sources, hub destinations, live states, records, back-pointer bytes }; backPointers (may be NULL; op 1)
 * receives (outLen + 1) * nStates words, [o][state], in the engine's (kind, index-in-list) format. */
int mb_lane_emulate (int32_t nStates, int32_t nInTok, int32_t nOutTok, int64_t nTrans,
                     const int32_t* src, const int32_t* dst, const int32_t* inTok, const int32_t* outTok, const double* logWeight,
                     const uint8_t* outTokens, int64_t outLen, int32_t op, double* result, int32_t* info, uint32_t* backPointers);

/* The column engine's reading of a generator without input whose states repeat with a period (a profile HMM: column =
 * period of the machine, row = read position), built and EXECUTED ON THE HOST for one read (no device needed: the CPU
 * tests check the analysis, the per-column weight tables and the prefix / suffix programs against known answers).
 * op: 0 log-sum-exp, 1 max-plus.  info[12] = { usable, period, first periodic state, columns, prefix states, suffix states,
 * carried states, accumulators, transition groups per cell, weight slots per column, left-going states, states read
 * from the row above }.  log (may be NULL): the NVRTC log of the generated strip kernel, compiled for sm_100a.  pathLen (may
 * be NULL; op 1): the number of transitions on the Viterbi path, walked back over the program's pointers; at most pathCap
 * ids are written to path. */
int mb_col_emulate (int32_t nStates, int32_t nInTok, int32_t nOutTok, int64_t nTrans,
                    const int32_t* src, const int32_t* dst, const int32_t* inTok, const int32_t* outTok, const double* logWeight,
                    const uint8_t* outTokens, int64_t outLen, int32_t op, double* result, int32_t* info, char* log, int64_t logCap,
                    int32_t* path, int64_t pathCap, int64_t* pathLen);

/* ---- measurement hooks (not part of the reference surface) ----
 * Device time, in milliseconds, of the kernels launched by the last compute call on this batch
 * (CUDA events on the launching stream), and how many kernels that was. */
int mb_last_kernel_ms (const mb_batch* b, double* ms, int64_t* nLaunches);
/* How many pairs of the last mb_forward / mb_backward / mb_counts / mb_pair_counts on this batch the scaled
 * linear-domain sweep handed over to the log-domain kernel (dangerous dynamic range, or -inf). */
int mb_last_redo (const mb_batch* b, int64_t* nPairs);

#ifdef __cplusplus
}
#endif
#endif /* MACHINEBOSS_B200_H */
