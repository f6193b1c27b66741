// mb_internal.h -- structures shared by the C-ABI layer and the engines.
#ifndef MB_INTERNAL_H
#define MB_INTERNAL_H

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/machineboss_b200.h"

namespace mb {

// The reference's table covers x in [0, 10) and returns 0 beyond (src/logsumexp.h:20,52-53).
// The device log-sum-exp evaluates log(1+exp(-x)) exactly and applies the same truncation, so it
// tracks the reference's table to the table's interpolation error (3e-10 per operation).
#define MB_LSE_CUTOFF 10.0

enum TransType { T_MATCH = 0, T_DELETE = 1, T_INSERT = 2, T_SILENT = 3 };

// Token-indexed transition lists: the role of EvaluatedMachineState::incoming / outgoing
// (src/eval.h:68-76).  key = (state * nIn1 + inTok) * nOut1 + outTok.  Within a key, entries are in
// the reference's multimap order: other-state ascending, then transition index.
struct DevCsr {
  const int64_t* off;
  const int32_t* other;
  const int32_t* id;
  const double* lw;
};

// Device view of an evaluated machine (passed to kernels by value).
struct DevMachine {
  int32_t S, nIn1, nOut1;
  DevCsr inc, out;
  // silent-dependency levels: states in one level have no silent transitions between them
  int32_t nFwdLevels, nBwdLevels;
  const int32_t* fwdLevelOff;
  const int32_t* fwdLevelStates;
  const int32_t* bwdLevelOff;
  const int32_t* bwdLevelStates;
  // every transition by id (mb_path_posteriors walks caller-supplied paths): source, destination, tokens, log-weight
  int64_t nTrans;
  const int32_t* tSrc;
  const int32_t* tDst;
  const int32_t* tIn;
  const int32_t* tOut;
  const double* tLw;
};

struct DevBatch {
  int64_t nPairs;
  const uint8_t* x;
  const int64_t* xOff;
  const uint8_t* y;
  const int64_t* yOff;
  // envelopes (src/seqpair.h:75-113): pair k's output row o keeps inPos in [envStart[r], envEnd[r]),
  // r = envOff[k] + o; envOff[k+1] == envOff[k] means the full matrix.  All null without envelopes.
  const int64_t* envOff;
  const int64_t* envStart;
  const int64_t* envEnd;
};

struct HostCsr {
  std::vector<int64_t> off;
  std::vector<int32_t> other, id;
  std::vector<double> lw;
};

// Tuning and diagnostic knobs.  mb_set_option sets the calling thread's defaults, which a machine copies when
// it is created; mb_machine_set_option changes one machine.  Nothing on the compute path reads the environment.
struct Options {
  std::vector<std::pair<std::string, int>> kv;
  bool has (const char* name) const { for (auto& e: kv) if (e.first == name) return true; return false; }
  int get (const char* name, int dflt) const { for (auto& e: kv) if (e.first == name) return e.second; return dflt; }
  void set (const char* name, int value) { for (auto& e: kv) if (e.first == name) { e.second = value; return; } kv.emplace_back (name, value); }
  void unset (const char* name) { for (size_t n = 0; n < kv.size(); ++n) if (kv[n].first == name) { kv.erase (kv.begin() + n); return; } }
};
bool option_known (const char* name);
// the calling thread's defaults (mb_set_option, mb_set_engine), for handing them to another thread
Options thread_options();
void set_thread_options (const Options& o);
int thread_engine();

void set_error (const std::string& msg);
bool cuda_ok (cudaError_t e, const char* what);

#define MB_CUDA(call) do { if (!mb::cuda_ok ((call), #call)) return 1; } while (0)

// Packed transition ids of a batch's stored paths (pooled device block) and where each path lies in it.  A batch keeps one
// store for its Viterbi traceback and one for its sampled paths, so neither call overwrites the other's result.
struct PathStore {
  int32_t* dPaths = nullptr;
  std::vector<int64_t> pathStart, pathLen;   // per path: offset into dPaths and length
  int64_t pathsPacked = 0;             // entries of dPaths the current call has placed (paths_place)
  int64_t pathsCapacity = 0;
  size_t pathsBytes = 0;               // size of the pooled block behind dPaths
  int64_t pathIdLimit = 0;             // transition ids of the stored paths are below this (the machine's nTrans)
};

// scratch device memory owned by one scope: cudaMalloc on alloc, cudaFree when the scope ends
struct DevBuf {
  void* p = nullptr;
  ~DevBuf() { if (p) cudaFree (p); }
  int alloc (size_t bytes) { MB_CUDA (cudaMalloc (&p, bytes ? bytes : 8)); return 0; }
  template<class T> T* as() { return (T*) p; }
};

}  // namespace mb

// ---- handles ----
struct mb_machine {
  int device = 0;
  int32_t S = 0, nIn = 0, nOut = 0;
  int64_t T = 0;
  std::vector<int32_t> src, dst, in, out;
  std::vector<double> lw;
  int engine = MB_ENGINE_GENERIC;
  mb::Options opt;         // copied from the creating thread's defaults (mb_set_option)

  // generic engine
  mb::HostCsr hInc, hOut;
  std::vector<int32_t> fwdLevelOff, fwdLevelStates, bwdLevelOff, bwdLevelStates;
  void* dBlob = nullptr;   // one device allocation holding everything below
  size_t blobBytes = 0;
  size_t incLwOffset = 0, outLwOffset = 0, lwOffset = 0;   // byte offsets of the three weight arrays inside the blob
  mb::DevMachine dev {};

  // jit engine (mb_jit.cu)
  void* jit = nullptr;
  // wide engine (mb_wide.cu)
  void* wide = nullptr;
  // lane engine (mb_lane.cu): batches without input sequences on a WIDE machine
  void* lane = nullptr;
  // big engine (mb_big.cu): generated straight-line Forward sweep for mid-size machines on full matrices
  void* big = nullptr;
  bool bigTried = false;
  // column engine (mb_col.cu): periodic generators swept as column = period, row = read position; prepared with the lane engine
  void* col = nullptr;
};

struct mb_batch {
  int device = 0;
  int64_t nPairs = 0;
  std::vector<int64_t> xOff, yOff;    // host copies, for planning
  uint8_t* dX = nullptr;
  uint8_t* dY = nullptr;
  int64_t* dXOff = nullptr;
  int64_t* dYOff = nullptr;
  void* dTokBlock = nullptr;           // the pooled allocation the four pointers above point into
  size_t tokBytes = 0;
  int* dTokRange = nullptr;            // { min, max input token, min, max output token }, computed on the device at creation
  int tokRange[4] = { 255, 0, 255, 0 };
  int64_t* dEnv = nullptr;             // envOff | envStart | envEnd in one allocation (null: full envelopes only)
  bool hasEnv = false;
  std::vector<int64_t> envOff, envStart, envEnd;   // host copies
  mb::DevBatch dev {};
  cudaStream_t stream = nullptr;
  cudaStream_t copyStream = nullptr;   // results on their way to the host while the next call's kernels run (mb_viterbi_paths_start)
  cudaEvent_t evCopy = nullptr;
  cudaEvent_t evStart = nullptr, evStop = nullptr;
  double lastMs = 0;
  int64_t lastLaunches = 0;
  int64_t lastRedo = 0;
  std::vector<int64_t> fullOrder;      // all pairs, longest first (planned once)
  bool wsOrderHoldsFull = false;       // WS_ORDER on the device currently holds fullOrder   // pairs the scaled linear sweep handed to the log-domain kernel in the last call
  // grow-only device workspace, reused across calls on this batch so that steady-state calls do
  // no cudaMalloc / cudaFree (slots: see enum WsSlot)
  struct WsEntry { void* p = nullptr; size_t bytes = 0; } ws[24];
  mb::PathStore viterbiPaths;          // result of the last mb_viterbi with traceback, a path per pair
  mb::PathStore sampledPaths;          // result of the last mb_sample_paths, path k * nSamples + j
  int32_t samplesPerPair = 0;          // nSamples of that call (0: no samples stored)
  mb::PathStore meaPaths;              // result of the last mb_mea, a path per pair
  double* dMeaPost = nullptr;          // posterior of each step of meaPaths, at the same offsets (pooled; meaPostCapacity entries)
  int64_t meaPostCapacity = 0;
  size_t meaPostBytes = 0;
  bool meaStored = false;              // the last mb_mea succeeded
};

namespace mb {

// ---- generic engine (mb_generic.cu) ----
// Each returns 0 on success.  Results are written to host arrays.
int generic_forward (mb_machine* m, mb_batch* b, double* loglike, bool backward);
int generic_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen);
// rows == nullptr: counts[nTrans] summed over the batch (may be null); otherwise pair k's counts to rows[k * nTrans ..)
int generic_counts (mb_machine* m, mb_batch* b, double* counts, double* loglike, double* rows = nullptr);
int generic_matrix (mb_machine* m, mb_batch* b, int64_t pair, int kind, double* cells);
// nSamples paths per pair drawn from the stored Forward matrices into b->sampledPaths (pathLen / pathStart set by the caller's size)
int generic_sample_paths (mb_machine* m, mb_batch* b, int32_t nSamples, uint64_t seed, double* loglike);
// the maximum expected accuracy path of every pair into b->meaPaths and its step posteriors into b->dMeaPost (pathLen / pathStart
// set by the caller's size); gain[k] its gain, loglike[k] (may be null) the Forward log-likelihood
int generic_mea (mb_machine* m, mb_batch* b, double* gain, double* loglike);
// posterior of each step of nPaths given paths: path r of pair pairOfPath[r] is ids[off[r] .. off[r + 1]) (packed), its step
// posteriors go to post[off[r] ..); a path that is not a path of its pair is an error naming the path and the step
int generic_path_posteriors (mb_machine* m, mb_batch* b, int64_t nPaths, const int64_t* pairOfPath, const std::vector<int32_t>& ids,
                             const std::vector<int64_t>& off, std::vector<double>& post);

// ---- jit engine (mb_jit.cu) ----
bool jit_supported (const mb_machine* m, std::string* why);
int jit_prepare (mb_machine* m);
int jit_compile_check (const mb_machine* m, std::string* log);
int jit_host_tables (const mb_machine* m, int which, std::vector<double>& out);
void jit_destroy (mb_machine* m);
int jit_update_weights (mb_machine* m);
int jit_forward (mb_machine* m, mb_batch* b, double* loglike, bool backward);
int jit_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen);
int jit_counts (mb_machine* m, mb_batch* b, double* counts, double* loglike, double* rows = nullptr);      // as generic_counts

// ---- wide engine (mb_wide.cu): Forward log-likelihood and Viterbi for mid-size and large machines ----
bool wide_supported (const mb_machine* m, std::string* why);
int wide_prepare (mb_machine* m);
void wide_destroy (mb_machine* m);
int wide_update_weights (mb_machine* m);
int wide_forward (mb_machine* m, mb_batch* b, double* loglike);
int wide_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen);

// ---- lane engine (mb_lane.cu): a read per lane, for batches without input sequences ----
int lane_prepare (mb_machine* m);
void lane_destroy (mb_machine* m);
int lane_update_weights (mb_machine* m);
bool lane_wanted (const mb_machine* m, const mb_batch* b);      // no input sequences, no envelopes
int lane_forward (mb_machine* m, mb_batch* b, double* loglike);
int lane_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen);
// the log-domain sweep over a subset of the batch, results into dResult[pair] (device): where the column engine sends the reads it flags
int lane_forward_log_subset (mb_machine* m, mb_batch* b, const std::vector<int64_t>& pairs, double* dResult, int32_t* dFlag);
std::vector<int64_t> lane_order (const mb_batch* b, const std::vector<int64_t>* subset);      // the pairs (all, or a subset), longest read first
// the windowed program of the lane engine, executed for one read on the host (diagnostic; op 0 sum, 1 max, 2 log-sum-exp)
int lane2_emulate (const mb_machine* m, const uint8_t* y, int64_t Lo, int op, double* result, std::vector<uint32_t>* bpOut);
int lane2_info (const mb_machine* m, int32_t* info);      // { usable, window states, ring slots, hub sources, hub destinations, live states, records, back-pointer bytes }

// ---- column engine (mb_col.cu): generators without input whose states repeat with a period (profile HMMs), swept as
// a two-dimensional recurrence by a generated strip kernel; the lane engine serves the sweeps it declines ----
int col_prepare (mb_machine* m, bool hostOnly);      // 0 also when the machine has no such structure (m->col stays null)
void col_destroy (mb_machine* m);
int col_update_weights (mb_machine* m);
bool col_usable (const mb_machine* m, bool sums);
int col_forward (mb_machine* m, mb_batch* b, double* loglike);
int col_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen);
int col_compile_check (const mb_machine* m, std::string* log);
int col_info (const mb_machine* m, int32_t* info);      // { usable, period, first state, columns, prefix, suffix, carried, accumulators, groups, weight slots, left-going, up }
int col_emulate (const mb_machine* m, const uint8_t* y, int64_t Lo, int op, double* result, std::vector<int64_t>* path);      // op 0 log-sum-exp, 1 max (path: the traceback, may be null)

// ---- big engine (mb_big.cu): machine-specialised Forward sweep for mid-size machines (a thread per cell, the cell as
// straight-line code); full two-dimensional matrices only; flagged pairs go back to the wide engine's log-domain sweep ----
bool big_supported (const mb_machine* m, std::string* why);
int big_compile_check (const mb_machine* m, std::string* log);      // generate + NVRTC-compile without a device
int big_prepare (mb_machine* m);
void big_destroy (mb_machine* m);
int big_update_weights (mb_machine* m);
bool big_wanted (const mb_machine* m, const mb_batch* b);
int big_forward (mb_machine* m, mb_batch* b, double* loglike);
bool big_wanted_viterbi (const mb_machine* m, const mb_batch* b);
int big_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen);
int wide_forward_log_subset (mb_machine* m, mb_batch* b, const std::vector<int64_t>& pairs, double* dResult);      // mb_wide.cu

// run-time compilation plumbing shared by the generated engines (mb_jit.cu)
void rt_set_cache_dir (const char* dir);      // compiled modules are kept in / taken from this directory (null or empty: no cache)
int rt_compile (const std::string& source, const char* dumpSuffix, std::vector<char>& cubin, std::string* log);
int rt_load (const std::vector<char>& cubin, void** module);
void rt_unload (void* module);
int rt_function (void* module, const char* name, void** fn);
int rt_global (void* module, const char* name, void** devPtr, size_t* bytes);
int rt_prepare (void* fn, int threads, size_t smemBytes, int* blocksPerSM);
int rt_launch (void* fn, unsigned grid, unsigned threads, size_t smemBytes, cudaStream_t stream, void** params);

// per-batch workspace (mb_api.cu)
enum WsSlot { WS_ORDER = 0, WS_BND, WS_RESULT, WS_RESULT2, WS_TB, WS_TBOFF, WS_F, WS_FOFF, WS_COUNTS, WS_PAIRS, WS_LEN, WS_OUTOFF, WS_COUNTER, WS_FLAG, WS_EF, WS_EFOFF, WS_PATHTMP, WS_PATHTMPOFF, WS_PATHNARROW, WS_ITEMS, WS_ITEMBND, WS_PROG, WS_ROWOF, WS_NSLOTS };
void* ws_reserve (mb_batch* b, int slot, size_t bytes);   // nullptr + error set on failure
void ws_release (mb_batch* b, int slot);
void ws_release_all (mb_batch* b);
size_t ws_bytes (const mb_batch* b, int slot);
size_t ws_pool_bytes (int device);
bool ws_pool_fits (int device, size_t bytes);   // a pooled block would serve this request   // freed blocks kept for reuse; released when an allocation fails
int paths_reserve (mb_batch* b, PathStore& ps, int64_t need);   // room for `need` packed path entries in ps.dPaths (pooled; keeps the content)
int mea_post_reserve (mb_batch* b, int64_t need);   // room for `need` step posteriors in b->dMeaPost (pooled; keeps the content)
// paths rows[0..n) of the store (a pair's index for Viterbi paths), after those the call has placed so far: copies their lengths
// (dLen, device) to the host, sets pathStart / pathLen, grows dPaths to hold them and writes each path's start into dOutOff
// (device) for the id pass
int paths_place (mb_batch* b, PathStore& ps, const int64_t* rows, int64_t n, const int64_t* dLen, int64_t* dOutOff);

// timing helpers
int timing_begin (mb_batch* b);
int timing_end (mb_batch* b, int64_t launches);

}  // namespace mb

#endif
