// mb_api.cu -- the C ABI declared in include/machineboss_b200.h: handle management, the host-side
// flattening of the evaluated machine (what EvaluatedMachine::init builds, src/eval.cpp:42-70) and
// dispatch to the engines.  No compute happens on the host.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <mutex>

#include "mb_internal.h"

namespace mb {

// per-thread library state: a host thread per GPU sets its own device, engine and options without
// touching another thread's
static thread_local std::string g_error;
static thread_local int g_device = 0;
static thread_local int g_forceEngine = -1;
static thread_local Options g_options;

static const char* const kOptionNames[] = {
  "verbose",                                                  // 1: engines report their launch geometry and flags on stderr
  "jit_narrow", "jit_no_linear", "jit_c", "jit_cv", "jit_minblocks", "jit_minblocks_v", "jit_minblocks_linv", "jit_minblocks_lin", "jit_minblocks_cnt", "jit_threads",
  "jit_tb_budget_mb", "jit_f_budget_mb",                      // cap on one chunk of back-pointer / stored-Forward scratch (tests force several chunks)
  "jit_chunks",                                               // pairs of a Viterbi call are traced back and copied out in this many pipeline stages
  "jit_no_norm",                                              // 1: never use the normalised linear kernels (score module)
  "jit_unroll",                                               // unroll factor of the steady-state step loop (1 - 4)
  "jit_fit_c",                                                // > 0: sweep with a score module of this many columns per lane whenever the batch fits one strip; 0: never fit a module to a batch
  "jit_split",                                                // 0: never split a pair over the warps of a CTA, 1: always (when it has more than one strip)
  "lane_r", "lane_warps", "no_lane", "lane_old", "lane_bs", "lane_la", "lane_wn", "lane_host_only", "lane_warps_per_cta", "wide_g", "wide_w", "no_big", "big_warps", "big_debug", "big_no_fold", "big_early_store", "big_smem_kb",
  "no_col", "col_no_traceback", "col_bp_budget_mb", "col_c", "col_sil_regs", "col_threads", "col_minblocks", "col_r", "col_bnd_budget_mb",      // column engine (mb_col.cu)
};

Options thread_options() { return g_options; }
void set_thread_options (const Options& o) { g_options = o; }
int thread_engine() { return g_forceEngine; }

bool option_known (const char* name) {
  for (const char* n: kOptionNames) if (!strcmp (n, name)) return true;
  return false;
}

void set_error (const std::string& msg) { g_error = msg; }

bool cuda_ok (cudaError_t e, const char* what) {
  if (e == cudaSuccess) return true;
  set_error (std::string ("CUDA error: ") + cudaGetErrorString (e) + " in " + what);
  return false;
}

int timing_begin (mb_batch* b) {
  b->lastMs = 0;
  b->lastLaunches = 0;
  MB_CUDA (cudaEventRecord (b->evStart, b->stream));
  return 0;
}

int timing_end (mb_batch* b, int64_t launches) {
  MB_CUDA (cudaEventRecord (b->evStop, b->stream));
  MB_CUDA (cudaEventSynchronize (b->evStop));
  float ms = 0;
  MB_CUDA (cudaEventElapsedTime (&ms, b->evStart, b->evStop));
  b->lastMs = ms;
  b->lastLaunches = launches;
  return 0;
}

// A small caching pool of freed workspace blocks per device: a batch created for one call (the
// host mirror's ForwardMatrix, the end-to-end bench leg) would otherwise pay cudaMalloc + cudaFree
// of its scratch (10 GB of back-pointers for the 10 k batch) on every call.
struct PoolBlock { void* p; size_t bytes; int device; };
static std::vector<PoolBlock> g_pool;
static std::mutex g_poolMutex;
static const size_t kPoolLimitBytes = (size_t) 48 << 30;

static void* pool_take (int device, size_t bytes, size_t* blockBytes) {
  std::lock_guard<std::mutex> lock (g_poolMutex);
  int best = -1;
  for (size_t n = 0; n < g_pool.size(); ++n)
    if (g_pool[n].device == device && g_pool[n].bytes >= bytes && g_pool[n].bytes <= 2 * bytes + (1 << 20)
        && (best < 0 || g_pool[n].bytes < g_pool[best].bytes)) best = (int) n;
  if (best < 0) return nullptr;
  void* p = g_pool[best].p;
  *blockBytes = g_pool[best].bytes;
  g_pool.erase (g_pool.begin() + best);
  return p;
}

static void pool_trim (int device, size_t keepBytes) {   // free pooled blocks until at most keepBytes remain
  std::lock_guard<std::mutex> lock (g_poolMutex);
  size_t total = 0;
  for (auto& bl: g_pool) if (bl.device == device) total += bl.bytes;
  for (size_t n = 0; n < g_pool.size() && total > keepBytes;) {
    if (g_pool[n].device == device) { cudaFree (g_pool[n].p); total -= g_pool[n].bytes; g_pool.erase (g_pool.begin() + n); }
    else ++n;
  }
}

// whether a block of the pool would serve a request of `bytes` (same rule as pool_take)
bool ws_pool_fits (int device, size_t bytes) {
  bytes = (bytes + 255) & ~(size_t) 255;
  std::lock_guard<std::mutex> lock (g_poolMutex);
  for (auto& bl: g_pool) if (bl.device == device && bl.bytes >= bytes && bl.bytes <= 2 * bytes + (1 << 20)) return true;
  return false;
}

size_t ws_pool_bytes (int device) {
  std::lock_guard<std::mutex> lock (g_poolMutex);
  size_t total = 0;
  for (auto& bl: g_pool) if (bl.device == device) total += bl.bytes;
  return total;
}

void ws_release (mb_batch* b, int slot) {
  if (b->ws[slot].p) {
    if (b->ws[slot].bytes <= kPoolLimitBytes / 2) {
      { std::lock_guard<std::mutex> lock (g_poolMutex); g_pool.push_back (PoolBlock { b->ws[slot].p, b->ws[slot].bytes, b->device }); }
      pool_trim (b->device, kPoolLimitBytes);
    } else cudaFree (b->ws[slot].p);
  }
  b->ws[slot].p = nullptr;
  b->ws[slot].bytes = 0;
}

void ws_release_all (mb_batch* b) { for (int s = 0; s < WS_NSLOTS; ++s) ws_release (b, s); }

size_t ws_bytes (const mb_batch* b, int slot) { return b->ws[slot].bytes; }

void* ws_reserve (mb_batch* b, int slot, size_t bytes) {
  if (bytes == 0) bytes = 8;
  if (b->ws[slot].bytes >= bytes) return b->ws[slot].p;
  ws_release (b, slot);
  bytes = (bytes + 255) & ~(size_t) 255;
  size_t got = bytes;
  void* p = pool_take (b->device, bytes, &got);
  if (!p) {
    got = bytes;
    cudaError_t e = cudaMalloc (&p, bytes);   // never evicts other slots: callers may hold pointers into them
    if (e != cudaSuccess) { cudaGetLastError(); pool_trim (b->device, 0); e = cudaMalloc (&p, bytes); }
    if (!cuda_ok (e, "cudaMalloc (workspace)")) { cudaGetLastError(); return nullptr; }
  }
  b->ws[slot].p = p;
  b->ws[slot].bytes = got;
  return p;
}

// pooled allocation for a batch's own buffers (tokens, packed paths): same pool as the workspace
static void* pooled_alloc (int device, size_t bytes, size_t* got) {
  bytes = (std::max<size_t> (bytes, 8) + 255) & ~(size_t) 255;
  void* p = pool_take (device, bytes, got);
  if (p) return p;
  *got = bytes;
  cudaError_t e = cudaMalloc (&p, bytes);
  if (e != cudaSuccess) { cudaGetLastError(); pool_trim (device, 0); e = cudaMalloc (&p, bytes); }
  if (!cuda_ok (e, "cudaMalloc")) { cudaGetLastError(); return nullptr; }
  return p;
}

static void pooled_free (int device, void* p, size_t bytes) {
  if (!p) return;
  if (bytes <= kPoolLimitBytes / 2) {
    { std::lock_guard<std::mutex> lock (g_poolMutex); g_pool.push_back (PoolBlock { p, bytes, device }); }
    pool_trim (device, kPoolLimitBytes);
  } else cudaFree (p);
}

// room for `need` packed path entries in b->dPaths, keeping what is already there (chunked tracebacks append)
int paths_reserve (mb_batch* b, int64_t need) {
  if (need <= b->pathsCapacity) return 0;
  const int64_t want = std::max<int64_t> (need, 2 * b->pathsCapacity);
  size_t got = 0;
  int32_t* p = (int32_t*) pooled_alloc (b->device, (size_t) want * 4, &got);
  if (!p) return 1;
  if (b->dPaths) {
    MB_CUDA (cudaMemcpyAsync (p, b->dPaths, (size_t) b->pathsCapacity * 4, cudaMemcpyDeviceToDevice, b->stream));
    MB_CUDA (cudaStreamSynchronize (b->stream));
    pooled_free (b->device, b->dPaths, b->pathsBytes);
  }
  b->dPaths = p;
  b->pathsBytes = got;
  b->pathsCapacity = (int64_t) (got / 4);
  return 0;
}

int paths_place (mb_batch* b, const int64_t* pairs, int64_t n, const int64_t* dLen, int64_t* dOutOff) {
  std::vector<int64_t> len ((size_t) n), off ((size_t) n);
  MB_CUDA (cudaMemcpyAsync (len.data(), dLen, (size_t) n * 8, cudaMemcpyDeviceToHost, b->stream));
  MB_CUDA (cudaStreamSynchronize (b->stream));
  for (int64_t q = 0; q < n; ++q) {
    off[q] = b->pathsPacked;
    b->pathStart[pairs[q]] = b->pathsPacked;
    b->pathLen[pairs[q]] = len[q];
    b->pathsPacked += len[q];
  }
  if (paths_reserve (b, b->pathsPacked)) return 1;
  MB_CUDA (cudaMemcpyAsync (dOutOff, off.data(), (size_t) n * 8, cudaMemcpyHostToDevice, b->stream));
  return 0;
}

// Stable counting sort of the transitions into token-indexed lists (see DevCsr).
static void build_csr (const mb_machine* m, bool incoming, HostCsr& c) {
  const int64_t T = m->T;
  const int nIn1 = m->nIn + 1, nOut1 = m->nOut + 1;
  const int64_t nKeys = (int64_t) m->S * nIn1 * nOut1;
  auto keyOf = [&] (int64_t t) {
    const int st = incoming ? m->dst[t] : m->src[t];
    return ((int64_t) st * nIn1 + m->in[t]) * nOut1 + m->out[t];
  };
  // A silent transition that does not advance can only sit on state 0 (machine.cpp:759 exempts it from
  // isAdvancingMachine).  In the reference's fill it reads the cell being computed, which still holds the
  // -inf it was initialised with (dpmatrix.defs.h:36), so it never contributes: it is left out of the lists.
  std::vector<int64_t> order;
  order.reserve ((size_t) T);
  for (int64_t t = 0; t < T; ++t)
    if (!(m->in[t] == 0 && m->out[t] == 0 && m->dst[t] <= m->src[t])) order.push_back (t);
  const int64_t nKept = (int64_t) order.size();
  if (!incoming)   // destination ascending, ties by id; ids already ascend with the source state
    std::stable_sort (order.begin(), order.end(), [&] (int64_t a, int64_t b) { return m->dst[a] < m->dst[b]; });
  c.off.assign ((size_t) nKeys + 1, 0);
  for (int64_t t: order) c.off[keyOf (t) + 1]++;
  for (int64_t k = 0; k < nKeys; ++k) c.off[k + 1] += c.off[k];
  std::vector<int64_t> pos (c.off.begin(), c.off.end() - 1);
  c.other.resize ((size_t) nKept);
  c.id.resize ((size_t) nKept);
  c.lw.resize ((size_t) nKept);
  for (int64_t n = 0; n < nKept; ++n) {
    const int64_t t = order[n];
    const int64_t p = pos[keyOf (t)]++;
    c.other[p] = incoming ? m->src[t] : m->dst[t];
    c.id[p] = (int32_t) t;
    c.lw[p] = m->lw[t];
  }
}

static void build_levels (const mb_machine* m, bool forward, std::vector<int32_t>& off, std::vector<int32_t>& states) {
  const int S = m->S;
  std::vector<int32_t> level ((size_t) S, 0);
  // silent transitions go to strictly higher states (checked at creation), so one ordered pass suffices
  std::vector<std::vector<int32_t>> silentTo ((size_t) S);   // forward: sources of silent edges into s; backward: destinations out of s
  for (int64_t t = 0; t < m->T; ++t)
    if (m->in[t] == 0 && m->out[t] == 0 && m->src[t] < m->dst[t]) {
      if (forward) silentTo[m->dst[t]].push_back (m->src[t]);
      else silentTo[m->src[t]].push_back (m->dst[t]);
    }
  int maxLevel = 0;
  if (forward)
    for (int s = 0; s < S; ++s) { for (int p: silentTo[s]) level[s] = std::max (level[s], level[p] + 1); maxLevel = std::max (maxLevel, level[s]); }
  else
    for (int s = S - 1; s >= 0; --s) { for (int p: silentTo[s]) level[s] = std::max (level[s], level[p] + 1); maxLevel = std::max (maxLevel, level[s]); }
  off.assign ((size_t) maxLevel + 2, 0);
  for (int s = 0; s < S; ++s) off[level[s] + 1]++;
  for (int l = 0; l <= maxLevel; ++l) off[l + 1] += off[l];
  states.resize ((size_t) S);
  std::vector<int32_t> pos (off.begin(), off.end() - 1);
  for (int s = 0; s < S; ++s) states[pos[level[s]]++] = s;
}

template<class T> static size_t blob_reserve (size_t& bytes, const std::vector<T>& v) {
  const size_t at = (bytes + 255) & ~(size_t) 255;
  bytes = at + std::max<size_t> (v.size(), 1) * sizeof (T);
  return at;
}

static int upload_machine (mb_machine* m) {
  size_t bytes = 0;
  const size_t oIncOff = blob_reserve (bytes, m->hInc.off), oIncOther = blob_reserve (bytes, m->hInc.other),
    oIncId = blob_reserve (bytes, m->hInc.id), oIncLw = blob_reserve (bytes, m->hInc.lw),
    oOutOff = blob_reserve (bytes, m->hOut.off), oOutOther = blob_reserve (bytes, m->hOut.other),
    oOutId = blob_reserve (bytes, m->hOut.id), oOutLw = blob_reserve (bytes, m->hOut.lw),
    oFLO = blob_reserve (bytes, m->fwdLevelOff), oFLS = blob_reserve (bytes, m->fwdLevelStates),
    oBLO = blob_reserve (bytes, m->bwdLevelOff), oBLS = blob_reserve (bytes, m->bwdLevelStates);
  std::vector<char> host (bytes, 0);
  auto put = [&] (size_t at, const void* p, size_t n) { if (n) memcpy (host.data() + at, p, n); };
  put (oIncOff, m->hInc.off.data(), m->hInc.off.size() * 8); put (oIncOther, m->hInc.other.data(), m->hInc.other.size() * 4);
  put (oIncId, m->hInc.id.data(), m->hInc.id.size() * 4); put (oIncLw, m->hInc.lw.data(), m->hInc.lw.size() * 8);
  put (oOutOff, m->hOut.off.data(), m->hOut.off.size() * 8); put (oOutOther, m->hOut.other.data(), m->hOut.other.size() * 4);
  put (oOutId, m->hOut.id.data(), m->hOut.id.size() * 4); put (oOutLw, m->hOut.lw.data(), m->hOut.lw.size() * 8);
  put (oFLO, m->fwdLevelOff.data(), m->fwdLevelOff.size() * 4); put (oFLS, m->fwdLevelStates.data(), m->fwdLevelStates.size() * 4);
  put (oBLO, m->bwdLevelOff.data(), m->bwdLevelOff.size() * 4); put (oBLS, m->bwdLevelStates.data(), m->bwdLevelStates.size() * 4);
  MB_CUDA (cudaSetDevice (m->device));
  MB_CUDA (cudaMalloc (&m->dBlob, bytes));
  MB_CUDA (cudaMemcpy (m->dBlob, host.data(), bytes, cudaMemcpyHostToDevice));
  m->blobBytes = bytes;
  m->incLwOffset = oIncLw;
  m->outLwOffset = oOutLw;
  char* d = (char*) m->dBlob;
  DevMachine& dm = m->dev;
  dm.S = m->S; dm.nIn1 = m->nIn + 1; dm.nOut1 = m->nOut + 1;
  dm.inc = { (const int64_t*) (d + oIncOff), (const int32_t*) (d + oIncOther), (const int32_t*) (d + oIncId), (const double*) (d + oIncLw) };
  dm.out = { (const int64_t*) (d + oOutOff), (const int32_t*) (d + oOutOther), (const int32_t*) (d + oOutId), (const double*) (d + oOutLw) };
  dm.nFwdLevels = (int32_t) m->fwdLevelOff.size() - 1;
  dm.nBwdLevels = (int32_t) m->bwdLevelOff.size() - 1;
  dm.fwdLevelOff = (const int32_t*) (d + oFLO); dm.fwdLevelStates = (const int32_t*) (d + oFLS);
  dm.bwdLevelOff = (const int32_t*) (d + oBLO); dm.bwdLevelStates = (const int32_t*) (d + oBLS);
  return 0;
}

}  // namespace mb

using namespace mb;

// smallest and largest token of each sequence set, r = { minX, maxX, minY, maxY } (preset to 255, 0, 255, 0):
// checked against the machine's alphabets by every compute call (a token beyond them would index past the
// emission tables; 0 is epsilon and never appears in data)
__global__ void token_range_kernel (const uint8_t* __restrict__ x, int64_t nx, const uint8_t* __restrict__ y, int64_t ny, int* __restrict__ r) {
  int lo[2] = { 255, 255 }, hi[2] = { 0, 0 };
  const int64_t stride = (int64_t) gridDim.x * blockDim.x, t0 = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  for (int64_t q = t0; q < nx; q += stride) { const int v = x[q]; lo[0] = min (lo[0], v); hi[0] = max (hi[0], v); }
  for (int64_t q = t0; q < ny; q += stride) { const int v = y[q]; lo[1] = min (lo[1], v); hi[1] = max (hi[1], v); }
#pragma unroll
  for (int w = 0; w < 2; ++w) {
    lo[w] = __reduce_min_sync (0xffffffffu, lo[w]);
    hi[w] = __reduce_max_sync (0xffffffffu, hi[w]);
  }
  if ((threadIdx.x & 31) == 0) {
    if (lo[0] < 255) atomicMin (r + 0, lo[0]);
    if (hi[0] > 0) atomicMax (r + 1, hi[0]);
    if (lo[1] < 255) atomicMin (r + 2, lo[1]);
    if (hi[1] > 0) atomicMax (r + 3, hi[1]);
  }
}

template<class T>
__global__ void narrow_ids_kernel (const int32_t* __restrict__ in, T* __restrict__ out, int64_t n) {
  for (int64_t q = (int64_t) blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (int64_t) gridDim.x * blockDim.x) out[q] = (T) in[q];
}

extern "C" {

const char* mb_last_error (void) { return g_error.c_str(); }
int mb_version (void) { return 100; }

int mb_set_kernel_cache_dir (const char* dir) { rt_set_cache_dir (dir); return 0; }

int mb_device_count (int* count) {
  MB_CUDA (cudaGetDeviceCount (count));
  return 0;
}

int mb_set_device (int device) {
  MB_CUDA (cudaSetDevice (device));
  g_device = device;
  return 0;
}

int mb_set_engine (int engine) {
  if (engine < -1 || engine > MB_ENGINE_WIDE) { set_error ("mb_set_engine: unknown engine"); return 1; }
  g_forceEngine = engine;
  return 0;
}

int mb_set_option (const char* name, int32_t value) {
  if (!name || !option_known (name)) { set_error (std::string ("mb_set_option: unknown option '") + (name ? name : "") + "'"); return 1; }
  if (value == MB_OPTION_UNSET) g_options.unset (name); else g_options.set (name, value);
  return 0;
}

int mb_machine_set_option (mb_machine* m, const char* name, int32_t value) {
  if (!m) { set_error ("null machine"); return 1; }
  if (!name || !option_known (name)) { set_error (std::string ("mb_machine_set_option: unknown option '") + (name ? name : "") + "'"); return 1; }
  if (value == MB_OPTION_UNSET) m->opt.unset (name); else m->opt.set (name, value);
  return 0;
}

int mb_machine_create (mb_machine** out, int32_t nStates, int32_t nInTok, int32_t nOutTok, int64_t nTrans,
                       const int32_t* src, const int32_t* dst, const int32_t* inTok, const int32_t* outTok,
                       const double* logWeight) {
  if (!out) { set_error ("mb_machine_create: null output"); return 1; }
  *out = nullptr;
  if (nStates < 1) { set_error ("EvaluatedMachine has no states"); return 1; }   // eval.cpp:77
  if (nInTok < 0 || nOutTok < 0 || nInTok > 255 || nOutTok > 255) { set_error ("mb_machine_create: alphabets must have 0..255 symbols"); return 1; }
  if (nTrans < 0 || nTrans > 0x7fffffff) { set_error ("mb_machine_create: bad transition count"); return 1; }
  for (int64_t t = 0; t < nTrans; ++t) {
    if (src[t] < 0 || src[t] >= nStates || dst[t] < 0 || dst[t] >= nStates || inTok[t] < 0 || inTok[t] > nInTok || outTok[t] < 0 || outTok[t] > nOutTok) {
      set_error ("mb_machine_create: transition " + std::to_string (t) + " is out of range"); return 1;
    }
    if (t && src[t] < src[t - 1]) { set_error ("mb_machine_create: transitions must be listed by ascending source state (eval.cpp:49-69)"); return 1; }
    // machine.cpp:758-764 isAdvancingMachine, asserted at eval.cpp:44 (state 0 is not checked there)
    if (src[t] >= 1 && inTok[t] == 0 && outTok[t] == 0 && dst[t] <= src[t]) { set_error ("Machine is not topologically sorted"); return 1; }
  }
  mb_machine* m = new mb_machine;
  m->device = g_device;
  m->opt = g_options;
  m->S = nStates; m->nIn = nInTok; m->nOut = nOutTok; m->T = nTrans;
  m->src.assign (src, src + nTrans); m->dst.assign (dst, dst + nTrans);
  m->in.assign (inTok, inTok + nTrans); m->out.assign (outTok, outTok + nTrans);
  m->lw.assign (logWeight, logWeight + nTrans);
  build_csr (m, true, m->hInc);
  build_csr (m, false, m->hOut);
  build_levels (m, true, m->fwdLevelOff, m->fwdLevelStates);
  build_levels (m, false, m->bwdLevelOff, m->bwdLevelStates);
  if (upload_machine (m)) { mb_machine_destroy (m); return 1; }
  // Engine choice.  A forced engine that cannot take the machine is an error; in automatic mode a
  // failing preparation (NVRTC unavailable, tables too large, ...) falls through to the next engine --
  // the generic engine, already uploaded, runs any machine.
  std::string why;
  const bool automatic = g_forceEngine < 0;
  bool chosen = g_forceEngine == MB_ENGINE_GENERIC;
  if (!chosen && (g_forceEngine == MB_ENGINE_JIT || (automatic && jit_supported (m, &why)))) {
    if (!jit_supported (m, &why)) { set_error ("mb_set_engine(JIT): " + why); mb_machine_destroy (m); return 1; }
    if (jit_prepare (m) == 0) { m->engine = MB_ENGINE_JIT; chosen = true; }
    else if (!automatic) { mb_machine_destroy (m); return 1; }
    else jit_destroy (m);
  }
  if (!chosen && (g_forceEngine == MB_ENGINE_WIDE || (automatic && (wide_supported (m, &why) || m->nIn == 0)))) {
    // a machine without input alphabet only ever sees batches without input sequences, which the lane
    // engine (mb_lane.cu) sweeps whatever the number of states; the two-dimensional strip sweep needs
    // a cell to fit in shared memory
    bool ok = true;
    if (wide_supported (m, &why)) { ok = wide_prepare (m) == 0; if (!ok) wide_destroy (m); }
    else if (m->nIn != 0) { set_error ("mb_set_engine(WIDE): " + why); mb_machine_destroy (m); return 1; }
    if (ok) { m->engine = MB_ENGINE_WIDE; chosen = true; }
    else if (!automatic && m->nIn != 0) { mb_machine_destroy (m); return 1; }
    else if (m->nIn == 0) { m->engine = MB_ENGINE_WIDE; chosen = true; }      // the lane sweep needs no wide tables
  }
  *out = m;
  return 0;
}

int mb_machine_update_weights (mb_machine* m, const double* logWeight) {
  if (!m) { set_error ("null machine"); return 1; }
  m->lw.assign (logWeight, logWeight + m->T);
  for (size_t p = 0; p < m->hInc.id.size(); ++p) { m->hInc.lw[p] = m->lw[m->hInc.id[p]]; m->hOut.lw[p] = m->lw[m->hOut.id[p]]; }
  MB_CUDA (cudaSetDevice (m->device));
  if (!m->hInc.lw.empty()) {
    MB_CUDA (cudaMemcpy ((char*) m->dBlob + m->incLwOffset, m->hInc.lw.data(), m->hInc.lw.size() * 8, cudaMemcpyHostToDevice));
    MB_CUDA (cudaMemcpy ((char*) m->dBlob + m->outLwOffset, m->hOut.lw.data(), m->hOut.lw.size() * 8, cudaMemcpyHostToDevice));
  }
  if (lane_update_weights (m) || col_update_weights (m)) return 1;
  const int rc = big_update_weights (m);
  if (rc == 2) {      // the new weights' ratios changed which insert groups are proportional: generate the big engine again
    big_destroy (m);
    if (big_supported (m, nullptr) && big_prepare (m)) big_destroy (m);      // (without it the wide engine's sweeps serve)
  } else if (rc) return 1;
  return wide_update_weights (m) || jit_update_weights (m);
}

int mb_machine_info (const mb_machine* m, int32_t* nStates, int64_t* nTrans, int32_t* engine) {
  if (!m) { set_error ("null machine"); return 1; }
  if (nStates) *nStates = m->S;
  if (nTrans) *nTrans = m->T;
  if (engine) *engine = m->engine;
  return 0;
}

void mb_machine_destroy (mb_machine* m) {
  if (!m) return;
  cudaSetDevice (m->device);
  jit_destroy (m);
  wide_destroy (m);
  lane_destroy (m);
  col_destroy (m);
  big_destroy (m);
  if (m->dBlob) cudaFree (m->dBlob);
  delete m;
}

int mb_batch_create (mb_batch** out, int64_t nPairs, const uint8_t* inTokens, const int64_t* inOff,
                     const uint8_t* outTokens, const int64_t* outOff) {
  if (!out) { set_error ("mb_batch_create: null output"); return 1; }
  *out = nullptr;
  if (nPairs < 0) { set_error ("mb_batch_create: negative pair count"); return 1; }
  for (int64_t k = 0; k < nPairs; ++k)
    if (inOff[k + 1] < inOff[k] || outOff[k + 1] < outOff[k]) { set_error ("mb_batch_create: offsets must be non-decreasing"); return 1; }
  mb_batch* b = new mb_batch;
  b->device = g_device;
  b->nPairs = nPairs;
  b->xOff.assign (inOff, inOff + nPairs + 1);
  b->yOff.assign (outOff, outOff + nPairs + 1);
  const size_t nx = (size_t) (b->xOff[nPairs] - b->xOff[0]), ny = (size_t) (b->yOff[nPairs] - b->yOff[0]);
  const int64_t x0 = b->xOff[0], y0 = b->yOff[0];
  for (auto& v: b->xOff) v -= x0;
  for (auto& v: b->yOff) v -= y0;
  auto fail = [&] () { mb_batch_destroy (b); return 1; };
  if (!cuda_ok (cudaSetDevice (b->device), "cudaSetDevice")) return fail();
  if (!cuda_ok (cudaStreamCreateWithFlags (&b->stream, cudaStreamNonBlocking), "cudaStreamCreate")) return fail();
  if (!cuda_ok (cudaEventCreate (&b->evStart), "cudaEventCreate") || !cuda_ok (cudaEventCreate (&b->evStop), "cudaEventCreate")) return fail();
  // one pooled block: offsets, then the tokens with 16 bytes of slack each so kernels may read whole words past the last token
  {
    const size_t offB = ((size_t) (nPairs + 1) * 8 + 255) & ~(size_t) 255, xB = (nx + 16 + 255) & ~(size_t) 255, yB = (ny + 16 + 255) & ~(size_t) 255;
    char* blk = (char*) pooled_alloc (b->device, 2 * offB + xB + yB + 256, &b->tokBytes);
    if (!blk) return fail();
    b->dTokBlock = blk;
    b->dXOff = (int64_t*) blk; b->dYOff = (int64_t*) (blk + offB);
    b->dX = (uint8_t*) (blk + 2 * offB); b->dY = (uint8_t*) (blk + 2 * offB + xB);
    b->dTokRange = (int*) (blk + 2 * offB + xB + yB);
  }
  if (!cuda_ok (cudaMemsetAsync (b->dX, 1, nx + 16, b->stream), "memset") || !cuda_ok (cudaMemsetAsync (b->dY, 1, ny + 16, b->stream), "memset")) return fail();
  if (nx && !cuda_ok (cudaMemcpyAsync (b->dX, inTokens + x0, nx, cudaMemcpyHostToDevice, b->stream), "H2D tokens")) return fail();
  if (ny && !cuda_ok (cudaMemcpyAsync (b->dY, outTokens + y0, ny, cudaMemcpyHostToDevice, b->stream), "H2D tokens")) return fail();
  if (!cuda_ok (cudaMemcpyAsync (b->dXOff, b->xOff.data(), (size_t) (nPairs + 1) * 8, cudaMemcpyHostToDevice, b->stream), "H2D offsets")
      || !cuda_ok (cudaMemcpyAsync (b->dYOff, b->yOff.data(), (size_t) (nPairs + 1) * 8, cudaMemcpyHostToDevice, b->stream), "H2D offsets"))
    return fail();
  {   // token range, on the device (the host never walks the sequences)
    const int init[4] = { 255, 0, 255, 0 };
    if (!cuda_ok (cudaMemcpyAsync (b->dTokRange, init, sizeof init, cudaMemcpyHostToDevice, b->stream), "H2D")) return fail();
    if (nx + ny) {
      const unsigned grid = (unsigned) std::min<size_t> ((std::max (nx, ny) + 255) / 256, 148 * 8);
      token_range_kernel<<<grid, 256, 0, b->stream>>> (b->dX, (int64_t) nx, b->dY, (int64_t) ny, b->dTokRange);
      if (!cuda_ok (cudaGetLastError(), "token_range_kernel")) return fail();
    }
    if (!cuda_ok (cudaMemcpyAsync (b->tokRange, b->dTokRange, sizeof init, cudaMemcpyDeviceToHost, b->stream), "D2H")) return fail();
  }
  if (!cuda_ok (cudaStreamSynchronize (b->stream), "sync")) return fail();
  b->dev = { nPairs, b->dX, b->dXOff, b->dY, b->dYOff, nullptr, nullptr, nullptr };
  *out = b;
  return 0;
}

int mb_batch_set_envelopes (mb_batch* b, const int64_t* rowOff, const int64_t* inStart, const int64_t* inEnd) {
  if (!b) { set_error ("null batch"); return 1; }
  MB_CUDA (cudaSetDevice (b->device));
  if (b->dEnv) { cudaFree (b->dEnv); b->dEnv = nullptr; }
  b->hasEnv = false;
  b->envOff.clear(); b->envStart.clear(); b->envEnd.clear();
  b->dev.envOff = b->dev.envStart = b->dev.envEnd = nullptr;
  if (!rowOff) return 0;
  const int64_t n = b->nPairs, r0 = rowOff[0];
  bool any = false;
  for (int64_t k = 0; k < n; ++k) {
    const int64_t rows = rowOff[k + 1] - rowOff[k];
    const int64_t Li = b->xOff[k + 1] - b->xOff[k], Lo = b->yOff[k + 1] - b->yOff[k];
    if (rows == 0) continue;
    any = true;
    // DPMatrix::alloc asserts env.fits(seqPair) and env.connected() (dpmatrix.defs.h:31-32, seqpair.cpp:170-180)
    if (rows != Lo + 1) { set_error ("Envelope/sequence mismatch: pair " + std::to_string (k) + " has " + std::to_string (rows) + " envelope rows for output length " + std::to_string (Lo)); return 1; }
    const int64_t* s = inStart + rowOff[k];
    const int64_t* e = inEnd + rowOff[k];
    auto overlapping = [] (int64_t s1, int64_t e1, int64_t s2, int64_t e2) { return !(s1 >= e2 || s2 >= e1); };   // seqpair.h:89-93
    bool conn = overlapping (s[0], e[0], 0, 1);
    for (int64_t y = 0; y <= Lo; ++y) {
      if (s[y] < 0 || e[y] > Li + 1 || s[y] > e[y]) { set_error ("Envelope/sequence mismatch: pair " + std::to_string (k) + " row " + std::to_string (y) + " is outside the input"); return 1; }
      if (y) conn = conn && overlapping (s[y - 1], e[y - 1] + 1, s[y], e[y]);
    }
    conn = conn && overlapping (s[Lo], e[Lo], Li, Li + 1);
    if (!conn) { set_error ("Envelope is not connected: pair " + std::to_string (k)); return 1; }
  }
  if (!any) return 0;
  const int64_t R = rowOff[n] - r0;
  b->envOff.assign (rowOff, rowOff + n + 1);
  for (auto& v: b->envOff) v -= r0;
  b->envStart.assign (inStart + r0, inStart + r0 + R);
  b->envEnd.assign (inEnd + r0, inEnd + r0 + R);
  MB_CUDA (cudaMalloc (&b->dEnv, (size_t) (n + 1 + 2 * R) * 8));
  MB_CUDA (cudaMemcpy (b->dEnv, b->envOff.data(), (size_t) (n + 1) * 8, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (b->dEnv + n + 1, b->envStart.data(), (size_t) R * 8, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (b->dEnv + n + 1 + R, b->envEnd.data(), (size_t) R * 8, cudaMemcpyHostToDevice));
  b->dev.envOff = b->dEnv; b->dev.envStart = b->dEnv + n + 1; b->dev.envEnd = b->dEnv + n + 1 + R;
  b->hasEnv = true;
  return 0;
}

void mb_batch_destroy (mb_batch* b) {
  if (!b) return;
  cudaSetDevice (b->device);
  if (b->dEnv) cudaFree (b->dEnv);
  pooled_free (b->device, b->dTokBlock, b->tokBytes);
  pooled_free (b->device, b->dPaths, b->pathsBytes);
  ws_release_all (b);
  if (b->copyStream) { cudaStreamSynchronize (b->copyStream); cudaStreamDestroy (b->copyStream); }
  if (b->evCopy) cudaEventDestroy (b->evCopy);
  if (b->evStart) cudaEventDestroy (b->evStart);
  if (b->evStop) cudaEventDestroy (b->evStop);
  if (b->stream) cudaStreamDestroy (b->stream);
  delete b;
}

int mb_batch_trim (mb_batch* b) {
  if (!b) { set_error ("null batch"); return 1; }
  MB_CUDA (cudaSetDevice (b->device));
  for (int s = 0; s < WS_NSLOTS; ++s)
    if (b->ws[s].p) { cudaFree (b->ws[s].p); b->ws[s].p = nullptr; b->ws[s].bytes = 0; }
  return 0;
}

static int check_call (const mb_machine* m, const mb_batch* b) {
  if (!m || !b) { set_error ("null handle"); return 1; }
  if (m->device != b->device) { set_error ("machine and batch live on different devices"); return 1; }
  // Tokenizer::tokenize throws on a symbol outside the alphabet (eval.h:33-37); a pre-tokenised batch is held to the same rule
  if (b->tokRange[1] > m->nIn || b->tokRange[3] > m->nOut || (b->tokRange[1] && b->tokRange[0] == 0) || (b->tokRange[3] && b->tokRange[2] == 0)) {
    set_error ("batch tokens are outside the machine's alphabets: input tokens " + std::to_string (b->tokRange[0]) + ".." + std::to_string (b->tokRange[1])
               + " (machine: 1.." + std::to_string (m->nIn) + "), output tokens " + std::to_string (b->tokRange[2]) + ".." + std::to_string (b->tokRange[3])
               + " (machine: 1.." + std::to_string (m->nOut) + "); 0 is epsilon and never appears in data");
    return 1;
  }
  MB_CUDA (cudaSetDevice (m->device));
  return 0;
}

enum Pass { PASS_FORWARD, PASS_VITERBI_PATHS, PASS_VITERBI_SCORES, PASS_BACKWARD, PASS_COUNTS, PASS_MATRIX };
enum Route { ROUTE_ERROR = -1, ROUTE_NONE, ROUTE_JIT, ROUTE_BIG, ROUTE_COL, ROUTE_LANE, ROUTE_WIDE, ROUTE_GENERIC };

// The engine that serves a call, after any lazy preparation it needs (ROUTE_NONE: nothing to do; ROUTE_ERROR: a preparation
// failed, error set).  A failed preparation destroys what it built, so the engine's handle is null again.
static int route_of (mb_machine* m, mb_batch* b, Pass pass) {
  const bool sweep = pass == PASS_FORWARD || pass == PASS_VITERBI_PATHS || pass == PASS_VITERBI_SCORES;
  if (pass == PASS_MATRIX || m->engine == MB_ENGINE_GENERIC) return ROUTE_GENERIC;
  if (m->engine == MB_ENGINE_JIT) {
    // the strip kernels sweep full matrices; with envelopes the wide engine takes the sweeps it can, the generic engine the rest
    if (!b->hasEnv) return ROUTE_JIT;
    if (!sweep || !wide_supported (m, nullptr)) return ROUTE_GENERIC;
    if (!m->wide && wide_prepare (m)) { wide_destroy (m); return ROUTE_ERROR; }
    return ROUTE_WIDE;
  }
  if (!sweep) return ROUTE_GENERIC;
  if (b->nPairs == 0) return ROUTE_NONE;
  if (lane_wanted (m, b)) {      // no input sequences: a read per lane, or the column engine for periodic generators
    if (!m->lane) {
      if (lane_prepare (m)) { lane_destroy (m); return ROUTE_ERROR; }
      if (col_prepare (m, false)) {      // (if it cannot be built, the lane sweeps serve)
        if (m->opt.get ("verbose", 0)) fprintf (stderr, "lane engine: the column engine could not be prepared (%s); using the lane sweeps\n", mb_last_error());
        col_destroy (m);
      }
    }
    const bool colTraces = !(pass == PASS_VITERBI_PATHS && m->opt.get ("col_no_traceback", 0));
    return col_usable (m, pass == PASS_FORWARD) && colTraces ? ROUTE_COL : ROUTE_LANE;
  }
  if (!m->wide) return ROUTE_GENERIC;      // too large for the two-dimensional strip sweep
  if (!b->hasEnv) {      // full matrices of a mid-size machine: the generated thread-per-cell sweep (mb_big.cu)
    if (!m->bigTried) {      // a machine the generator cannot handle after all (NVRTC out of resources, ...) stays with the table-driven sweep
      m->bigTried = true;
      if (big_supported (m, nullptr) && big_prepare (m)) {
        if (m->opt.get ("verbose", 0)) fprintf (stderr, "big engine: not available for this machine (%s); using the wide engine\n", mb_last_error());
        big_destroy (m);
      }
    }
    if (pass == PASS_FORWARD ? big_wanted (m, b) : big_wanted_viterbi (m, b)) return ROUTE_BIG;
  }
  return ROUTE_WIDE;
}

// route_of, and with the verbose option one line on stderr naming the pass and the engine
static int route (mb_machine* m, mb_batch* b, Pass pass) {
  const int r = route_of (m, b, pass);
  if (r != ROUTE_ERROR && m->opt.get ("verbose", 0)) {
    static const char* const passNames[] = { "mb_forward", "mb_viterbi", "mb_viterbi (scores)", "mb_backward", "mb_counts", "mb_matrix" };
    static const char* const engineNames[] = { "no engine (empty batch)", "jit engine", "big engine", "column engine", "lane engine", "wide engine", "generic engine" };
    fprintf (stderr, "%s: %s\n", passNames[pass], engineNames[r]);
  }
  return r;
}

int mb_forward (mb_machine* m, mb_batch* b, double* loglike) {
  if (check_call (m, b)) return 1;
  if (m->engine == MB_ENGINE_WIDE) b->lastRedo = 0;      // (the generic engine, which re-runs nothing, does not set it)
  switch (route (m, b, PASS_FORWARD)) {
    case ROUTE_NONE: return 0;
    case ROUTE_JIT: return jit_forward (m, b, loglike, false);
    case ROUTE_BIG: return big_forward (m, b, loglike);
    case ROUTE_COL: return col_forward (m, b, loglike);
    case ROUTE_LANE: return lane_forward (m, b, loglike);
    case ROUTE_WIDE: return wide_forward (m, b, loglike);
    case ROUTE_GENERIC: return generic_forward (m, b, loglike, false);
    default: return 1;
  }
}

int mb_backward (mb_machine* m, mb_batch* b, double* loglike) {
  if (check_call (m, b)) return 1;
  return route (m, b, PASS_BACKWARD) == ROUTE_JIT ? jit_forward (m, b, loglike, true) : generic_forward (m, b, loglike, true);
}

int mb_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen) {
  if (check_call (m, b)) return 1;
  if (b->copyStream) MB_CUDA (cudaStreamSynchronize (b->copyStream));      // paths of the previous call still on their way out
  b->pathIdLimit = m->T;
  b->pathStart.clear();
  b->pathLen.clear();
  const int r = route (m, b, pathLen ? PASS_VITERBI_PATHS : PASS_VITERBI_SCORES);
  if (pathLen) {      // the engine places each pair's path with paths_place
    b->pathStart.assign ((size_t) b->nPairs, 0);
    b->pathLen.assign ((size_t) b->nPairs, 0);
    b->pathsPacked = 0;
  }
  int rc = 1;
  switch (r) {
    case ROUTE_NONE: rc = 0; break;
    case ROUTE_JIT: rc = jit_viterbi (m, b, score, pathLen); break;
    case ROUTE_BIG: rc = big_viterbi (m, b, score, pathLen); break;
    case ROUTE_COL: rc = col_viterbi (m, b, score, pathLen); break;
    case ROUTE_LANE: rc = lane_viterbi (m, b, score, pathLen); break;
    case ROUTE_WIDE: rc = wide_viterbi (m, b, score, pathLen); break;
    case ROUTE_GENERIC: rc = generic_viterbi (m, b, score, pathLen); break;
  }
  if (rc) { b->pathStart.clear(); b->pathLen.clear(); return 1; }      // no traceback stored
  if (pathLen) for (int64_t k = 0; k < b->nPairs; ++k) pathLen[k] = b->pathLen[k];
  return 0;
}

int mb_viterbi_paths (mb_batch* b, int32_t* pathTrans, const int64_t* pathOff) {
  if (!b) { set_error ("null batch"); return 1; }
  if ((int64_t) b->pathLen.size() != b->nPairs) { set_error ("mb_viterbi_paths: no traceback stored; call mb_viterbi with pathLen first"); return 1; }
  MB_CUDA (cudaSetDevice (b->device));
  // paths are packed on the device in pair order; one D2H copy, then scatter to the caller's offsets
  int64_t total = 0;
  for (int64_t k = 0; k < b->nPairs; ++k) total += b->pathLen[k];
  if (!total) return 0;
  bool contiguous = true;
  for (int64_t k = 0; k < b->nPairs && contiguous; ++k) contiguous = (pathOff[k] - pathOff[0] == b->pathStart[k]);
  if (contiguous) {
    MB_CUDA (cudaMemcpy (pathTrans + pathOff[0], b->dPaths, (size_t) total * 4, cudaMemcpyDeviceToHost));
    return 0;
  }
  std::vector<int32_t> tmp ((size_t) total);
  MB_CUDA (cudaMemcpy (tmp.data(), b->dPaths, (size_t) total * 4, cudaMemcpyDeviceToHost));
  for (int64_t k = 0; k < b->nPairs; ++k)
    memcpy (pathTrans + pathOff[k], tmp.data() + b->pathStart[k], (size_t) b->pathLen[k] * 4);
  return 0;
}

int mb_viterbi_paths_narrow (mb_batch* b, void* pathTrans, int32_t bytesPerId, const int64_t* pathOff) {
  if (!b) { set_error ("null batch"); return 1; }
  if ((int64_t) b->pathLen.size() != b->nPairs) { set_error ("mb_viterbi_paths_narrow: no traceback stored; call mb_viterbi with pathLen first"); return 1; }
  if (bytesPerId == 4) return mb_viterbi_paths (b, (int32_t*) pathTrans, pathOff);
  if (bytesPerId != 1 && bytesPerId != 2) { set_error ("mb_viterbi_paths_narrow: bytesPerId must be 1, 2 or 4"); return 1; }
  if (b->pathIdLimit > (bytesPerId == 1 ? 256 : 65536)) { set_error ("mb_viterbi_paths_narrow: the machine's transition ids do not fit in " + std::to_string (bytesPerId) + " byte(s)"); return 1; }
  MB_CUDA (cudaSetDevice (b->device));
  int64_t total = 0;
  for (int64_t k = 0; k < b->nPairs; ++k) total += b->pathLen[k];
  if (!total) return 0;
  bool contiguous = true;      // the engines pack in their own order (JIT: pair order; wide, lane: longest first)
  for (int64_t k = 0; k < b->nPairs && contiguous; ++k) contiguous = (pathOff[k] - pathOff[0] == b->pathStart[k]);
  void* tmp = ws_reserve (b, WS_PATHNARROW, (size_t) total * bytesPerId);
  if (!tmp) return 1;
  const unsigned grid = (unsigned) std::min<int64_t> ((total + 255) / 256, 148 * 16);
  if (bytesPerId == 1) narrow_ids_kernel<uint8_t><<<grid, 256, 0, b->stream>>> (b->dPaths, (uint8_t*) tmp, total);
  else narrow_ids_kernel<uint16_t><<<grid, 256, 0, b->stream>>> (b->dPaths, (uint16_t*) tmp, total);
  MB_CUDA (cudaGetLastError());
  if (contiguous) {
    MB_CUDA (cudaMemcpyAsync ((char*) pathTrans + pathOff[0] * bytesPerId, tmp, (size_t) total * bytesPerId, cudaMemcpyDeviceToHost, b->stream));
    MB_CUDA (cudaStreamSynchronize (b->stream));
    return 0;
  }
  std::vector<char> host ((size_t) total * bytesPerId);
  MB_CUDA (cudaMemcpyAsync (host.data(), tmp, host.size(), cudaMemcpyDeviceToHost, b->stream));
  MB_CUDA (cudaStreamSynchronize (b->stream));
  for (int64_t k = 0; k < b->nPairs; ++k)
    memcpy ((char*) pathTrans + pathOff[k] * bytesPerId, host.data() + b->pathStart[k] * bytesPerId, (size_t) b->pathLen[k] * bytesPerId);
  return 0;
}

int mb_viterbi_paths_start (mb_batch* b, void* pathTrans, int32_t bytesPerId, const int64_t* pathOff) {
  if (!b) { set_error ("null batch"); return 1; }
  if ((int64_t) b->pathLen.size() != b->nPairs) { set_error ("mb_viterbi_paths_start: no traceback stored; call mb_viterbi with pathLen first"); return 1; }
  if (bytesPerId != 1 && bytesPerId != 2 && bytesPerId != 4) { set_error ("mb_viterbi_paths_start: bytesPerId must be 1, 2 or 4"); return 1; }
  if (bytesPerId < 4 && b->pathIdLimit > (bytesPerId == 1 ? 256 : 65536)) { set_error ("mb_viterbi_paths_start: the machine's transition ids do not fit in " + std::to_string (bytesPerId) + " byte(s)"); return 1; }
  int64_t total = 0;
  for (int64_t k = 0; k < b->nPairs; ++k) total += b->pathLen[k];
  bool contiguous = true;
  for (int64_t k = 0; k < b->nPairs && contiguous; ++k) contiguous = (pathOff[k] - pathOff[0] == b->pathStart[k]);
  if (!contiguous) return mb_viterbi_paths_narrow (b, pathTrans, bytesPerId, pathOff);      // scattered offsets: the blocking path
  if (!total) return 0;
  MB_CUDA (cudaSetDevice (b->device));
  if (!b->copyStream) {
    MB_CUDA (cudaStreamCreateWithFlags (&b->copyStream, cudaStreamNonBlocking));
    MB_CUDA (cudaEventCreateWithFlags (&b->evCopy, cudaEventDisableTiming));
  }
  const void* src = b->dPaths;
  if (bytesPerId < 4) {
    void* tmp = ws_reserve (b, WS_PATHNARROW, (size_t) total * bytesPerId);
    if (!tmp) return 1;
    const unsigned grid = (unsigned) std::min<int64_t> ((total + 255) / 256, 148 * 16);
    if (bytesPerId == 1) narrow_ids_kernel<uint8_t><<<grid, 256, 0, b->stream>>> (b->dPaths, (uint8_t*) tmp, total);
    else narrow_ids_kernel<uint16_t><<<grid, 256, 0, b->stream>>> (b->dPaths, (uint16_t*) tmp, total);
    MB_CUDA (cudaGetLastError());
    src = tmp;
  }
  // the copy engine takes it from here; later kernels on the batch's stream do not wait for it (they never write the paths)
  MB_CUDA (cudaEventRecord (b->evCopy, b->stream));
  MB_CUDA (cudaStreamWaitEvent (b->copyStream, b->evCopy, 0));
  MB_CUDA (cudaMemcpyAsync ((char*) pathTrans + pathOff[0] * bytesPerId, src, (size_t) total * bytesPerId, cudaMemcpyDeviceToHost, b->copyStream));
  return 0;
}

int mb_batch_wait (mb_batch* b) {
  if (!b) { set_error ("null batch"); return 1; }
  if (b->copyStream) MB_CUDA (cudaStreamSynchronize (b->copyStream));
  return 0;
}

int mb_counts (mb_machine* m, mb_batch* b, double* counts, double* loglike) {
  if (check_call (m, b)) return 1;
  return route (m, b, PASS_COUNTS) == ROUTE_JIT ? jit_counts (m, b, counts, loglike) : generic_counts (m, b, counts, loglike);
}

int mb_matrix (mb_machine* m, mb_batch* b, int64_t pair, int32_t kind, double* cells) {
  if (check_call (m, b)) return 1;
  if (!cells) { set_error ("mb_matrix: null output"); return 1; }
  route (m, b, PASS_MATRIX);
  return generic_matrix (m, b, pair, kind, cells);
}

int mb_jit_compile_check (int32_t nStates, int32_t nInTok, int32_t nOutTok, int64_t nTrans,
                          const int32_t* src, const int32_t* dst, const int32_t* inTok, const int32_t* outTok,
                          char* log, int64_t logCap) {
  mb_machine m;
  m.opt = g_options;
  m.S = nStates; m.nIn = nInTok; m.nOut = nOutTok; m.T = nTrans;
  m.src.assign (src, src + nTrans); m.dst.assign (dst, dst + nTrans);
  m.in.assign (inTok, inTok + nTrans); m.out.assign (outTok, outTok + nTrans);
  m.lw.assign ((size_t) nTrans, 0.);
  std::string l;
  const int rc = m.S > 16 ? big_compile_check (&m, &l) : jit_compile_check (&m, &l);      // mid-size machines: the big engine's generated sweep
  if (log && logCap > 0) { strncpy (log, l.c_str(), (size_t) logCap - 1); log[logCap - 1] = 0; }
  return rc;
}

int mb_jit_host_tables (int32_t nStates, int32_t nInTok, int32_t nOutTok, int64_t nTrans,
                        const int32_t* src, const int32_t* dst, const int32_t* inTok, const int32_t* outTok, const double* logWeight,
                        int32_t which, double* out, int64_t cap, int64_t* n) {
  mb_machine m;
  m.opt = g_options;
  m.S = nStates; m.nIn = nInTok; m.nOut = nOutTok; m.T = nTrans;
  m.src.assign (src, src + nTrans); m.dst.assign (dst, dst + nTrans);
  m.in.assign (inTok, inTok + nTrans); m.out.assign (outTok, outTok + nTrans);
  m.lw.assign (logWeight, logWeight + nTrans);
  std::vector<double> v;
  if (jit_host_tables (&m, which, v)) return 1;
  if (n) *n = (int64_t) v.size();
  if (out) for (int64_t q = 0; q < (int64_t) v.size() && q < cap; ++q) out[q] = v[q];
  return 0;
}

int mb_lane_emulate (int32_t nStates, int32_t nInTok, int32_t nOutTok, int64_t nTrans,
                     const int32_t* src, const int32_t* dst, const int32_t* inTok, const int32_t* outTok, const double* logWeight,
                     const uint8_t* outTokens, int64_t outLen, int32_t op, double* result, int32_t* info, uint32_t* backPointers) {
  mb_machine m;
  m.opt = g_options;
  m.opt.set ("lane_host_only", 1);
  m.S = nStates; m.nIn = nInTok; m.nOut = nOutTok; m.T = nTrans;
  m.src.assign (src, src + nTrans); m.dst.assign (dst, dst + nTrans);
  m.in.assign (inTok, inTok + nTrans); m.out.assign (outTok, outTok + nTrans);
  m.lw.assign (logWeight, logWeight + nTrans);
  build_csr (&m, true, m.hInc);
  int rc = lane_prepare (&m);
  int32_t inf[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
  if (!rc) rc = lane2_info (&m, inf);
  if (info) for (int q = 0; q < 8; ++q) info[q] = inf[q];
  std::vector<uint32_t> bp;
  if (!rc && inf[0] && result) rc = lane2_emulate (&m, outTokens, outLen, op, result, backPointers ? &bp : nullptr);
  if (!rc && backPointers) for (size_t q = 0; q < bp.size(); ++q) backPointers[q] = bp[q];
  lane_destroy (&m);
  return rc;
}

int mb_col_emulate (int32_t nStates, int32_t nInTok, int32_t nOutTok, int64_t nTrans,
                    const int32_t* src, const int32_t* dst, const int32_t* inTok, const int32_t* outTok, const double* logWeight,
                    const uint8_t* outTokens, int64_t outLen, int32_t op, double* result, int32_t* info, char* log, int64_t logCap,
                    int32_t* path, int64_t pathCap, int64_t* pathLen) {
  mb_machine m;
  m.opt = g_options;
  m.S = nStates; m.nIn = nInTok; m.nOut = nOutTok; m.T = nTrans;
  m.src.assign (src, src + nTrans); m.dst.assign (dst, dst + nTrans);
  m.in.assign (inTok, inTok + nTrans); m.out.assign (outTok, outTok + nTrans);
  m.lw.assign (logWeight, logWeight + nTrans);
  int rc = col_prepare (&m, true);
  int32_t inf[12];
  col_info (&m, inf);
  if (info) for (int q = 0; q < 12; ++q) info[q] = inf[q];
  std::vector<int64_t> walked;
  if (!rc && inf[0] && result) rc = col_emulate (&m, outTokens, outLen, op, result, pathLen ? &walked : nullptr);
  if (!rc && pathLen) { *pathLen = (int64_t) walked.size(); for (int64_t q = 0; q < (int64_t) walked.size() && q < pathCap; ++q) path[q] = (int32_t) walked[q]; }
  if (!rc && inf[0] && log && logCap > 0) {      // compile the generated strip kernel too (NVRTC, no device)
    std::string l;
    rc = col_compile_check (&m, &l);
    strncpy (log, l.c_str(), (size_t) logCap - 1); log[logCap - 1] = 0;
  }
  col_destroy (&m);
  return rc;
}

int mb_last_kernel_ms (const mb_batch* b, double* ms, int64_t* nLaunches) {
  if (!b) { set_error ("null batch"); return 1; }
  if (ms) *ms = b->lastMs;
  if (nLaunches) *nLaunches = b->lastLaunches;
  return 0;
}

int mb_last_redo (const mb_batch* b, int64_t* nPairs) {
  if (!b) { set_error ("null batch"); return 1; }
  if (nPairs) *nPairs = b->lastRedo;
  return 0;
}

}  // extern "C"
