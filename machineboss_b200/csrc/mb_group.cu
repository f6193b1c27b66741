// mb_group.cu -- one batch over several GPUs of a box (SURVEY.md section 8e; BASELINE north_star: "the
// SeqPairList batch is length-bucketed and sharded across the 8 GPUs of one box; only the EM count reduction
// crosses NVLink, via an NCCL allreduce").
//
// The reference walks its list of sequence pairs in one loop on one core (src/counts.cpp:37-43 for the
// E-step, src/fitter.cpp:23-47 around it, target/boss.cpp:796,826 for -L and -A).  Pairs are independent, so
// here the list is dealt to the devices of a group -- longest-processing-time first by cell count
// (Li+1)(Lo+1), each pair to the least loaded device -- the machine is replicated, and one host thread per
// device drives that device's share through the single-device entry points (mb_forward, mb_viterbi,
// mb_counts) on its own stream.  Forward and Viterbi need no communication: results are gathered by pair
// index.  The E-step has the path's one exchange step: every device's nTrans + 1 doubles (its counts and its
// summed log-likelihood) are summed across devices with ncclAllReduce(sum, ncclDouble), in place in device
// memory, over NVLink.  NCCL is resolved at run time (libnccl.so.2); a group of one device, or a box without
// the library, adds the per-device vectors on the host instead (mb_group_info reports which).
#include <dlfcn.h>
#include <unistd.h>

#include <algorithm>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <queue>
#include <thread>

#include "mb_internal.h"

namespace mb {

// ---------------------------------------------------------------------------------------------
// LPT dealing of pairs to shards
// ---------------------------------------------------------------------------------------------
void shard_pairs (int64_t nPairs, const int64_t* inOff, const int64_t* outOff, int nShards, int32_t* shardOfPair, double* loadOut) {
  std::vector<int64_t> order ((size_t) nPairs);
  std::vector<double> cost ((size_t) nPairs);
  for (int64_t k = 0; k < nPairs; ++k) {
    order[k] = k;
    cost[k] = (double) (inOff[k + 1] - inOff[k] + 1) * (double) (outOff[k + 1] - outOff[k] + 1);
  }
  std::stable_sort (order.begin(), order.end(), [&] (int64_t a, int64_t b) { return cost[a] > cost[b]; });
  typedef std::pair<double, int> Load;      // (cells so far, shard): the smallest load first, ties to the lowest shard
  std::priority_queue<Load, std::vector<Load>, std::greater<Load>> heap;
  for (int s = 0; s < nShards; ++s) heap.push (Load (0., s));
  for (int64_t k: order) {
    Load l = heap.top();
    heap.pop();
    shardOfPair[k] = l.second;
    l.first += cost[k];
    heap.push (l);
  }
  if (loadOut) {
    for (int s = 0; s < nShards; ++s) loadOut[s] = 0;
    for (int64_t k = 0; k < nPairs; ++k) loadOut[shardOfPair[k]] += cost[k];
  }
}

// ---------------------------------------------------------------------------------------------
// NCCL, resolved at run time
// ---------------------------------------------------------------------------------------------
typedef void* nccl_comm;
struct Nccl {
  void* lib = nullptr;
  int (*CommInitAll) (nccl_comm*, int, const int*) = nullptr;
  int (*CommDestroy) (nccl_comm) = nullptr;
  int (*AllReduce) (const void*, void*, size_t, int, int, nccl_comm, cudaStream_t) = nullptr;
  const char* (*GetErrorString) (int) = nullptr;
  bool ok = false;
};
static Nccl g_nccl;
static std::mutex g_ncclMutex;
static const int kNcclFloat64 = 8, kNcclSum = 0;      // nccl.h: ncclDouble = ncclFloat64 = 8, ncclSum = 0

static bool load_nccl() {
  std::lock_guard<std::mutex> lock (g_ncclMutex);
  if (g_nccl.ok) return true;
  if (g_nccl.lib) return false;
  for (const char* name: { "libnccl.so.2", "libnccl.so" }) { g_nccl.lib = dlopen (name, RTLD_NOW | RTLD_GLOBAL); if (g_nccl.lib) break; }
  if (!g_nccl.lib) { g_nccl.lib = (void*) 1; return false; }
  g_nccl.CommInitAll = (decltype (g_nccl.CommInitAll)) dlsym (g_nccl.lib, "ncclCommInitAll");
  g_nccl.CommDestroy = (decltype (g_nccl.CommDestroy)) dlsym (g_nccl.lib, "ncclCommDestroy");
  g_nccl.AllReduce = (decltype (g_nccl.AllReduce)) dlsym (g_nccl.lib, "ncclAllReduce");
  g_nccl.GetErrorString = (decltype (g_nccl.GetErrorString)) dlsym (g_nccl.lib, "ncclGetErrorString");
  g_nccl.ok = g_nccl.CommInitAll && g_nccl.CommDestroy && g_nccl.AllReduce;
  return g_nccl.ok;
}

// ---------------------------------------------------------------------------------------------
// one host thread per device
// ---------------------------------------------------------------------------------------------
struct Worker {
  int device;
  std::thread th;
  std::mutex mu;
  std::condition_variable cv;
  std::function<int()> job;
  bool hasJob = false, done = false, quit = false;
  int rc = 0;
  std::string error;

  explicit Worker (int dev) : device (dev) {
    th = std::thread ([this] {
      mb_set_device (device);      // this thread's handles live on this device (per-thread library state)
      for (;;) {
        std::function<int()> j;
        {
          std::unique_lock<std::mutex> lk (mu);
          cv.wait (lk, [this] { return hasJob || quit; });
          if (quit) return;
          j = job;
        }
        const int r = j();
        const std::string err = r ? std::string (mb_last_error()) : std::string();
        {
          std::lock_guard<std::mutex> lk (mu);
          rc = r; error = err; hasJob = false; done = true;
        }
        cv.notify_all();
      }
    });
  }
  void start (std::function<int()> j) {
    { std::lock_guard<std::mutex> lk (mu); job = std::move (j); hasJob = true; done = false; }
    cv.notify_all();
  }
  int wait() {
    std::unique_lock<std::mutex> lk (mu);
    cv.wait (lk, [this] { return done; });
    return rc;
  }
  ~Worker() {
    { std::lock_guard<std::mutex> lk (mu); quit = true; }
    cv.notify_all();
    if (th.joinable()) th.join();
  }
};

}  // namespace mb

using namespace mb;

struct mb_group {
  std::vector<int> devices;
  std::vector<std::unique_ptr<Worker>> workers;
  std::vector<nccl_comm> comms;      // empty: counts are added on the host
  // machines and batches of the group keep it alive: mb_group_destroy with children still around only marks it, and the last
  // child's destruction frees it (a caller that tears its handles down in any order -- an interpreter at exit -- stays safe)
  int children = 0;
  bool released = false;
  // job(d) on every device's thread at once; the first failure's message becomes this thread's last error
  int run (const std::function<int (int)>& job) {
    for (size_t d = 0; d < workers.size(); ++d) workers[d]->start ([=] { return job ((int) d); });
    int rc = 0;
    for (size_t d = 0; d < workers.size(); ++d)
      if (workers[d]->wait() && !rc) { rc = 1; set_error ("device " + std::to_string (devices[d]) + ": " + workers[d]->error); }
    return rc;
  }
};

struct mb_gmachine {
  mb_group* g = nullptr;
  int32_t S = 0;
  int64_t T = 0;
  std::vector<mb_machine*> m;          // one replica per device
  std::vector<double*> dReduce;        // per device: nTrans + 1 doubles for the all-reduce
  double lastLogLike = 0;              // summed over every pair of the last mb_group_counts
};

struct mb_gbatch {
  mb_group* g = nullptr;
  int64_t nPairs = 0;
  std::vector<int32_t> shardOf;                  // device slot of every pair
  std::vector<std::vector<int64_t>> pairsOf;     // per device slot: its pairs, ascending
  std::vector<mb_batch*> b;
  std::vector<double> load;                      // cells per device slot
};

extern "C" {

int mb_shard_pairs (int64_t nPairs, const int64_t* inOff, const int64_t* outOff, int32_t nShards, int32_t* shardOfPair) {
  if (nPairs < 0 || nShards < 1 || (nPairs && (!inOff || !outOff || !shardOfPair))) { set_error ("mb_shard_pairs: bad arguments"); return 1; }
  shard_pairs (nPairs, inOff, outOff, nShards, shardOfPair, nullptr);
  return 0;
}

int mb_group_create (mb_group** out, const int32_t* devices, int32_t nDevices) {
  if (!out) { set_error ("mb_group_create: null output"); return 1; }
  *out = nullptr;
  int visible = 0;
  MB_CUDA (cudaGetDeviceCount (&visible));
  std::vector<int> devs;
  if (nDevices <= 0) for (int d = 0; d < visible; ++d) devs.push_back (d);      // every visible device
  else for (int n = 0; n < nDevices; ++n) devs.push_back (devices[n]);
  if (devs.empty()) { set_error ("mb_group_create: no CUDA device"); return 1; }
  for (size_t n = 0; n < devs.size(); ++n) {
    if (devs[n] < 0 || devs[n] >= visible) { set_error ("mb_group_create: no device " + std::to_string (devs[n])); return 1; }
    for (size_t q = 0; q < n; ++q) if (devs[q] == devs[n]) { set_error ("mb_group_create: device " + std::to_string (devs[n]) + " listed twice"); return 1; }
  }
  mb_group* g = new mb_group;
  g->devices = devs;
  for (int d: devs) g->workers.emplace_back (new Worker (d));
  if (devs.size() > 1 && load_nccl()) {
    g->comms.assign (devs.size(), nullptr);
    // NCCL announces itself on STANDARD OUTPUT when NCCL_DEBUG is set in the environment ("NCCL version ..."): a program whose
    // standard output is its result (boss_b200 prints JSON) must not have that mixed in, so file descriptor 1 points at
    // standard error while the communicators are made
    fflush (stdout);
    const int savedOut = dup (1);
    if (savedOut >= 0) dup2 (2, 1);
    const int r = g_nccl.CommInitAll (g->comms.data(), (int) devs.size(), devs.data());
    if (savedOut >= 0) { fflush (stdout); dup2 (savedOut, 1); close (savedOut); }
    if (r != 0) g->comms.clear();      // no peer path between these devices: add on the host
  }
  *out = g;
  return 0;
}

int mb_group_info (const mb_group* g, int32_t* nDevices, int32_t* devices, int32_t* usesNccl) {
  if (!g) { set_error ("null group"); return 1; }
  if (nDevices) *nDevices = (int32_t) g->devices.size();
  if (devices) for (size_t d = 0; d < g->devices.size(); ++d) devices[d] = g->devices[d];
  if (usesNccl) *usesNccl = g->comms.empty() ? 0 : 1;
  return 0;
}

static void group_free (mb_group* g) {
  for (nccl_comm c: g->comms) if (c) g_nccl.CommDestroy (c);
  delete g;
}

static void group_child_gone (mb_group* g) {
  if (--g->children == 0 && g->released) group_free (g);
}

void mb_group_destroy (mb_group* g) {
  if (!g) return;
  if (g->children > 0) { g->released = true; return; }
  group_free (g);
}

int mb_group_machine_create (mb_group* g, mb_gmachine** out, int32_t nStates, int32_t nInTok, int32_t nOutTok, int64_t nTrans,
                             const int32_t* src, const int32_t* dst, const int32_t* inTok, const int32_t* outTok, const double* logWeight) {
  if (!g || !out) { set_error ("mb_group_machine_create: null argument"); return 1; }
  *out = nullptr;
  mb_gmachine* gm = new mb_gmachine;
  gm->g = g; gm->S = nStates; gm->T = nTrans;
  ++g->children;
  gm->m.assign (g->devices.size(), nullptr);
  gm->dReduce.assign (g->devices.size(), nullptr);
  const Options opts = thread_options();      // the caller's defaults apply to every replica
  const int engine = thread_engine();
  const int rc = g->run ([&] (int d) {
    set_thread_options (opts);
    mb_set_engine (engine);
    if (mb_machine_create (&gm->m[d], nStates, nInTok, nOutTok, nTrans, src, dst, inTok, outTok, logWeight)) return 1;
    MB_CUDA (cudaMalloc (&gm->dReduce[d], (size_t) (nTrans + 1) * 8));
    return 0;
  });
  if (rc) { const std::string e = mb_last_error(); mb_group_machine_destroy (gm); set_error (e); return 1; }
  *out = gm;
  return 0;
}

int mb_group_machine_update_weights (mb_gmachine* gm, const double* logWeight) {
  if (!gm) { set_error ("null machine"); return 1; }
  return gm->g->run ([&] (int d) { return mb_machine_update_weights (gm->m[d], logWeight); });
}

int mb_group_machine_set_option (mb_gmachine* gm, const char* name, int32_t value) {
  if (!gm) { set_error ("null machine"); return 1; }
  for (mb_machine* m: gm->m) if (m && mb_machine_set_option (m, name, value)) return 1;
  return 0;
}

int mb_group_machine_info (const mb_gmachine* gm, int32_t* nStates, int64_t* nTrans, int32_t* engine) {
  if (!gm || gm->m.empty() || !gm->m[0]) { set_error ("null machine"); return 1; }
  return mb_machine_info (gm->m[0], nStates, nTrans, engine);
}

void mb_group_machine_destroy (mb_gmachine* gm) {
  if (!gm) return;
  gm->g->run ([&] (int d) {
    if (gm->m[d]) mb_machine_destroy (gm->m[d]);
    if (gm->dReduce[d]) cudaFree (gm->dReduce[d]);
    return 0;
  });
  mb_group* g = gm->g;
  delete gm;
  group_child_gone (g);
}

int mb_group_batch_create (mb_group* g, mb_gbatch** out, int64_t nPairs, const uint8_t* inTokens, const int64_t* inOff,
                           const uint8_t* outTokens, const int64_t* outOff) {
  if (!g || !out) { set_error ("mb_group_batch_create: null argument"); return 1; }
  *out = nullptr;
  if (nPairs < 0) { set_error ("mb_group_batch_create: negative pair count"); return 1; }
  for (int64_t k = 0; k < nPairs; ++k)
    if (inOff[k + 1] < inOff[k] || outOff[k + 1] < outOff[k]) { set_error ("mb_group_batch_create: offsets must be non-decreasing"); return 1; }
  const int nDev = (int) g->devices.size();
  mb_gbatch* gb = new mb_gbatch;
  gb->g = g; gb->nPairs = nPairs;
  ++g->children;
  gb->shardOf.assign ((size_t) nPairs, 0);
  gb->load.assign ((size_t) nDev, 0.);
  gb->pairsOf.assign ((size_t) nDev, std::vector<int64_t>());
  gb->b.assign ((size_t) nDev, nullptr);
  shard_pairs (nPairs, inOff, outOff, nDev, gb->shardOf.data(), gb->load.data());
  for (int64_t k = 0; k < nPairs; ++k) gb->pairsOf[gb->shardOf[k]].push_back (k);
  // every device thread gathers its own pairs' tokens and uploads them
  const int rc = g->run ([&] (int d) {
    const std::vector<int64_t>& mine = gb->pairsOf[d];
    std::vector<int64_t> xo (1, 0), yo (1, 0);
    for (int64_t k: mine) { xo.push_back (xo.back() + (inOff[k + 1] - inOff[k])); yo.push_back (yo.back() + (outOff[k + 1] - outOff[k])); }
    std::vector<uint8_t> x ((size_t) xo.back() + 1), y ((size_t) yo.back() + 1);
    for (size_t q = 0; q < mine.size(); ++q) {
      const int64_t k = mine[q];
      if (inOff[k + 1] > inOff[k]) memcpy (x.data() + xo[q], inTokens + inOff[k], (size_t) (inOff[k + 1] - inOff[k]));
      if (outOff[k + 1] > outOff[k]) memcpy (y.data() + yo[q], outTokens + outOff[k], (size_t) (outOff[k + 1] - outOff[k]));
    }
    return mb_batch_create (&gb->b[d], (int64_t) mine.size(), x.data(), xo.data(), y.data(), yo.data());
  });
  if (rc) { const std::string e = mb_last_error(); mb_group_batch_destroy (gb); set_error (e); return 1; }
  *out = gb;
  return 0;
}

int mb_group_batch_set_envelopes (mb_gbatch* gb, const int64_t* rowOff, const int64_t* inStart, const int64_t* inEnd) {
  if (!gb) { set_error ("null batch"); return 1; }
  return gb->g->run ([&] (int d) {
    if (!rowOff) return mb_batch_set_envelopes (gb->b[d], nullptr, nullptr, nullptr);
    std::vector<int64_t> off (1, 0), st, en;
    for (int64_t k: gb->pairsOf[d]) {
      st.insert (st.end(), inStart + rowOff[k], inStart + rowOff[k + 1]);
      en.insert (en.end(), inEnd + rowOff[k], inEnd + rowOff[k + 1]);
      off.push_back ((int64_t) st.size());
    }
    st.push_back (0); en.push_back (0);      // never empty
    return mb_batch_set_envelopes (gb->b[d], off.data(), st.data(), en.data());
  });
}

int mb_group_batch_shard (const mb_gbatch* gb, int32_t* deviceOfPair, double* cellsPerDevice) {
  if (!gb) { set_error ("null batch"); return 1; }
  if (deviceOfPair) for (int64_t k = 0; k < gb->nPairs; ++k) deviceOfPair[k] = gb->g->devices[gb->shardOf[k]];
  if (cellsPerDevice) for (size_t d = 0; d < gb->load.size(); ++d) cellsPerDevice[d] = gb->load[d];
  return 0;
}

void mb_group_batch_destroy (mb_gbatch* gb) {
  if (!gb) return;
  gb->g->run ([&] (int d) { if (gb->b[d]) mb_batch_destroy (gb->b[d]); return 0; });
  mb_group* g = gb->g;
  delete gb;
  group_child_gone (g);
}

}  // extern "C"

static int check_group_call (const mb_gmachine* gm, const mb_gbatch* gb) {
  if (!gm || !gb) { set_error ("null handle"); return 1; }
  if (gm->g != gb->g) { set_error ("machine and batch belong to different groups"); return 1; }
  return 0;
}

// per-pair results of every device, gathered by pair index
template<class F>
static int per_pair (mb_gmachine* gm, mb_gbatch* gb, double* result, F call) {
  return gb->g->run ([&] (int d) {
    const std::vector<int64_t>& mine = gb->pairsOf[d];
    std::vector<double> r (mine.size() + 1);
    if (call (gm->m[d], gb->b[d], r.data())) return 1;
    for (size_t q = 0; q < mine.size(); ++q) result[mine[q]] = r[q];
    return 0;
  });
}

extern "C" {

int mb_group_forward (mb_gmachine* gm, mb_gbatch* gb, double* loglike) {
  if (check_group_call (gm, gb)) return 1;
  return per_pair (gm, gb, loglike, [] (mb_machine* m, mb_batch* b, double* r) { return mb_forward (m, b, r); });
}

int mb_group_backward (mb_gmachine* gm, mb_gbatch* gb, double* loglike) {
  if (check_group_call (gm, gb)) return 1;
  return per_pair (gm, gb, loglike, [] (mb_machine* m, mb_batch* b, double* r) { return mb_backward (m, b, r); });
}

int mb_group_viterbi (mb_gmachine* gm, mb_gbatch* gb, double* score, int64_t* pathLen) {
  if (check_group_call (gm, gb)) return 1;
  return gb->g->run ([&] (int d) {
    const std::vector<int64_t>& mine = gb->pairsOf[d];
    std::vector<double> sc (mine.size() + 1);
    std::vector<int64_t> len (mine.size() + 1, 0);
    if (mb_viterbi (gm->m[d], gb->b[d], sc.data(), pathLen ? len.data() : nullptr)) return 1;
    for (size_t q = 0; q < mine.size(); ++q) { score[mine[q]] = sc[q]; if (pathLen) pathLen[mine[q]] = len[q]; }
    return 0;
  });
}

int mb_group_viterbi_paths_narrow (mb_gbatch* gb, void* pathTrans, int32_t bytesPerId, const int64_t* pathOff) {
  if (!gb) { set_error ("null batch"); return 1; }
  return gb->g->run ([&] (int d) {
    const std::vector<int64_t>& mine = gb->pairsOf[d];
    if (mine.empty()) return 0;
    std::vector<int64_t> off (mine.size());      // each device scatters its pairs' paths to the caller's offsets
    for (size_t q = 0; q < mine.size(); ++q) off[q] = pathOff[mine[q]];
    return mb_viterbi_paths_narrow (gb->b[d], pathTrans, bytesPerId, off.data());
  });
}

int mb_group_viterbi_paths (mb_gbatch* gb, int32_t* pathTrans, const int64_t* pathOff) { return mb_group_viterbi_paths_narrow (gb, pathTrans, 4, pathOff); }

int mb_group_counts (mb_gmachine* gm, mb_gbatch* gb, double* counts, double* loglike) {
  if (check_group_call (gm, gb)) return 1;
  mb_group* g = gb->g;
  const size_t nDev = g->devices.size();
  const size_t T = (size_t) gm->T;
  std::vector<std::vector<double>> part (nDev, std::vector<double> (T + 1, 0.));
  const bool nccl = !g->comms.empty();
  const int rc = g->run ([&] (int d) {
    const std::vector<int64_t>& mine = gb->pairsOf[d];
    std::vector<double> ll (mine.size() + 1, 0.);
    std::vector<double>& v = part[d];
    if (mb_counts (gm->m[d], gb->b[d], counts ? v.data() : nullptr, ll.data())) return 1;
    double sum = 0;
    for (size_t q = 0; q < mine.size(); ++q) { if (loglike) loglike[mine[q]] = ll[q]; sum += ll[q]; }
    v[T] = sum;
    if (nccl) {
      // the exchange step: sum over devices of (counts, log-likelihood), in place in device memory, over NVLink
      cudaStream_t st = gb->b[d]->stream;
      MB_CUDA (cudaMemcpyAsync (gm->dReduce[d], v.data(), (T + 1) * 8, cudaMemcpyHostToDevice, st));
      const int r = g_nccl.AllReduce (gm->dReduce[d], gm->dReduce[d], T + 1, kNcclFloat64, kNcclSum, g->comms[d], st);
      if (r != 0) { set_error (std::string ("ncclAllReduce: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString (r) : "failed")); return 1; }
      MB_CUDA (cudaMemcpyAsync (v.data(), gm->dReduce[d], (T + 1) * 8, cudaMemcpyDeviceToHost, st));
      MB_CUDA (cudaStreamSynchronize (st));
    }
    return 0;
  });
  if (rc) return 1;
  if (!nccl) for (size_t d = 1; d < nDev; ++d) for (size_t t = 0; t <= T; ++t) part[0][t] += part[d][t];
  if (counts) for (size_t t = 0; t < T; ++t) counts[t] = part[0][t];
  gm->lastLogLike = part[0][T];
  return 0;
}

int mb_group_pair_counts (mb_gmachine* gm, mb_gbatch* gb, double* counts, double* loglike) {
  if (check_group_call (gm, gb)) return 1;
  if (!counts) { set_error ("mb_group_pair_counts: null counts (mb_group_counts gives the log-likelihoods alone)"); return 1; }
  const size_t T = (size_t) gm->T;
  return gb->g->run ([&] (int d) {      // each device's rows, scattered into list order; nothing crosses devices
    const std::vector<int64_t>& mine = gb->pairsOf[d];
    std::vector<double> rows (mine.size() * T + 1), ll (mine.size() + 1);
    if (mb_pair_counts (gm->m[d], gb->b[d], rows.data(), ll.data())) return 1;
    for (size_t q = 0; q < mine.size(); ++q) {
      if (T) memcpy (counts + mine[q] * (int64_t) T, rows.data() + q * T, T * 8);
      if (loglike) loglike[mine[q]] = ll[q];
    }
    return 0;
  });
}

int mb_group_last_loglike (const mb_gmachine* gm, double* total) {
  if (!gm) { set_error ("null machine"); return 1; }
  if (total) *total = gm->lastLogLike;
  return 0;
}

int mb_group_last_kernel_ms (const mb_gbatch* gb, double* maxMs, int64_t* nLaunches) {
  if (!gb) { set_error ("null batch"); return 1; }
  double ms = 0;
  int64_t n = 0;
  for (mb_batch* b: gb->b) if (b) { ms = std::max (ms, b->lastMs); n += b->lastLaunches; }
  if (maxMs) *maxMs = ms;
  if (nLaunches) *nLaunches = n;
  return 0;
}

}  // extern "C"
