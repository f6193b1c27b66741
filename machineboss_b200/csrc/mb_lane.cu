// mb_lane.cu -- the lane engine: Forward log-likelihood and Viterbi (+ traceback) of batches WITHOUT
// input sequences (generator machines: a profile HMM, or a profile composed with an error model,
// scoring a million reads -- SURVEY.md section 8, config 5) on machines of any size.
//
//   reference                                              here
//   MappedForwardMatrix::fill / logLike  forward.defs.h:22-55   lane_kernel<OP_SUM>  (scaled linear domain)
//                                                               lane_kernel<OP_LSE>  (log domain: flagged reads, extreme weights)
//   ViterbiMatrix::fill / logLike        viterbi.cpp:18-47      lane_kernel<OP_MAX>  (FP64 add + compare: bit-exact)
//   DPMatrix::traceBack                  dpmatrix.defs.h:82-110 wide_traceback_kernel over the lane-interleaved pointers
//
// Why another mapping.  With no input sequence the matrix of a read is one column of Lo+1 cells, and
// a cell is a sparse matrix-vector product through the silent transitions in dependency order.  A
// profile HMM's delete chain makes that order hundreds of levels deep (488 levels for PF00516, 979
// once composed with protpsw), so spreading the STATES of a cell over lanes (mb_wide.cu) leaves the
// lanes waiting on one another.  Here every LANE owns a READ instead: the 32 reads of a warp walk
// the same transition program in lockstep -- destination states in index order, which is a
// topological order of the silent transitions (eval.cpp:44 requires an advancing machine) -- one
// multiply-add per transition per lane, no barrier anywhere.  The program is a flat stream of
// 16-byte records read through uniform (broadcast) loads; the emitting transitions of a
// destination are stored as the union over output tokens with a token-indexed weight table, so
// that reads with different residues still share the stream.  State vectors live in global memory
// interleaved by lane, v[state][lane], so every load and store of the warp is one 256-byte line;
// two vectors per lane (previous cell, this cell).
//
// Arithmetic as in mb_wide.cu.  Forward: probabilities with one power-of-two frame per cell and
// lane; the previous cell enters through one exact power-of-two factor; a cell whose values span
// more than 2^600 flags the read, and flagged reads are re-run in the log domain.  Viterbi:
// log-weights, FP64 add + strict '<' in the reference's candidate order (insert sources, then
// silent sources, each by ascending source state then transition index), so scores and paths are
// identical to the reference's.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>

#include "mb_internal.h"

namespace mb {

enum { L_SUM = 0, L_MAX = 1, L_LSE = 2 };
#define L_SENT (-(1 << 29))
#define L_SPREAD 600
// record control word: low bits flags, high 16 bits the candidate index (silent terms, Viterbi)
#define L_EMIT 1u      // term reads the previous cell; w holds the row of the token-indexed tables
#define L_SCALE 2u     // last emitting term of its destination: bring the sum into this cell's frame
#define L_END 4u       // last term of its destination: store the state
#define L_NOTERM 8u    // a destination without incoming transitions

struct LRec { double w; uint32_t src; uint32_t ctl; };      // src: source state * 32 (element offset in a lane-interleaved vector)

// ---------------------------------------------------------------------------------------------
// The windowed program (lane2): the same read-per-lane sweep with the cell's state vector kept ON CHIP.
//
// The first version of this engine kept two whole state vectors per read in global memory; every term of the
// program loaded its source from there, and a profile's delete chain (D_k -> D_k+1 -> ...) became a chain of
// dependent loads at L2 / HBM latency: 180 GCUPS, 2 % of the multiply-add roofline, 10.8 long-scoreboard stall
// cycles per issued instruction (profiles/r01_ncu_summary.md).  What a cell really needs is little:
//   * a silent transition's source is a state computed a few states earlier (dst - src < WN for all but a handful
//     of hub states): the last WN states of the current cell live in a shared-memory WINDOW, win[state % WN][lane];
//   * the few long-range silent edges go through HUBS: a hub SOURCE (the profile's begin state feeding every match
//     state) keeps its value in a pinned shared-memory slot for the whole cell; a hub DESTINATION (the end state
//     fed by every match state) is accumulated in PUSH form -- each source adds its term right after it has been
//     finalised, in ascending source order, which is the reference's candidate order, so the Viterbi tie-break
//     is unchanged;
//   * emitting transitions read the PREVIOUS cell, and only LIVE states (sources of emitting transitions: 975 of
//     PF00516's 2439) ever cross cells: they alone are written to global memory, compactly, and streamed back
//     through a shared-memory RING with cp.async, LA blocks of BS states ahead of their use (sources sit within a
//     few states of their destinations, so the ring is read almost in order).
// Per cell and read the global traffic is the live vector once out and once in; everything else is shared memory
// and registers.  The program is checked when it is built (every window, ring and hub access provably hits the
// value it means to); a machine whose structure does not fit keeps the first version of the sweep.
// ---------------------------------------------------------------------------------------------
enum { K_EMIT = 0, K_WIN = 1, K_HUBS = 2, K_PUSH = 3, K_NONE = 4, K_LOAD = 5, K_CTRL = 6 };
// The stream the kernel executes: single-purpose records { double w; uint32 a; uint32 op }, op & 15 = opcode.  Every
// shared-memory operand is a ROW of the warp's region (window rows, then ring rows, then hub sources, then hub
// destinations), so a term is: one address shift, one load per read, one multiply-add per read.
enum { X_TERM = 0,       // acc = fma (w, region[a], acc)                 (window or hub-source row a; op >> 16 = candidate index)
       X_EMIT = 1,       // acc = fma (emission[w-bits row][token], region[a], acc)  (ring row a); op & 16: then acc *= f
       X_PUSH = 2,       // region[a] = fma (w, vlast, region[a])         (hub-destination row a; (op >> 4) & 7 = its slot)
       X_END = 3,        // region[a] = vlast = res = acc; acc = 0        (window row a); op & 16: live (store to the live vector, track the
                         //                                                range); op & 32: also to hub-source row (w-bits)
       X_HINIT = 4,      // acc = region[a]                               (hub-destination row a; (op >> 4) & 7 = its slot)
       X_PRESTORE = 5,   // region[a] = acc; acc = 0                      (likewise)
       X_LOAD = 6,       // ring row a <- previous live vector, index (w-bits)   (cp.async)
       X_CTRL = 7,       // a: L3_COMMIT | L3_WAIT | L3_ORIGIN
       X_NOP = 8 };
#define L3_NREC 64          // records per chunk
#define L3_EMAX 16          // emission rows per chunk
#define L3_COMMIT 1u        // K_CTRL (in the record's `src` field): close the group of ring loads issued so far
#define L3_WAIT 2u          // K_CTRL: wait until all but the last LA groups have landed (the next block's values are in the ring)
#define L3_ORIGIN 4u        // K_CTRL: the accumulator takes the origin cell's start value
#define L2_SCALE 8u         // last emitting term of its destination: bring the sum into this cell's frame
#define L2_END 16u          // finalise the destination after this record
#define L2_LIVE 32u         // ... and store it to the live vector
#define L2_HSTORE 64u       // ... and to hub-source slot L2_HS (ctl)
#define L2_HINIT 128u       // first record of a hub destination: the accumulator starts from hub slot L2_HD (ctl)
#define L2_PRESTORE 256u    // preamble: the accumulator (a hub destination's emitting terms) goes to hub slot (ctl >> 12) & 7
#define L2_HS(ctl) (((ctl) >> 9) & 7u)       // hub-source slot of an L2_HSTORE record
#define L2_HD(ctl) (((ctl) >> 12) & 7u)      // hub-destination slot of an L2_HINIT / L2_PRESTORE record
#define L2_MAXHUB 8

struct L2Prog {
  bool ok = false;
  std::string why;
  int WN = 32, RN = 64, BS = 8, LA = 3;
  int nHubS = 0, nHubD = 0, nLive = 0, nBlk = 0;      // blocks include block 0 = the preamble
  std::vector<LRec> recLin, recLog;
  std::vector<int64_t> recPerm;             // silent (window / hub / push) record -> hInc entry, -1 otherwise
  std::vector<int32_t> recWant;             // (host only) what the record means to read: live index (emit), source state (window, hub source)
  std::vector<int32_t> blkRec, blkLoad, loadIdx;
  // The program as the kernel reads it: ONE flat stream per cell -- the ring loads of a block (K_LOAD) and the group
  // commit / wait points (K_CTRL) are records like the others -- cut into CHUNKS of at most L3_NREC records that use at
  // most L3_EMAX emission rows; a chunk is one contiguous blob (records | its emission rows, nOut doubles each |
  // their candidate indices) that a CTA fetches with ONE bulk copy (TMA) into shared memory, double buffered, while
  // its warps -- all walking the same program position on different reads -- work through the previous chunk.
  std::vector<LRec> flat;                   // weights filled per blob
  std::vector<int64_t> flatPerm;            // silent record -> hInc entry (-1 otherwise)
  std::vector<int32_t> flatWant, flatRow;   // (host) what a record means to read; table row of an emitting record
  std::vector<int32_t> chunkFirst;          // [nChunks + 1] first flat record of each chunk
  int nChunks = 0, blobBytes = 0, emOff = 0, idxOff = 0;
  std::vector<char> blobLin, blobLog;
  char* dBlobLin = nullptr; char* dBlobLog = nullptr;
};

struct LHost {
  std::vector<LRec> recLin, recLog;       // identical but for the weights
  std::vector<double> emLin, emLog;       // [row][nOut] token-indexed weights of the emitting terms
  std::vector<uint16_t> emIdx;            // [row][nOut] candidate index in the token-selected list (Viterbi back-pointer)
  std::vector<int64_t> recPerm;           // silent record n carries hInc entry recPerm[n] (-1 otherwise)
  std::vector<int64_t> emPerm;            // table entry -> hInc entry (-1: no such transition)
  LRec* dRecLin = nullptr; LRec* dRecLog = nullptr;
  double* dEmLin = nullptr; double* dEmLog = nullptr;
  uint16_t* dEmIdx = nullptr;
  int64_t nRec = 0;
  int S = 0, nOut = 0, bpBytes = 2;
  bool linearOk = false;
  int numSMs = 148;
  // per destination state: its emitting rows (table row, source state) in candidate order -- what lane2_build starts from
  std::vector<std::vector<std::pair<int, int>>> destRows;
  L2Prog l2;
};

struct LParams {
  const LRec* rec; int64_t nRec;
  const double* em; const uint16_t* emIdx;
  int32_t S, nOut, bpBytes;
  DevBatch b;
  const int64_t* order; int64_t nWork;       // reads, longest first; task n = reads [32n, 32n+32)
  unsigned long long* counter;
  double* result; int32_t* flag;
  double* vec;                                // per resident warp: 2 vectors of S * 32 doubles
  unsigned char* bp; const int64_t* bpOff;   // back-pointers of task n at bpOff[n]: [o][state][lane]
};

__device__ __forceinline__ double l_ninf() { return __longlong_as_double (0xfff0000000000000LL); }
__device__ __forceinline__ double l_pow2 (int e) { return e < -1022 ? 0. : __longlong_as_double ((long long) (e > 1023 ? 2046 : e + 1023) << 52); }
__device__ __forceinline__ double l_lse (double a, double b) {      // as w_lse in mb_wide.cu
  const double mx = fmax (a, b), mn = fmin (a, b);
  const float d = (float) (mn - mx);
  if (!(d > -40.f)) return mx;
  return mx + (double) __logf (1.f + __expf (d));
}

// R reads per lane (reads lane, lane+32, ... of the task): R independent multiply-add chains and R
// loads in flight per thread hide the latency of the state vectors, which stream from L2 / HBM, and
// every record of the program is fetched and decoded once for 32*R reads.
template<int OP, int R>
__global__ void __launch_bounds__(128) lane_kernel (const __grid_constant__ LParams p) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nWarps = blockDim.x >> 5;
  const int S = p.S;
  constexpr int LPT = 32 * R;      // reads (vector lanes) per task
  double* v0 = p.vec + ((size_t) blockIdx.x * nWarps + warp) * 2 * (size_t) S * LPT + lane;
  double* v1 = v0 + (size_t) S * LPT;
  const double ZERO = OP == L_SUM ? 0. : l_ninf(), ONE = OP == L_SUM ? 1. : 0.;
  const unsigned kb = p.bpBytes == 1 ? 6 : 14;
  const double LN2 = 0.693147180559945309417232121458;
  for (;;) {
    long long task = 0;
    if (lane == 0) task = (long long) atomicAdd (p.counter, 1ULL);
    task = __shfl_sync (0xffffffffu, task, 0);
    if (task * LPT >= p.nWork) break;
    int64_t k[R];
    const uint8_t* y[R];
    int Lo[R], maxLo = -1;
#pragma unroll
    for (int q = 0; q < R; ++q) {
      const long long rd = task * LPT + q * 32 + lane;
      const bool have = rd < p.nWork;
      k[q] = have ? p.order[rd] : 0;
      y[q] = p.b.y + p.b.yOff[k[q]];
      Lo[q] = have ? (int) (p.b.yOff[k[q] + 1] - p.b.yOff[k[q]]) : -1;
      maxLo = max (maxLo, Lo[q]);
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) maxLo = max (maxLo, __shfl_xor_sync (0xffffffffu, maxLo, off));
    unsigned char* bp = OP == L_MAX && p.bp ? p.bp + p.bpOff[task] + (size_t) lane * p.bpBytes : nullptr;
    bool bad[R];
    int Fprev[R], Gprev[R];
#pragma unroll
    for (int q = 0; q < R; ++q) { bad[q] = false; Fprev[q] = 0; Gprev[q] = L_SENT; }
    for (int o = 0; o <= maxLo; ++o) {
      double* cur = (o & 1) ? v1 : v0;
      const double* prev = (o & 1) ? v0 : v1;
      int tok[R], F[R], mx[R];
      unsigned mn[R], best[R];
      double f[R], acc[R], res[R];
#pragma unroll
      for (int q = 0; q < R; ++q) {
        tok[q] = (o <= Lo[q] && o > 0) ? y[q][o - 1] - 1 : 0;
        F[q] = 0; f[q] = 1.;
        if (OP == L_SUM && o > 0) { if (Gprev[q] == L_SENT) f[q] = 0.; else { F[q] = Gprev[q]; f[q] = l_pow2 (Fprev[q] - F[q]); } }
        mx[q] = 0; mn[q] = 0xffffffffu; best[q] = 0xffffu;
        acc[q] = o == 0 ? ONE : ZERO;      // the origin cell's start state (forward.defs.h:36)
        res[q] = ZERO;
      }
      const bool usePrev = o > 0;
      double* out = cur;
      unsigned char* bpRow = bp ? bp + (size_t) o * S * LPT * p.bpBytes : nullptr;
      const LRec* r = p.rec;
      uint4 nx = __ldg (reinterpret_cast<const uint4*> (r));
      for (int64_t n = 0; n < p.nRec; ++n) {
        const uint4 u = nx;
        nx = __ldg (reinterpret_cast<const uint4*> (r + n + 1));      // the stream ends with a spare record
        const unsigned ctl = u.w;
        if (!(ctl & L_NOTERM)) {
          if (ctl & L_EMIT) {
            if (usePrev) {
              double x[R], w[R];
              unsigned ix[R];
#pragma unroll
              for (int q = 0; q < R; ++q) {
                x[q] = prev[(size_t) u.z * R + q * 32];
                w[q] = __ldg (p.em + (size_t) u.x * p.nOut + tok[q]);
                if (OP == L_MAX) ix[q] = __ldg (p.emIdx + (size_t) u.x * p.nOut + tok[q]);
              }
#pragma unroll
              for (int q = 0; q < R; ++q) {
                if (OP == L_SUM) acc[q] = fma (w[q], x[q], acc[q]);
                else if (OP == L_LSE) acc[q] = l_lse (acc[q], x[q] + w[q]);
                else { const double c = x[q] + w[q]; if (acc[q] < c) { acc[q] = c; best[q] = ((unsigned) T_INSERT << kb) | ix[q]; } }
              }
            }
            if (OP == L_SUM && (ctl & L_SCALE)) {
#pragma unroll
              for (int q = 0; q < R; ++q) acc[q] *= f[q];
            }
          } else {
            const double w = __hiloint2double ((int) u.y, (int) u.x);
            double x[R];
#pragma unroll
            for (int q = 0; q < R; ++q) x[q] = cur[(size_t) u.z * R + q * 32];
#pragma unroll
            for (int q = 0; q < R; ++q) {
              if (OP == L_SUM) acc[q] = fma (w, x[q], acc[q]);
              else if (OP == L_LSE) acc[q] = l_lse (acc[q], x[q] + w);
              else { const double c = x[q] + w; if (acc[q] < c) { acc[q] = c; best[q] = ((unsigned) T_SILENT << kb) | (ctl >> 16); } }
            }
          }
        }
        if (ctl & L_END) {
#pragma unroll
          for (int q = 0; q < R; ++q) {
            out[q * 32] = acc[q];
            if (OP == L_SUM) {
              const int hi = __double2hiint (acc[q]);
              mx[q] = max (mx[q], hi);
              mn[q] = min (mn[q], (unsigned) (hi - 0x00100000));      // zeros and denormals wrap to the top and drop out
            } else if (OP == L_MAX && bpRow) {
              if (p.bpBytes == 1) bpRow[q * 32] = (unsigned char) best[q]; else reinterpret_cast<uint16_t*> (bpRow)[q * 32] = (uint16_t) best[q];
            }
            res[q] = acc[q];      // after the last record: the end state
            acc[q] = ZERO;
            best[q] = 0xffffu;
          }
          out += LPT;
          if (OP == L_MAX && bpRow) bpRow += LPT * p.bpBytes;
        }
      }
#pragma unroll
      for (int q = 0; q < R; ++q) {
        if (OP == L_SUM) {
          int Gc = L_SENT;
          if (mx[q] >= 0x00100000) {
            const int emx = mx[q] >> 20;
            Gc = F[q] + emx - 1023;
            if (o <= Lo[q] && (emx == 0x7ff || (mn[q] != 0xffffffffu && emx - (int) ((mn[q] >> 20) + 1) > L_SPREAD))) bad[q] = true;
          }
          Fprev[q] = F[q]; Gprev[q] = Gc;
        }
        if (o == Lo[q]) {
          if (OP == L_SUM) { p.result[k[q]] = res[q] > 0. ? log (res[q]) + F[q] * LN2 : l_ninf(); p.flag[k[q]] = bad[q] || !(res[q] > 0.) || !(res[q] < 1e300); }
          else p.result[k[q]] = res[q];
        }
      }
      __syncwarp();
    }
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static LHost* lh (const mb_machine* m) { return static_cast<LHost*> (m->lane); }
static void lane2_build (const mb_machine* m, LHost* h);
static void lane2_fill_weights (const mb_machine* m, LHost* h);
static int lane2_upload (mb_machine* m, LHost* h, bool all);

static void lane_fill_weights (const mb_machine* m, LHost* h) {
  bool ok = true;
  const double lim = 30. * 0.6931471805599453;
  auto check = [&] (double lw) { if (std::isnan (lw) || (std::isfinite (lw) && fabs (lw) > lim) || lw == INFINITY) ok = false; };
  for (size_t n = 0; n < h->recPerm.size(); ++n) {
    if (h->recPerm[n] < 0) continue;
    const double lw = m->hInc.lw[h->recPerm[n]];
    h->recLog[n].w = lw;
    h->recLin[n].w = exp (lw);
    check (lw);
  }
  for (size_t n = 0; n < h->emPerm.size(); ++n) {
    if (h->emPerm[n] < 0) { h->emLin[n] = 0.; h->emLog[n] = -INFINITY; continue; }
    const double lw = m->hInc.lw[h->emPerm[n]];
    h->emLog[n] = lw;
    h->emLin[n] = exp (lw);
    check (lw);
  }
  h->linearOk = ok;
}

void lane_destroy (mb_machine* m) {
  LHost* h = lh (m);
  if (!h) return;
  for (void* p: { (void*) h->dRecLin, (void*) h->dRecLog, (void*) h->dEmLin, (void*) h->dEmLog, (void*) h->dEmIdx, (void*) h->l2.dBlobLin, (void*) h->l2.dBlobLog }) if (p) cudaFree (p);
  delete h;
  m->lane = nullptr;
}

static int lane_upload (mb_machine* m, LHost* h, bool all) {
  MB_CUDA (cudaSetDevice (m->device));
  const size_t rb = h->recLin.size() * sizeof (LRec), eb = std::max<size_t> (h->emLin.size(), 1) * 8;
  if (all) {
    MB_CUDA (cudaMalloc (&h->dRecLin, rb)); MB_CUDA (cudaMalloc (&h->dRecLog, rb));
    MB_CUDA (cudaMalloc (&h->dEmLin, eb)); MB_CUDA (cudaMalloc (&h->dEmLog, eb));
    MB_CUDA (cudaMalloc (&h->dEmIdx, std::max<size_t> (h->emIdx.size(), 1) * 2));
    if (!h->emIdx.empty()) MB_CUDA (cudaMemcpy (h->dEmIdx, h->emIdx.data(), h->emIdx.size() * 2, cudaMemcpyHostToDevice));
  }
  MB_CUDA (cudaMemcpy (h->dRecLin, h->recLin.data(), rb, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (h->dRecLog, h->recLog.data(), rb, cudaMemcpyHostToDevice));
  if (!h->emLin.empty()) {
    MB_CUDA (cudaMemcpy (h->dEmLin, h->emLin.data(), h->emLin.size() * 8, cudaMemcpyHostToDevice));
    MB_CUDA (cudaMemcpy (h->dEmLog, h->emLog.data(), h->emLog.size() * 8, cudaMemcpyHostToDevice));
  }
  return 0;
}

int lane_update_weights (mb_machine* m) {
  LHost* h = lh (m);
  if (!h) return 0;
  lane_fill_weights (m, h);
  if (h->l2.ok) lane2_fill_weights (m, h);
  return lane_upload (m, h, false) || lane2_upload (m, h, false);
}

// The transition program: destinations in index order; per destination the emitting terms (union
// over output tokens of the token-selected insert lists, in list order), then the silent terms.
int lane_prepare (mb_machine* m) {
  LHost* h = new LHost;
  m->lane = h;
  const int S = m->S, nOut = m->nOut, nIn1 = m->nIn + 1, nOut1 = nOut + 1;
  const HostCsr& inc = m->hInc;
  h->S = S; h->nOut = nOut;
  int maxList = 0;
  LRec blank; blank.w = 0; blank.src = 0; blank.ctl = 0;
  for (int d = 0; d < S; ++d) {
    const size_t first = h->recLin.size();
    // union of the insert lists of d over the output tokens: key (source, rank among equals) keeps each list's order
    std::map<std::pair<int, int>, int> rowOf;      // -> table row
    std::vector<std::pair<int, int>> keys;
    for (int c = 1; c <= nOut; ++c) {
      const int64_t key = ((int64_t) d * nIn1) * nOut1 + c;
      maxList = std::max<int> (maxList, (int) (inc.off[key + 1] - inc.off[key]));
      std::map<int, int> seen;
      for (int64_t q = inc.off[key]; q < inc.off[key + 1]; ++q) {
        const std::pair<int, int> kk (inc.other[q], seen[inc.other[q]]++);
        if (!rowOf.count (kk)) { rowOf[kk] = -1; keys.push_back (kk); }
      }
    }
    std::sort (keys.begin(), keys.end());
    h->destRows.resize ((size_t) S);
    for (auto& kk: keys) {
      const int row = (int) (h->emPerm.size() / std::max (nOut, 1));
      rowOf[kk] = row;
      h->destRows[d].push_back (std::make_pair (row, kk.first));
      h->emPerm.resize (h->emPerm.size() + nOut, -1);
      h->emIdx.resize (h->emIdx.size() + nOut, 0x3fff);
      LRec r = blank;
      const uint64_t rowBits = (uint64_t) row;
      memcpy (&r.w, &rowBits, 8);
      r.src = (uint32_t) kk.first * 32u;
      r.ctl = L_EMIT;
      h->recLin.push_back (r);
      h->recPerm.push_back (-1);
    }
    for (int c = 1; c <= nOut; ++c) {
      const int64_t key = ((int64_t) d * nIn1) * nOut1 + c;
      std::map<int, int> seen;
      for (int64_t q = inc.off[key]; q < inc.off[key + 1]; ++q) {
        const int row = rowOf[std::make_pair (inc.other[q], seen[inc.other[q]]++)];
        h->emPerm[(size_t) row * nOut + (c - 1)] = q;
        h->emIdx[(size_t) row * nOut + (c - 1)] = (uint16_t) (q - inc.off[key]);
      }
    }
    if (!keys.empty()) h->recLin.back().ctl |= L_SCALE;
    if (d > 0) {      // state 0's only possible silent source is its own self-loop, which contributes nothing (machine.cpp:759)
      const int64_t key = (int64_t) d * nIn1 * nOut1;
      maxList = std::max<int> (maxList, (int) (inc.off[key + 1] - inc.off[key]));
      for (int64_t q = inc.off[key]; q < inc.off[key + 1]; ++q) {
        LRec r = blank;
        r.src = (uint32_t) inc.other[q] * 32u;
        r.ctl = (uint32_t) (q - inc.off[key]) << 16;
        h->recLin.push_back (r);
        h->recPerm.push_back (q);
      }
    }
    if (h->recLin.size() == first) { LRec r = blank; r.ctl = L_NOTERM; h->recLin.push_back (r); h->recPerm.push_back (-1); }
    h->recLin.back().ctl |= L_END;
  }
  if (maxList > 16382) { set_error ("lane engine: a transition list has more than 16382 entries"); return 1; }
  h->bpBytes = maxList <= 63 ? 1 : 2;
  h->nRec = (int64_t) h->recLin.size();
  { LRec r = blank; r.ctl = L_NOTERM; h->recLin.push_back (r); h->recPerm.push_back (-1); }      // spare record: the sweep keeps one in flight
  h->recLog = h->recLin;
  h->emLin.assign (h->emPerm.size(), 0.);
  h->emLog.assign (h->emPerm.size(), -INFINITY);
  lane_fill_weights (m, h);
  lane2_build (m, h);
  if (h->l2.ok) lane2_fill_weights (m, h);
  if (m->opt.get ("lane_host_only", 0)) return 0;      // (diagnostic: build the programs without touching a device)
  if (lane_upload (m, h, true) || lane2_upload (m, h, true)) return 1;
  MB_CUDA (cudaDeviceGetAttribute (&h->numSMs, cudaDevAttrMultiProcessorCount, m->device));
  if (m->opt.get ("verbose", 0))
    fprintf (stderr, "lane engine: S=%d records=%lld (emitting rows %zu x %d tokens), bp %d bytes\n", S, (long long) h->nRec, h->emPerm.size() / std::max (nOut, 1), nOut, h->bpBytes);
  return 0;
}

// ---------------------------------------------------------------------------------------------
// lane2: building the windowed program
// ---------------------------------------------------------------------------------------------
static LRec l2_rec (uint32_t kind, uint32_t a, uint32_t flags) { LRec r; r.w = 0; r.src = a; r.ctl = kind | flags; return r; }

static bool lane2_try (const mb_machine* m, LHost* h, int WN, int RN, int BS, int LA) {
  L2Prog& P = h->l2;
  const int S = m->S, nIn1 = m->nIn + 1, nOut1 = m->nOut + 1;
  const HostCsr& inc = m->hInc;
  auto fail = [&] (const std::string& w) { P.ok = false; P.why = w; return false; };
  P = L2Prog();
  P.WN = WN; P.RN = RN; P.BS = BS; P.LA = LA;
  // ---- long-range silent edges and the hubs that carry them
  struct Edge { int src, dst; };
  std::vector<Edge> far;
  for (int d = 1; d < S; ++d) {
    const int64_t key = (int64_t) d * nIn1 * nOut1;
    for (int64_t q = inc.off[key]; q < inc.off[key + 1]; ++q) if (d - inc.other[q] >= WN) far.push_back (Edge { inc.other[q], d });
  }
  std::vector<int> hubS ((size_t) S, -1), hubD ((size_t) S, -1);
  for (;;) {      // greedy cover: the state with most uncovered long-range edges becomes a hub
    std::vector<int> nOut ((size_t) S, 0), nIn ((size_t) S, 0);
    int left = 0;
    for (auto& e: far) if (hubS[e.src] < 0 && hubD[e.dst] < 0) { ++nOut[e.src]; ++nIn[e.dst]; ++left; }
    if (!left) break;
    int bestS = 0, bestD = 0;
    for (int s = 0; s < S; ++s) { if (nOut[s] > nOut[bestS]) bestS = s; if (nIn[s] > nIn[bestD]) bestD = s; }
    if (nOut[bestS] >= nIn[bestD]) { if (P.nHubS == L2_MAXHUB) return fail ("more than 8 hub sources"); hubS[bestS] = P.nHubS++; }
    else { if (P.nHubD == L2_MAXHUB) return fail ("more than 8 hub destinations"); hubD[bestD] = P.nHubD++; }
  }
  // ---- live states: sources of emitting rows
  std::vector<int> liveIdx ((size_t) S, -1);
  { std::vector<char> isLive ((size_t) S, 0);
    for (int d = 0; d < S; ++d) for (auto& rs: h->destRows[d]) isLive[rs.second] = 1;
    for (int s = 0; s < S; ++s) if (isLive[s]) liveIdx[s] = P.nLive++; }
  // ---- pushes: every silent term of a hub destination, attached to its source, in the destination's list order
  struct Push { int hd; int64_t q; uint32_t cand; };
  std::vector<std::vector<Push>> pushOf ((size_t) S);
  for (int d = 1; d < S; ++d) {
    if (hubD[d] < 0) continue;
    const int64_t key = (int64_t) d * nIn1 * nOut1;
    for (int64_t q = inc.off[key]; q < inc.off[key + 1]; ++q) pushOf[inc.other[q]].push_back (Push { hubD[d], q, (uint32_t) (q - inc.off[key]) });
  }
  // ---- records, block by block
  std::vector<std::vector<int>> blkLive;      // live indices each block's emitting terms read, in order of use
  auto emit_terms = [&] (int d, std::vector<int>& liveUse) {
    const auto& rows = h->destRows[d];
    for (size_t n = 0; n < rows.size(); ++n) {
      LRec r = l2_rec (K_EMIT, (uint32_t) (liveIdx[rows[n].second] & (RN - 1)), n + 1 == rows.size() ? L2_SCALE : 0u);
      const uint64_t rowBits = (uint64_t) rows[n].first;
      memcpy (&r.w, &rowBits, 8);
      P.recLin.push_back (r);
      P.recPerm.push_back (-1);
      P.recWant.push_back (liveIdx[rows[n].second]);
      liveUse.push_back (liveIdx[rows[n].second]);
    }
  };
  P.blkRec.push_back (0);
  blkLive.emplace_back();
  for (int d = 0; d < S; ++d) {      // block 0, the preamble: emitting terms of hub destinations go to their hub slot first
    if (hubD[d] < 0 || h->destRows[d].empty()) continue;
    emit_terms (d, blkLive.back());
    P.recLin.push_back (l2_rec (K_NONE, 0, L2_PRESTORE | ((uint32_t) hubD[d] << 12)));
    P.recPerm.push_back (-1);
    P.recWant.push_back (-1);
  }
  P.blkRec.push_back ((int32_t) P.recLin.size());
  for (int d0 = 0; d0 < S; d0 += BS) {
    blkLive.emplace_back();
    for (int d = d0; d < std::min (S, d0 + BS); ++d) {
      const size_t first = P.recLin.size();
      if (hubD[d] >= 0) { P.recLin.push_back (l2_rec (K_NONE, 0, L2_HINIT | ((uint32_t) hubD[d] << 12))); P.recPerm.push_back (-1); P.recWant.push_back (-1); }
      else {
        emit_terms (d, blkLive.back());
        if (d > 0) {
          const int64_t key = (int64_t) d * nIn1 * nOut1;
          for (int64_t q = inc.off[key]; q < inc.off[key + 1]; ++q) {
            const int src = inc.other[q];
            const uint32_t cand = (uint32_t) (q - inc.off[key]) << 16;
            if (hubS[src] >= 0) P.recLin.push_back (l2_rec (K_HUBS, (uint32_t) hubS[src], cand));
            else if (d - src < WN) P.recLin.push_back (l2_rec (K_WIN, (uint32_t) (src & (WN - 1)), cand));
            else return fail ("a long-range silent edge is not covered by a hub");
            P.recPerm.push_back (q);
            P.recWant.push_back (src);
          }
        }
        if (P.recLin.size() == first) { P.recLin.push_back (l2_rec (K_NONE, 0, 0)); P.recPerm.push_back (-1); P.recWant.push_back (-1); }
      }
      P.recLin.back().ctl |= L2_END | (liveIdx[d] >= 0 ? L2_LIVE : 0u) | (hubS[d] >= 0 ? (L2_HSTORE | ((uint32_t) hubS[d] << 9)) : 0u);
      for (auto& pu: pushOf[d]) { P.recLin.push_back (l2_rec (K_PUSH, (uint32_t) pu.hd, pu.cand << 16)); P.recPerm.push_back (pu.q); P.recWant.push_back (-1); }
    }
    P.blkRec.push_back ((int32_t) P.recLin.size());
  }
  P.nBlk = (int) P.blkRec.size() - 1;
  LA = std::min (LA, P.nBlk);      // (a program of fewer blocks than the lookahead: everything is requested up front)
  P.LA = LA;
  // ---- ring schedule: block b's loads are issued LA blocks early; a slot may only be refilled once every block that
  // still reads its old content has been processed
  std::vector<int> lastUse ((size_t) std::max (P.nLive, 1), -1), tag ((size_t) RN, -1);
  for (int b = 0; b < P.nBlk; ++b) for (int j: blkLive[b]) lastUse[j] = b;
  P.blkLoad.push_back (0);
  for (int b = 0; b < P.nBlk; ++b) {
    for (int j: blkLive[b]) {
      const int slot = j & (RN - 1);
      if (tag[slot] == j) continue;
      // the load is issued while block b - LA is being processed (blocks before that are done)
      if (tag[slot] >= 0 && lastUse[tag[slot]] >= b - LA) return fail ("the ring of previous-cell values is too small for this machine");
      tag[slot] = j;
      P.loadIdx.push_back (j);
    }
    P.blkLoad.push_back ((int32_t) P.loadIdx.size());
  }
  { LRec r = l2_rec (K_NONE, 0, 0); P.recLin.push_back (r); P.recPerm.push_back (-1); P.recWant.push_back (-1); }      // spare record: the sweep keeps one in flight
  P.recLog = P.recLin;
  P.ok = true;
  return true;
}

// the flat stream: single-purpose records; per block its ring loads travel LA blocks ahead of the block itself
static void lane2_flatten (LHost* h) {
  L2Prog& P = h->l2;
  const uint32_t rowWin = 0, rowRing = (uint32_t) P.WN, rowHubS = rowRing + (uint32_t) P.RN, rowHubD = rowHubS + (uint32_t) P.nHubS;
  auto put = [&] (uint32_t opcode, uint32_t a, uint32_t aux, uint64_t wbits, int64_t perm, int32_t want, int32_t row) {
    LRec r; r.src = a; r.ctl = opcode | aux;
    memcpy (&r.w, &wbits, 8);
    P.flat.push_back (r); P.flatPerm.push_back (perm); P.flatWant.push_back (want); P.flatRow.push_back (row);
  };
  auto loads = [&] (int blk) {
    if (blk < P.nBlk)
      for (int j = P.blkLoad[blk]; j < P.blkLoad[blk + 1]; ++j)
        put (X_LOAD, rowRing + (uint32_t) (P.loadIdx[j] & (P.RN - 1)), 0, (uint64_t) P.loadIdx[j], -1, P.loadIdx[j], -1);
    put (X_CTRL, L3_COMMIT, 0, 0, -1, -1, -1);      // (an empty group keeps the count uniform)
  };
  int d = 0;      // destination state of the next END
  for (int blk = 0; blk < std::min (P.LA, P.nBlk); ++blk) loads (blk);
  for (int blk = 0; blk < P.nBlk; ++blk) {
    if (blk + P.LA < P.nBlk) loads (blk + P.LA); else put (X_CTRL, L3_COMMIT, 0, 0, -1, -1, -1);
    put (X_CTRL, L3_WAIT | (blk == 1 ? L3_ORIGIN : 0u), 0, 0, -1, -1, -1);
    for (int n = P.blkRec[blk]; n < P.blkRec[blk + 1]; ++n) {
      const LRec& r = P.recLin[n];
      const uint32_t ctl = r.ctl, kind = ctl & 7u, cand = ctl & 0xffff0000u;
      if (ctl & L2_HINIT) put (X_HINIT, rowHubD + L2_HD (ctl), L2_HD (ctl) << 4, 0, -1, -1, -1);
      if (kind == K_EMIT) {
        uint64_t row; memcpy (&row, &r.w, 8);
        put (X_EMIT, rowRing + r.src, (ctl & L2_SCALE) ? 16u : 0u, 0, -1, P.recWant[n], (int32_t) row);
      } else if (kind == K_WIN) put (X_TERM, rowWin + r.src, cand, 0, P.recPerm[n], P.recWant[n], -1);
      else if (kind == K_HUBS) put (X_TERM, rowHubS + r.src, cand, 0, P.recPerm[n], P.recWant[n], -1);
      else if (kind == K_PUSH) put (X_PUSH, rowHubD + r.src, cand | (r.src << 4), 0, P.recPerm[n], -1, -1);
      if (ctl & L2_PRESTORE) put (X_PRESTORE, rowHubD + L2_HD (ctl), L2_HD (ctl) << 4, 0, -1, -1, -1);
      if (ctl & L2_END) {
        put (X_END, rowWin + (uint32_t) (d & (P.WN - 1)), ((ctl & L2_LIVE) ? 16u : 0u) | ((ctl & L2_HSTORE) ? 32u : 0u), (uint64_t) (rowHubS + L2_HS (ctl)), -1, d, -1);
        ++d;
      }
    }
  }
  // chunks
  P.chunkFirst.assign (1, 0);
  int nRec = 0, nEm = 0;
  for (size_t n = 0; n < P.flat.size(); ++n) {
    const bool isEmit = (P.flat[n].ctl & 15u) == X_EMIT;
    if (nRec == L3_NREC || (isEmit && nEm == L3_EMAX)) { P.chunkFirst.push_back ((int32_t) n); nRec = 0; nEm = 0; }
    ++nRec;
    if (isEmit) ++nEm;
  }
  P.chunkFirst.push_back ((int32_t) P.flat.size());
  P.nChunks = (int) P.chunkFirst.size() - 1;
  P.emOff = (L3_NREC + 1) * (int) sizeof (LRec);      // (one spare record: the sweep reads one ahead)
  P.idxOff = P.emOff + L3_EMAX * std::max (h->nOut, 1) * 8;
  P.blobBytes = (P.idxOff + L3_EMAX * std::max (h->nOut, 1) * 2 + 15) & ~15;
}

// blobs for the current weights: the records (silent weights inside), each chunk's emission rows and candidate indices
static void lane2_fill_weights (const mb_machine* m, LHost* h) {
  L2Prog& P = h->l2;
  const int nOut = std::max (h->nOut, 1);
  P.blobLin.assign ((size_t) P.nChunks * P.blobBytes, 0);
  P.blobLog = P.blobLin;
  LRec nop; nop.w = 0; nop.src = 0; nop.ctl = X_NOP;
  for (int c = 0; c < P.nChunks; ++c) {
    char* bl = P.blobLin.data() + (size_t) c * P.blobBytes;
    char* bg = P.blobLog.data() + (size_t) c * P.blobBytes;
    int nEm = 0;
    for (int n = P.chunkFirst[c]; n < P.chunkFirst[c + 1]; ++n) {
      LRec rl = P.flat[n], rg = P.flat[n];
      if ((rl.ctl & 15u) == X_EMIT) {
        const uint64_t local = (uint64_t) nEm;      // the row's place in this chunk's emission area
        memcpy (&rl.w, &local, 8); memcpy (&rg.w, &local, 8);
        for (int t = 0; t < h->nOut; ++t) {
          ((double*) (bl + P.emOff))[nEm * nOut + t] = h->emLin[(size_t) P.flatRow[n] * h->nOut + t];
          ((double*) (bg + P.emOff))[nEm * nOut + t] = h->emLog[(size_t) P.flatRow[n] * h->nOut + t];
          ((uint16_t*) (bl + P.idxOff))[nEm * nOut + t] = ((uint16_t*) (bg + P.idxOff))[nEm * nOut + t] = h->emIdx[(size_t) P.flatRow[n] * h->nOut + t];
        }
        ++nEm;
      } else if (P.flatPerm[n] >= 0) {
        const double lw = m->hInc.lw[P.flatPerm[n]];
        rg.w = lw;
        rl.w = exp (lw);
      }
      memcpy (bl + (size_t) (n - P.chunkFirst[c]) * sizeof (LRec), &rl, sizeof (LRec));
      memcpy (bg + (size_t) (n - P.chunkFirst[c]) * sizeof (LRec), &rg, sizeof (LRec));
    }
    for (int n = P.chunkFirst[c + 1] - P.chunkFirst[c]; n <= L3_NREC; ++n) {      // the rest of the record area, spare record included
      memcpy (bl + (size_t) n * sizeof (LRec), &nop, sizeof (LRec));
      memcpy (bg + (size_t) n * sizeof (LRec), &nop, sizeof (LRec));
    }
  }
}

static int lane2_upload (mb_machine* m, LHost* h, bool all) {
  L2Prog& P = h->l2;
  if (!P.ok) return 0;
  if (all) { MB_CUDA (cudaMalloc (&P.dBlobLin, P.blobLin.size())); MB_CUDA (cudaMalloc (&P.dBlobLog, P.blobLog.size())); }
  MB_CUDA (cudaMemcpy (P.dBlobLin, P.blobLin.data(), P.blobLin.size(), cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (P.dBlobLog, P.blobLog.data(), P.blobLog.size(), cudaMemcpyHostToDevice));
  return 0;
}

int lane2_info (const mb_machine* m, int32_t* info) {
  LHost* h = lh (m);
  if (!h) { set_error ("lane engine not prepared"); return 1; }
  const L2Prog& P = h->l2;
  const int32_t v[8] = { P.ok ? 1 : 0, P.WN, P.RN, P.nHubS, P.nHubD, P.nLive, (int32_t) P.flat.size(), h->bpBytes };
  for (int q = 0; q < 8; ++q) info[q] = v[q];
  if (!P.ok) set_error ("lane2: " + P.why);
  return 0;
}

static void lane2_build (const mb_machine* m, LHost* h) {
  if (m->opt.get ("lane_old", 0)) { h->l2.ok = false; h->l2.why = "disabled (option lane_old)"; return; }
  const int BS = std::max (1, std::min (64, m->opt.get ("lane_bs", 8))), LA = std::max (1, std::min (8, m->opt.get ("lane_la", 3)));
  for (int WN: { 32, 64, 128 }) {
    if (m->opt.has ("lane_wn") && WN != m->opt.get ("lane_wn", 32)) continue;
    for (int RN: { 16, 32, 64, 128 }) if (lane2_try (m, h, WN, RN, BS, LA)) { lane2_flatten (h); return; }
  }
}

// The program executed for ONE read on the host, chunk by chunk and row by row as the kernel does it (the same blobs,
// the same region rows, every row tagged with what it holds so that a stale read is an error): what the CPU test checks
// against known answers.  op: L_SUM (scaled linear domain, frame per cell), L_MAX, L_LSE.  Returns 0, or 1 with the error set.
int lane2_emulate (const mb_machine* m, const uint8_t* y, int64_t Lo, int op, double* result, std::vector<uint32_t>* bpOut) {
  LHost* h = lh (m);
  if (!h || !h->l2.ok) { set_error (std::string ("lane2: no windowed program for this machine") + (h ? ": " + h->l2.why : std::string())); return 1; }
  const L2Prog& P = h->l2;
  const std::vector<char>& blob = op == L_SUM ? P.blobLin : P.blobLog;
  const int nOut = std::max (h->nOut, 1), S = h->S;
  const double ZERO = op == L_SUM ? 0. : -INFINITY, ONE = op == L_SUM ? 1. : 0.;
  const unsigned kb = h->bpBytes == 1 ? 6 : 14;
  auto lse = [] (double a, double b) { const double mx = std::max (a, b), mn = std::min (a, b); return mn == -INFINITY ? mx : mx + log1p (exp (mn - mx)); };
  const int rows = P.WN + P.RN + P.nHubS + P.nHubD, rowHubD = P.WN + P.RN + P.nHubS;
  std::vector<double> region ((size_t) rows, ZERO), live[2];
  std::vector<int> tag ((size_t) rows, -1);
  std::vector<uint32_t> hubDB (L2_MAXHUB);
  live[0].assign ((size_t) std::max (P.nLive, 1), ZERO); live[1] = live[0];
  int Fprev = 0, Gprev = L_SENT;
  double res = ZERO;
  int Fres = 0;
  if (bpOut) bpOut->assign ((size_t) (Lo + 1) * S, 0xffffu);
  for (int64_t o = 0; o <= Lo; ++o) {
    std::vector<double>& cur = live[o & 1];
    const std::vector<double>& prev = live[(o & 1) ^ 1];
    const int tok = o > 0 ? y[o - 1] - 1 : 0;
    int F = 0; double f = 1.;
    if (op == L_SUM && o > 0) { if (Gprev == L_SENT) f = 0.; else { F = Gprev; f = std::ldexp (1., Fprev - F); } }
    std::fill (tag.begin(), tag.end(), -1);      // a new cell: nothing of it is in the window, nothing of the previous vector in the ring
    for (int hd = 0; hd < P.nHubD; ++hd) { region[rowHubD + hd] = ZERO; hubDB[hd] = 0xffffu; }
    double acc = ZERO, vlast = ZERO;
    uint32_t best = 0xffffu;
    int mx = 0; unsigned mn = 0xffffffffu;
    int d = 0, nl = 0;
    // ring loads land when their group is waited for: pending[g] = (row, live index) of group g; a WAIT completes all but the last LA groups
    std::vector<std::vector<std::pair<int, int>>> pending (1);
    size_t landed = 0;
    for (int c = 0; c < P.nChunks; ++c) {
      const char* bl = blob.data() + (size_t) c * P.blobBytes;
      const double* em = (const double*) (bl + P.emOff);
      const uint16_t* emIdx = (const uint16_t*) (bl + P.idxOff);
      for (int q = 0; q < L3_NREC; ++q) {
        LRec r;
        memcpy (&r, bl + (size_t) q * sizeof (LRec), sizeof (LRec));
        const int n = P.chunkFirst[c] + q;      // (flat index, for the tags; records past the chunk's end are X_NOP)
        const uint32_t opc = r.ctl & 15u;
        uint64_t wbits; memcpy (&wbits, &r.w, 8);
        if ((int) r.src >= rows && opc != X_CTRL && opc != X_NOP) { set_error ("lane2 emulation: a row outside the warp's region"); return 1; }
        switch (opc) {
          case X_LOAD: if (o > 0) pending.back().push_back (std::make_pair ((int) r.src, (int) wbits)); break;
          case X_CTRL:
            if (r.src & L3_COMMIT) pending.emplace_back();
            if (r.src & L3_WAIT) {
              const size_t done = pending.size() - 1 > (size_t) P.LA ? pending.size() - 1 - (size_t) P.LA : 0;
              for (; landed < done; ++landed) for (auto& ld: pending[landed]) { region[ld.first] = prev[ld.second]; tag[ld.first] = ld.second; }
            }
            if (r.src & L3_ORIGIN) acc = o == 0 ? ONE : ZERO;      // the origin cell's start state (forward.defs.h:36), after the preamble
            break;
          case X_HINIT: acc = region[r.src]; best = hubDB[(r.ctl >> 4) & 7u]; break;
          case X_EMIT:
            if (o > 0) {
              if (wbits >= L3_EMAX) { set_error ("lane2 emulation: an emission row outside the chunk's area"); return 1; }
              if (tag[r.src] != P.flatWant[n]) { set_error ("lane2 emulation: a ring row does not hold the previous-cell value the term means to read"); return 1; }
              const double x = region[r.src], w = em[(size_t) wbits * nOut + tok];
              if (op == L_SUM) acc = fma (w, x, acc);
              else if (op == L_LSE) acc = lse (acc, x + w);
              else { const double cnd = x + w; if (acc < cnd) { acc = cnd; best = ((uint32_t) T_INSERT << kb) | emIdx[(size_t) wbits * nOut + tok]; } }
            }
            if (op == L_SUM && (r.ctl & 16u)) acc *= f;
            break;
          case X_TERM: {
            if (tag[r.src] != P.flatWant[n]) { set_error ("lane2 emulation: a window or hub row does not hold the state the term means to read"); return 1; }
            const double x = region[r.src];
            if (op == L_SUM) acc = fma (r.w, x, acc);
            else if (op == L_LSE) acc = lse (acc, x + r.w);
            else { const double cnd = x + r.w; if (acc < cnd) { acc = cnd; best = ((uint32_t) T_SILENT << kb) | (r.ctl >> 16); } }
            break;
          }
          case X_PUSH: {
            double& a = region[r.src];
            if (op == L_SUM) a = fma (r.w, vlast, a);
            else if (op == L_LSE) a = lse (a, vlast + r.w);
            else { const double cnd = vlast + r.w; if (a < cnd) { a = cnd; hubDB[(r.ctl >> 4) & 7u] = ((uint32_t) T_SILENT << kb) | (r.ctl >> 16); } }
            break;
          }
          case X_PRESTORE: region[r.src] = acc; hubDB[(r.ctl >> 4) & 7u] = best; acc = ZERO; best = 0xffffu; break;
          case X_END:
            region[r.src] = acc; tag[r.src] = d;
            vlast = acc;
            if (r.ctl & 32u) { region[wbits] = acc; tag[wbits] = d; }
            if (r.ctl & 16u) {
              cur[nl++] = acc;
              if (op == L_SUM) {      // only live values cross cells: they set the next frame
                int64_t bits; memcpy (&bits, &acc, 8);
                const int hi = (int) (bits >> 32);
                mx = std::max (mx, hi); mn = std::min (mn, (unsigned) (hi - 0x00100000));
              }
            }
            if (op == L_MAX && bpOut) (*bpOut)[(size_t) o * S + d] = best;
            res = acc; Fres = F;
            acc = ZERO; best = 0xffffu;
            ++d;
            break;
          default: break;
        }
      }
    }
    if (d != S || nl != P.nLive) { set_error ("lane2 emulation: the program does not visit every state"); return 1; }
    if (op == L_SUM) {
      int Gc = L_SENT;
      if (mx >= 0x00100000) Gc = F + (mx >> 20) - 1023;
      Fprev = F; Gprev = Gc;
    }
  }
  *result = op == L_SUM ? (res > 0. ? log (res) + Fres * 0.693147180559945309417232121458 : -INFINITY) : res;
  return 0;
}

// ---------------------------------------------------------------------------------------------
// lane2: the kernel.  A CTA of W warps = 32 W reads; its warps walk the SAME program position, so the program is
// fetched once per CTA: thread 0 issues one bulk copy (TMA, cp.async.bulk + mbarrier) per chunk into a double
// buffer in shared memory while the warps work through the previous chunk, and every record, emission weight
// and state value a term needs is then a shared-memory read.  Per warp: the window, the ring, the hub slots
// (rows of 32 doubles: every access of the warp is one conflict-free 256-byte row).  Global memory sees the
// tokens, the live vectors (out once, back in once through the ring, per cell) and the Viterbi back-pointers.
// ---------------------------------------------------------------------------------------------
struct L2Params {
  const char* blob;
  int32_t nChunks, blobBytes, emOff, idxOff;
  int32_t LA, WN, RN, nHubS, nHubD, nLive;
  int32_t S, nOut, bpBytes;
  DevBatch b;
  const int64_t* order; int64_t nWork;       // reads, longest first; task n = reads [32n, 32n+32)
  unsigned long long* counter;
  double* result; int32_t* flag;
  double* vec;                                // per resident warp: 2 live vectors of nLive * 32 doubles
  unsigned char* bp; const int64_t* bpOff;   // back-pointers of task n at bpOff[n]: [o][state][lane]
};

__device__ __forceinline__ void l2_cp_async8 (void* smem, const void* gmem) {
  asm volatile ("cp.async.ca.shared.global [%0], [%1], 8;" :: "r"((unsigned) __cvta_generic_to_shared (smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void l2_commit() { asm volatile ("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void l2_wait (const int pending) {      // at most `pending` groups still in flight
  if (pending <= 0) asm volatile ("cp.async.wait_group 0;" ::: "memory");
  else if (pending == 1) asm volatile ("cp.async.wait_group 1;" ::: "memory");
  else if (pending == 2) asm volatile ("cp.async.wait_group 2;" ::: "memory");
  else if (pending == 3) asm volatile ("cp.async.wait_group 3;" ::: "memory");
  else if (pending == 4) asm volatile ("cp.async.wait_group 4;" ::: "memory");
  else if (pending == 5) asm volatile ("cp.async.wait_group 5;" ::: "memory");
  else if (pending == 6) asm volatile ("cp.async.wait_group 6;" ::: "memory");
  else if (pending == 7) asm volatile ("cp.async.wait_group 7;" ::: "memory");
  else asm volatile ("cp.async.wait_group 8;" ::: "memory");
}
// one-dimensional bulk copy global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void l2_mbar_init (const unsigned mbar, const unsigned count) { asm volatile ("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(mbar), "r"(count) : "memory"); }
__device__ __forceinline__ void l2_bulk_load (const unsigned dst, const void* src, const unsigned bytes, const unsigned mbar) {
  asm volatile ("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mbar), "r"(bytes) : "memory");
  asm volatile ("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" :: "r"(dst), "l"(src), "r"(bytes), "r"(mbar) : "memory");
}
__device__ __forceinline__ void l2_mbar_wait (const unsigned mbar, const unsigned parity) {
  unsigned ok;
  do {
    asm volatile ("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(mbar), "r"(parity) : "memory");
  } while (!ok);
}

template<int OP, int R>
__global__ void __launch_bounds__(256) lane2_kernel (const __grid_constant__ L2Params p) {
  extern __shared__ __align__(16) char l2smemRaw[];
  __shared__ long long sTask;
  __shared__ int sMaxLo;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nWarps = blockDim.x >> 5;
  constexpr int LPT = 32 * R;      // reads per warp: read q of a lane is read q * 32 + lane of the warp's task
  // shared memory: two chunk buffers | two mbarriers | per warp: its region (window, ring, hub sources, hub destinations: rows of
  // LPT doubles, every access of the warp one conflict-free 256-byte line) | (L_MAX) hub-destination pointers
  char* buf0 = l2smemRaw;
  const unsigned bufAddr = (unsigned) __cvta_generic_to_shared (buf0);
  const unsigned mbarAddr = bufAddr + 2u * (unsigned) p.blobBytes;
  double* warpBase = reinterpret_cast<double*> (l2smemRaw + 2 * p.blobBytes + 16);
  const int rows = p.WN + p.RN + p.nHubS + p.nHubD, rowHubD = p.WN + p.RN + p.nHubS;
  double* region = warpBase + (size_t) warp * rows * LPT + lane;
  unsigned* hubDB = reinterpret_cast<unsigned*> (warpBase + (size_t) nWarps * rows * LPT) + (size_t) warp * L2_MAXHUB * LPT + lane;      // L_MAX only
  double* v0 = p.vec + ((size_t) blockIdx.x * nWarps + warp) * 2 * (size_t) p.nLive * LPT + lane;
  double* v1 = v0 + (size_t) p.nLive * LPT;
  const double ZERO = OP == L_SUM ? 0. : l_ninf(), ONE = OP == L_SUM ? 1. : 0.;
  const unsigned kb = p.bpBytes == 1 ? 6 : 14;
  const double LN2 = 0.693147180559945309417232121458;
  if (tid == 0) {
    l2_mbar_init (mbarAddr, 1);
    l2_mbar_init (mbarAddr + 8, 1);
    asm volatile ("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  unsigned phase0 = 0, phase1 = 0;      // parity of the next completion of each buffer's mbarrier
  for (;;) {
    __syncthreads();      // (sTask, sMaxLo of the previous round have been read by everyone)
    if (tid == 0) { sTask = (long long) atomicAdd (p.counter, (unsigned long long) nWarps); sMaxLo = -1; }
    __syncthreads();
    const long long task = sTask + warp;
    if (sTask * LPT >= p.nWork) break;
    int64_t k[R];
    const uint8_t* y[R];
    int Lo[R], warpMaxLo = -1;
#pragma unroll
    for (int q = 0; q < R; ++q) {
      const long long rd = task * LPT + q * 32 + lane;
      const bool have = rd < p.nWork;
      k[q] = have ? p.order[rd] : 0;
      y[q] = p.b.y + p.b.yOff[k[q]];
      Lo[q] = have ? (int) (p.b.yOff[k[q] + 1] - p.b.yOff[k[q]]) : -1;
      warpMaxLo = max (warpMaxLo, Lo[q]);
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) warpMaxLo = max (warpMaxLo, __shfl_xor_sync (0xffffffffu, warpMaxLo, off));
    if (lane == 0) atomicMax (&sMaxLo, warpMaxLo);
    __syncthreads();
    const int ctaMaxLo = sMaxLo;
    unsigned char* bp = OP == L_MAX && p.bp && task * LPT < p.nWork ? p.bp + p.bpOff[task] + (size_t) lane * p.bpBytes : nullptr;
    bool bad[R];
    int Fprev[R], Gprev[R];
#pragma unroll
    for (int q = 0; q < R; ++q) { bad[q] = false; Fprev[q] = 0; Gprev[q] = L_SENT; }
    for (int o = 0; o <= ctaMaxLo; ++o) {
      const bool active = o <= warpMaxLo;      // (a warp whose reads have ended keeps the CTA's barriers company)
      double* cur = (o & 1) ? v1 : v0;
      const double* prev = (o & 1) ? v0 : v1;
      int tok[R], F[R], mx[R];
      unsigned mn[R], best[R];
      double f[R], acc[R], res[R], vlast[R];
#pragma unroll
      for (int q = 0; q < R; ++q) {
        tok[q] = (o <= Lo[q] && o > 0) ? y[q][o - 1] - 1 : 0;
        F[q] = 0; f[q] = 1.;
        if (OP == L_SUM && o > 0) { if (Gprev[q] == L_SENT) f[q] = 0.; else { F[q] = Gprev[q]; f[q] = l_pow2 (Fprev[q] - F[q]); } }
        mx[q] = 0; mn[q] = 0xffffffffu; best[q] = 0xffffu;
        acc[q] = ZERO; res[q] = ZERO; vlast[q] = ZERO;
      }
      if (active)
        for (int hd = 0; hd < p.nHubD; ++hd) {
#pragma unroll
          for (int q = 0; q < R; ++q) { region[(rowHubD + hd) * LPT + q * 32] = ZERO; if (OP == L_MAX) hubDB[hd * LPT + q * 32] = 0xffffu; }
        }
      const bool usePrev = o > 0;
      double* curOut = cur;
      unsigned char* bpRow = bp ? bp + (size_t) o * p.S * LPT * p.bpBytes : nullptr;
      __syncthreads();      // everyone has left the previous cell's last chunk: its buffer may be refilled
      if (tid == 0) l2_bulk_load (bufAddr, p.blob, (unsigned) p.blobBytes, mbarAddr);
      for (int c = 0; c < p.nChunks; ++c) {
        if (c > 0) __syncthreads();      // chunk c - 1 is done with: its buffer takes chunk c + 1
        if (tid == 0 && c + 1 < p.nChunks)
          l2_bulk_load (bufAddr + (unsigned) (((c + 1) & 1) * p.blobBytes), p.blob + (size_t) (c + 1) * p.blobBytes, (unsigned) p.blobBytes, mbarAddr + 8u * ((c + 1) & 1));
        if (c & 1) { l2_mbar_wait (mbarAddr + 8, phase1); phase1 ^= 1u; } else { l2_mbar_wait (mbarAddr, phase0); phase0 ^= 1u; }
        if (!active) continue;
        const char* bl = buf0 + (c & 1) * p.blobBytes;
        const uint4* rec = reinterpret_cast<const uint4*> (bl);
        const double* em = reinterpret_cast<const double*> (bl + p.emOff);
        const uint16_t* emIdx = reinterpret_cast<const uint16_t*> (bl + p.idxOff);
        uint4 nx = rec[0];
#pragma unroll 2
        for (int n = 0; n < L3_NREC; ++n) {
          const uint4 u = nx;
          nx = rec[n + 1];      // (the record area ends with a spare record)
          double* row = region + u.z * LPT;
          switch (u.w & 15u) {
            case X_TERM: {
              const double w = __hiloint2double ((int) u.y, (int) u.x);
              double x[R];
#pragma unroll
              for (int q = 0; q < R; ++q) x[q] = row[q * 32];
#pragma unroll
              for (int q = 0; q < R; ++q) {
                if (OP == L_SUM) acc[q] = fma (w, x[q], acc[q]);
                else if (OP == L_LSE) acc[q] = l_lse (acc[q], x[q] + w);
                else { const double cnd = x[q] + w; if (acc[q] < cnd) { acc[q] = cnd; best[q] = ((unsigned) T_SILENT << kb) | (u.w >> 16); } }
              }
              break;
            }
            case X_END: {
#pragma unroll
              for (int q = 0; q < R; ++q) {
                row[q * 32] = acc[q];
                vlast[q] = acc[q];
                res[q] = acc[q];      // after the last record: the end state
              }
              if (u.w & 32u) {
#pragma unroll
                for (int q = 0; q < R; ++q) region[u.x * LPT + q * 32] = acc[q];
              }
              if (u.w & 16u) {      // a live state: it crosses to the next cell, and sets that cell's frame
#pragma unroll
                for (int q = 0; q < R; ++q) {
                  curOut[q * 32] = acc[q];
                  if (OP == L_SUM) {
                    const int hi = __double2hiint (acc[q]);
                    mx[q] = max (mx[q], hi);
                    mn[q] = min (mn[q], (unsigned) (hi - 0x00100000));      // zeros and denormals wrap to the top and drop out
                  }
                }
                curOut += LPT;
              }
              if (OP == L_MAX && bpRow) {
#pragma unroll
                for (int q = 0; q < R; ++q) {
                  if (p.bpBytes == 1) bpRow[q * 32] = (unsigned char) best[q]; else reinterpret_cast<uint16_t*> (bpRow)[q * 32] = (uint16_t) best[q];
                }
                bpRow += LPT * p.bpBytes;
              }
#pragma unroll
              for (int q = 0; q < R; ++q) { acc[q] = ZERO; best[q] = 0xffffu; }
              break;
            }
            case X_EMIT: {
              if (usePrev) {
                double x[R], w[R];
#pragma unroll
                for (int q = 0; q < R; ++q) { x[q] = row[q * 32]; w[q] = em[u.x * p.nOut + tok[q]]; }
#pragma unroll
                for (int q = 0; q < R; ++q) {
                  if (OP == L_SUM) acc[q] = fma (w[q], x[q], acc[q]);
                  else if (OP == L_LSE) acc[q] = l_lse (acc[q], x[q] + w[q]);
                  else { const double cnd = x[q] + w[q]; if (acc[q] < cnd) { acc[q] = cnd; best[q] = ((unsigned) T_INSERT << kb) | emIdx[u.x * p.nOut + tok[q]]; } }
                }
              }
              if (OP == L_SUM && (u.w & 16u)) {
#pragma unroll
                for (int q = 0; q < R; ++q) acc[q] *= f[q];
              }
              break;
            }
            case X_PUSH: {
              const double w = __hiloint2double ((int) u.y, (int) u.x);
#pragma unroll
              for (int q = 0; q < R; ++q) {
                if (OP == L_SUM) row[q * 32] = fma (w, vlast[q], row[q * 32]);
                else if (OP == L_LSE) row[q * 32] = l_lse (row[q * 32], vlast[q] + w);
                else { const double cnd = vlast[q] + w; if (row[q * 32] < cnd) { row[q * 32] = cnd; hubDB[((u.w >> 4) & 7u) * LPT + q * 32] = ((unsigned) T_SILENT << kb) | (u.w >> 16); } }
              }
              break;
            }
            case X_LOAD: {
              if (usePrev) {
#pragma unroll
                for (int q = 0; q < R; ++q) l2_cp_async8 (row + q * 32, prev + (size_t) u.x * LPT + q * 32);
              }
              break;
            }
            case X_CTRL: {
              if (usePrev && (u.z & L3_COMMIT)) l2_commit();
              if (usePrev && (u.z & L3_WAIT)) { if (p.LA == 3) asm volatile ("cp.async.wait_group 3;" ::: "memory"); else l2_wait (p.LA); }
              if (u.z & L3_ORIGIN) {
#pragma unroll
                for (int q = 0; q < R; ++q) acc[q] = o == 0 ? ONE : ZERO;
              }
              break;
            }
            case X_HINIT: {
#pragma unroll
              for (int q = 0; q < R; ++q) { acc[q] = row[q * 32]; if (OP == L_MAX) best[q] = hubDB[((u.w >> 4) & 7u) * LPT + q * 32]; }
              break;
            }
            case X_PRESTORE: {
#pragma unroll
              for (int q = 0; q < R; ++q) {
                row[q * 32] = acc[q];
                if (OP == L_MAX) hubDB[((u.w >> 4) & 7u) * LPT + q * 32] = best[q];
                acc[q] = ZERO; best[q] = 0xffffu;
              }
              break;
            }
            default: break;
          }
        }
      }
      if (usePrev && active) l2_wait (0);
      if (active) {
#pragma unroll
        for (int q = 0; q < R; ++q) {
          if (OP == L_SUM) {
            int Gc = L_SENT;
            if (mx[q] >= 0x00100000) {
              const int emx = mx[q] >> 20;
              Gc = F[q] + emx - 1023;
              if (o <= Lo[q] && (emx == 0x7ff || (mn[q] != 0xffffffffu && emx - (int) ((mn[q] >> 20) + 1) > L_SPREAD))) bad[q] = true;
            }
            Fprev[q] = F[q]; Gprev[q] = Gc;
          }
          if (o == Lo[q]) {
            if (OP == L_SUM) { p.result[k[q]] = res[q] > 0. ? log (res[q]) + F[q] * LN2 : l_ninf(); p.flag[k[q]] = bad[q] || !(res[q] > 0.) || !(res[q] < 1e300); }
            else p.result[k[q]] = res[q];
          }
        }
      }
    }
  }
}

// reads per lane.  Measured on B200 (PF00516, reads of 275): with enough reads to give every SM some 40
// warps, one read per lane is fastest (262 144 reads: 175 GCUPS Forward, 132 Viterbi); with fewer, a second
// independent chain per thread makes up for the missing warps in the sums (65 536 reads: 40 -> 89 GCUPS),
// while the max-plus sweep, which carries a pointer per chain, stays at one.
static int lane_reads_per_lane (const mb_machine* m, const LHost* h, int64_t nWork, int op) {
  if (m->opt.has ("lane_r")) { const int r = m->opt.get ("lane_r", 1); return r >= 4 ? 4 : r >= 2 ? 2 : 1; }
  // the windowed sweep: one read per lane.  More reads per lane share the interpreter's work per record but cost warps
  // (shared memory), and the sweep lives on warps: measured on B200, PF00516, 65 536 ragged reads: 114 / 108 / 98 GCUPS
  // at 1 / 2 / 4 reads per lane
  if (h->l2.ok) return 1;
  if (op == L_MAX || nWork >= (int64_t) h->numSMs * 40 * 32) return 1;
  return nWork >= (int64_t) h->numSMs * 8 * 64 ? 2 : 1;
}

template<int OP, int R>
static int lane_launch_r (mb_machine* m, mb_batch* b, const std::vector<int64_t>& order, double* dResult, int32_t* dFlag,
                          unsigned char* dBp, const int64_t* dBpOff) {
  LHost* h = lh (m);
  constexpr int LPT = 32 * R;
  const int64_t nWork = (int64_t) order.size(), nTasks = (nWork + LPT - 1) / LPT;
  int ctas = 0;
  MB_CUDA (cudaOccupancyMaxActiveBlocksPerMultiprocessor (&ctas, lane_kernel<OP, R>, 128, 0));
  int warpsPerSM = 48;      // the sweep is bound by the latency of its state-vector loads: as many warps as the registers allow
  if (m->opt.has ("lane_warps")) warpsPerSM = std::max (4, m->opt.get ("lane_warps", 48));
  ctas = std::max (1, std::min (ctas, warpsPerSM / 4));
  // few tasks: one warp per CTA spreads them over the SMs
  const int threads = nTasks >= (int64_t) ctas * h->numSMs * 4 ? 128 : nTasks >= (int64_t) h->numSMs * 2 ? 64 : 32;
  const int wpc = threads / 32;
  const int grid = (int) std::max<int64_t> (1, std::min<int64_t> ((nTasks + wpc - 1) / wpc, (int64_t) ctas * h->numSMs));
  // scratch from the batch's grow-only workspace: a repeated call allocates nothing
  b->wsOrderHoldsFull = false;
  int64_t* dOrder = (int64_t*) ws_reserve (b, WS_ORDER, order.size() * 8);
  unsigned long long* dCounter = (unsigned long long*) ws_reserve (b, WS_COUNTER, 8);
  double* dVec = (double*) ws_reserve (b, WS_BND, (size_t) grid * wpc * 2 * h->S * LPT * 8);
  if (!dOrder || !dCounter || !dVec) return 1;
  MB_CUDA (cudaMemcpyAsync (dOrder, order.data(), order.size() * 8, cudaMemcpyHostToDevice, b->stream));
  MB_CUDA (cudaMemsetAsync (dCounter, 0, 8, b->stream));
  LParams p {};
  p.rec = OP == L_SUM ? h->dRecLin : h->dRecLog; p.nRec = h->nRec;
  p.em = OP == L_SUM ? h->dEmLin : h->dEmLog; p.emIdx = h->dEmIdx;
  p.S = h->S; p.nOut = h->nOut; p.bpBytes = h->bpBytes;
  p.b = b->dev;
  p.order = dOrder; p.nWork = nWork; p.counter = dCounter;
  p.result = dResult; p.flag = dFlag; p.vec = dVec;
  p.bp = dBp; p.bpOff = dBpOff;
  lane_kernel<OP, R><<<grid, threads, 0, b->stream>>> (p);
  MB_CUDA (cudaGetLastError());
  return 0;
}

// the windowed sweep (lane2): CTAs of W warps of 32 * R reads, as many per SM as shared memory holds
template<int OP, int R>
static int lane2_launch_r (mb_machine* m, mb_batch* b, const std::vector<int64_t>& order, double* dResult, int32_t* dFlag,
                           unsigned char* dBp, const int64_t* dBpOff) {
  LHost* h = lh (m);
  const L2Prog& P = h->l2;
  constexpr int LPT = 32 * R;
  const int64_t nWork = (int64_t) order.size(), nTasks = (nWork + LPT - 1) / LPT;
  const size_t perWarp = (size_t) (P.WN + P.RN + P.nHubS + P.nHubD) * LPT * 8 + (OP == L_MAX ? (size_t) L2_MAXHUB * LPT * 4 : 0);
  const size_t fixed = 2 * (size_t) P.blobBytes + 16 + 64;
  const size_t kSmem = 227 * 1024 - 2048;      // (the kernel's two static words included)
  // warps per CTA: the one of 8, 6, 4, 3, 2, 1 that gives the most warps per SM (the largest on a tie)
  int W = 1, ctasPerSM = 1, bestWarps = 0;
  const int wantW = m->opt.get ("lane_warps_per_cta", 0);
  for (int w: { 8, 6, 4, 3, 2, 1 }) {
    if (wantW && w != wantW) continue;
    const size_t need = fixed + (size_t) w * perWarp;
    if (need > kSmem) continue;
    const int c = (int) std::min<size_t> (kSmem / need, 32 / w);
    if (c * w > bestWarps) { bestWarps = c * w; W = w; ctasPerSM = c; }
  }
  if (!bestWarps) { set_error ("lane engine: the window does not fit in shared memory"); return 1; }
  // few reads: narrower CTAs (and as many of them as fit) spread the tasks over the SMs
  while (W > 1 && !wantW && nTasks < (int64_t) h->numSMs * W * ctasPerSM) {
    W = (W + 1) / 2;
    ctasPerSM = (int) std::min<size_t> (kSmem / (fixed + (size_t) W * perWarp), 32 / W);
  }
  if (m->opt.has ("lane_warps")) ctasPerSM = std::max (1, std::min (ctasPerSM, m->opt.get ("lane_warps", 16) / W));
  const int grid = (int) std::max<int64_t> (1, std::min<int64_t> ((nTasks + W - 1) / W, (int64_t) ctasPerSM * h->numSMs));
  const size_t smem = fixed + (size_t) W * perWarp;
  MB_CUDA (cudaFuncSetAttribute (lane2_kernel<OP, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem));
  b->wsOrderHoldsFull = false;
  int64_t* dOrder = (int64_t*) ws_reserve (b, WS_ORDER, order.size() * 8);
  unsigned long long* dCounter = (unsigned long long*) ws_reserve (b, WS_COUNTER, 8);
  double* dVec = (double*) ws_reserve (b, WS_BND, (size_t) grid * W * 2 * std::max (P.nLive, 1) * LPT * 8);
  if (!dOrder || !dCounter || !dVec) return 1;
  MB_CUDA (cudaMemcpyAsync (dOrder, order.data(), order.size() * 8, cudaMemcpyHostToDevice, b->stream));
  MB_CUDA (cudaMemsetAsync (dCounter, 0, 8, b->stream));
  L2Params p {};
  p.blob = OP == L_SUM ? P.dBlobLin : P.dBlobLog;
  p.nChunks = P.nChunks; p.blobBytes = P.blobBytes; p.emOff = P.emOff; p.idxOff = P.idxOff;
  p.LA = P.LA; p.WN = P.WN; p.RN = P.RN; p.nHubS = P.nHubS; p.nHubD = P.nHubD; p.nLive = P.nLive;
  p.S = h->S; p.nOut = std::max (h->nOut, 1); p.bpBytes = h->bpBytes;
  p.b = b->dev;
  p.order = dOrder; p.nWork = nWork; p.counter = dCounter;
  p.result = dResult; p.flag = dFlag; p.vec = dVec;
  p.bp = dBp; p.bpOff = dBpOff;
  if (m->opt.get ("verbose", 0))
    fprintf (stderr, "lane engine (windowed): %lld reads, %d per lane, grid %d x %d threads (%d CTAs per SM), %zu B smem per CTA, window %d, ring %d, hubs %d + %d, %d live of %d states, %zu records in %d chunks of %d B\n",
             (long long) nWork, R, grid, 32 * W, ctasPerSM, smem, P.WN, P.RN, P.nHubS, P.nHubD, P.nLive, h->S, P.flat.size(), P.nChunks, P.blobBytes);
  lane2_kernel<OP, R><<<grid, 32 * W, smem, b->stream>>> (p);
  MB_CUDA (cudaGetLastError());
  return 0;
}

template<int OP>
static int lane_launch (mb_machine* m, mb_batch* b, int R, const std::vector<int64_t>& order, double* dResult, int32_t* dFlag,
                        unsigned char* dBp, const int64_t* dBpOff) {
  if (lh (m)->l2.ok)
    return R >= 4 ? lane2_launch_r<OP, 4> (m, b, order, dResult, dFlag, dBp, dBpOff) : R == 2 ? lane2_launch_r<OP, 2> (m, b, order, dResult, dFlag, dBp, dBpOff)
                  : lane2_launch_r<OP, 1> (m, b, order, dResult, dFlag, dBp, dBpOff);
  return R == 4 ? lane_launch_r<OP, 4> (m, b, order, dResult, dFlag, dBp, dBpOff)
       : R == 2 ? lane_launch_r<OP, 2> (m, b, order, dResult, dFlag, dBp, dBpOff)
                : lane_launch_r<OP, 1> (m, b, order, dResult, dFlag, dBp, dBpOff);
}

std::vector<int64_t> lane_order (const mb_batch* b, const std::vector<int64_t>* subset) {
  std::vector<int64_t> order;
  if (subset) order = *subset;
  else { order.resize ((size_t) b->nPairs); for (int64_t k = 0; k < b->nPairs; ++k) order[k] = k; }
  std::stable_sort (order.begin(), order.end(), [&] (int64_t a, int64_t c) { return b->yOff[a + 1] - b->yOff[a] > b->yOff[c + 1] - b->yOff[c]; });
  return order;
}

bool lane_wanted (const mb_machine* m, const mb_batch* b) {
  if (b->hasEnv || m->opt.get ("no_lane", 0)) return false;
  for (int64_t k = 0; k < b->nPairs; ++k) if (b->xOff[k + 1] != b->xOff[k]) return false;
  return true;
}

int lane_forward_log_subset (mb_machine* m, mb_batch* b, const std::vector<int64_t>& pairs, double* dResult, int32_t* dFlag) {
  if (!m->lane) { set_error ("lane engine not prepared for this machine"); return 1; }
  return lane_launch<L_LSE> (m, b, lane_reads_per_lane (m, lh (m), (int64_t) pairs.size(), L_LSE), lane_order (b, &pairs), dResult, dFlag, nullptr, nullptr);
}

int lane_forward (mb_machine* m, mb_batch* b, double* loglike) {
  b->lastRedo = 0;
  if (b->nPairs == 0) return 0;
  LHost* h = lh (m);
  const std::vector<int64_t> order = lane_order (b, nullptr);
  DevBuf dRes, dFlag;
  if (dRes.alloc ((size_t) b->nPairs * 8) || dFlag.alloc ((size_t) b->nPairs * 4)) return 1;
  MB_CUDA (cudaMemsetAsync (dFlag.p, 0, (size_t) b->nPairs * 4, b->stream));
  if (timing_begin (b)) return 1;
  int64_t launches = 1;
  const int R = lane_reads_per_lane (m, h, b->nPairs, L_SUM);
  if (h->linearOk) {
    if (lane_launch<L_SUM> (m, b, R, order, dRes.as<double>(), dFlag.as<int32_t>(), nullptr, nullptr)) return 1;
    std::vector<int32_t> flag ((size_t) b->nPairs);
    MB_CUDA (cudaMemcpyAsync (flag.data(), dFlag.p, flag.size() * 4, cudaMemcpyDeviceToHost, b->stream));
    MB_CUDA (cudaStreamSynchronize (b->stream));
    std::vector<int64_t> redo;
    for (int64_t k = 0; k < b->nPairs; ++k) if (flag[k]) redo.push_back (k);
    if (!redo.empty()) {
      if (lane_forward_log_subset (m, b, redo, dRes.as<double>(), dFlag.as<int32_t>())) return 1;
      ++launches;
    }
    b->lastRedo = (int64_t) redo.size();
  } else if (lane_launch<L_LSE> (m, b, R, order, dRes.as<double>(), dFlag.as<int32_t>(), nullptr, nullptr)) return 1;
  if (timing_end (b, launches)) return 1;
  MB_CUDA (cudaMemcpy (loglike, dRes.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  return 0;
}

// traceback over lane-interleaved back-pointers (mb_wide.cu)
int wide_traceback_launch (mb_machine* m, mb_batch* b, const int64_t* dOrder, int64_t nWork, const unsigned char* dBp, const int64_t* dBpOff,
                           int bpBytes, int laneLayout, const double* dScore, int64_t* dLen, int32_t* dOut, const int64_t* dOutOff);

int lane_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen) {
  if (b->nPairs == 0) return 0;
  LHost* h = lh (m);
  const bool trace = pathLen != nullptr;
  const std::vector<int64_t> order = lane_order (b, nullptr);
  DevBuf dRes;
  if (dRes.alloc ((size_t) b->nPairs * 8)) return 1;
  if (!trace) {
    if (timing_begin (b)) return 1;
    if (lane_launch<L_MAX> (m, b, lane_reads_per_lane (m, h, b->nPairs, L_MAX), order, dRes.as<double>(), nullptr, nullptr, nullptr)) return 1;
    if (timing_end (b, 1)) return 1;
    MB_CUDA (cudaMemcpy (score, dRes.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
    return 0;
  }
  // chunks of whole tasks (LPT reads) whose back-pointers, (maxLo+1) * S * LPT bytes or half-words per task, fit in free memory
  const int R = lane_reads_per_lane (m, h, b->nPairs, L_MAX), LPT = 32 * R;
  size_t freeB = 0, totalB = 0;
  MB_CUDA (cudaMemGetInfo (&freeB, &totalB));
  const double vecBytes = (double) h->numSMs * 48 * 2 * h->S * LPT * 8;
  const double budget = 0.75 * ((double) freeB - vecBytes);
  int64_t launches = 0;
  double ms = 0;
  for (size_t c0 = 0; c0 < order.size();) {
    std::vector<int64_t> bpOff;
    double bytes = 0;
    size_t c1 = c0;
    while (c1 < order.size()) {
      const int64_t k = order[c1];      // the task's longest read
      const double need = (double) (b->yOff[k + 1] - b->yOff[k] + 1) * h->S * LPT * h->bpBytes;
      if (need > budget) { set_error ("a task of reads needs more device memory for its back-pointers than is free (" + std::to_string (need) + " bytes)"); return 1; }
      if (c1 > c0 && bytes + need > budget) break;
      bpOff.push_back ((int64_t) bytes);
      bytes += need;
      c1 = std::min (order.size(), c1 + (size_t) LPT);
    }
    std::vector<int64_t> chunk (order.begin() + c0, order.begin() + c1);
    c0 = c1;
    std::vector<int64_t> bpOffRead (chunk.size());      // the traceback kernel indexes by read
    for (size_t n = 0; n < chunk.size(); ++n) bpOffRead[n] = bpOff[n / LPT];
    DevBuf dBp, dBpOff, dBpOffRead, dOrder, dLen, dOutOff;
    if (dBp.alloc ((size_t) bytes) || dBpOff.alloc (bpOff.size() * 8) || dBpOffRead.alloc (chunk.size() * 8) || dOrder.alloc (chunk.size() * 8) || dLen.alloc (chunk.size() * 8)
        || dOutOff.alloc (chunk.size() * 8)) return 1;
    MB_CUDA (cudaMemcpyAsync (dBpOff.p, bpOff.data(), bpOff.size() * 8, cudaMemcpyHostToDevice, b->stream));
    MB_CUDA (cudaMemcpyAsync (dBpOffRead.p, bpOffRead.data(), bpOffRead.size() * 8, cudaMemcpyHostToDevice, b->stream));
    MB_CUDA (cudaMemcpyAsync (dOrder.p, chunk.data(), chunk.size() * 8, cudaMemcpyHostToDevice, b->stream));
    if (timing_begin (b)) return 1;
    if (lane_launch<L_MAX> (m, b, R, chunk, dRes.as<double>(), nullptr, dBp.as<unsigned char>(), dBpOff.as<int64_t>())) return 1;
    const int64_t nWork = (int64_t) chunk.size();
    if (wide_traceback_launch (m, b, dOrder.as<int64_t>(), nWork, dBp.as<unsigned char>(), dBpOffRead.as<int64_t>(), h->bpBytes, LPT,
                               dRes.as<double>(), dLen.as<int64_t>(), nullptr, nullptr)) return 1;
    if (paths_place (b, chunk.data(), nWork, dLen.as<int64_t>(), dOutOff.as<int64_t>())) return 1;
    if (wide_traceback_launch (m, b, dOrder.as<int64_t>(), nWork, dBp.as<unsigned char>(), dBpOffRead.as<int64_t>(), h->bpBytes, LPT,
                               dRes.as<double>(), dLen.as<int64_t>(), b->dPaths, dOutOff.as<int64_t>())) return 1;
    launches += 3;
    if (timing_end (b, launches)) return 1;
    ms += b->lastMs;
  }
  b->lastMs = ms;
  b->lastLaunches = launches;
  MB_CUDA (cudaMemcpy (score, dRes.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  return 0;
}

}  // namespace mb
