// mb_wide.cu -- the wide engine: Forward log-likelihood and Viterbi (+ traceback) for machines too
// large for the register-resident strip kernels of mb_jit.cu (composed transducers with tens to
// thousands of states: SURVEY.md section 8 configs 4-5), and for batches that carry envelopes.
//
//   reference                                              here
//   MappedForwardMatrix::fill / logLike  forward.defs.h:22-55   wide_kernel<OP_SUM>  (scaled linear domain)
//                                                               wide_kernel<OP_LSE>  (log domain: flagged pairs, extreme weights)
//   ViterbiMatrix::fill / logLike        viterbi.cpp:18-47      wide_kernel<OP_MAX>  (FP64 add + compare: bit-exact)
//   DPMatrix::traceBack                  dpmatrix.defs.h:82-110 wide_traceback_kernel (stored back-pointers)
//
// Mapping.  A group of G lanes (32, 16 or 8, chosen per machine) owns one input position (a matrix
// column); the states of a cell are spread over its lanes.  A CTA of W column warps (+1 loader
// warp) sweeps a strip of W*32/G columns down the output rows in a skew (column j works on output
// row t-j at step t), so the three neighbour cells a cell needs -- (i,o-1) own previous step,
// (i-1,o) left neighbour's previous step, (i-1,o-1) left neighbour's step before that -- sit in a
// ring of 2-3 cells per column in SHARED memory, with one CTA barrier per step.  The last column
// of a strip hands its live states (sources of input-consuming transitions) to the next strip
// through an L2-resident row buffer that the loader warp streams back in one row ahead.
//
// Within a cell the work is a sparse matrix-vector product over the token-selected transition
// lists.  The host lays every dependency-free set of lists (one silent level, or one token context
// of match / delete / insert) out as ROWS of G 16-byte entries: lane l walks its column of the
// table, one multiply-add per row, lists back to back (longest-processing-time-first over the
// lanes), with per-entry flags saying where a list starts, where it ends (add into the destination
// state) and where the group has to synchronise before the next dependency level.  A list much
// longer than its level's share is cut into 2^k pieces on adjacent lanes that are combined with
// shuffles.  The tables live in shared memory when they fit, next to the rings.
//
// Arithmetic.  Forward: probabilities, one FMA per transition; every cell carries a power-of-two
// frame (F) and the exponent of its largest value (G); a cell is computed in the frame
// max(G of its neighbours), the neighbour sums entering through one exact power-of-two factor each,
// so nothing is ever renormalised in place.  A cell whose values span more than 2^600, or whose
// neighbours' frames are that far apart, flags the pair; flagged pairs are re-run in the log domain
// (mb_last_redo counts them).  Viterbi: log-weights, FP64 add + compare in the reference's
// candidate order with a strict '<' (first maximum wins), so scores and paths are identical; a
// back-pointer (kind, index in the token-selected list) is stored per cell-state.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "mb_internal.h"

namespace mb {

enum { OP_SUM = 0, OP_MAX = 1, OP_LSE = 2 };      // scaled linear sum, max-plus with back-pointers, log-sum-exp
#define W_SENT (-(1 << 29))      // G of an empty (all-zero) cell
#define W_SPREAD 600             // exponent spread that hands a pair to the log-domain sweep
// entry word z: source state (16) | candidate index in its list (14) | first of a list | last of a list
#define W_FIRST 0x40000000u
#define W_LAST 0x80000000u
// entry word w: destination state (16) | log2 pieces (3) | reduce row | sync row | store | end of a list piece.
// One test of the last four bits separates the plain rows (load, multiply-add) from the rest.
#define W_REDUCE 0x80000u
#define W_SYNC 0x100000u
#define W_STORE 0x200000u
#define W_PEND 0x400000u
#define W_SPECIAL (W_REDUCE | W_SYNC | W_STORE | W_PEND)

struct WEntry { double w; uint32_t z; uint32_t d; };

struct WideTables {       // byte offsets into one blob (entries first: the two blobs differ only in their weights)
  uint32_t oEnt, oPhM, oPhD, oPhI, oLive, bytes;
  uint32_t silRow0, silRow1;
  int32_t S, nIn, nOut, hasMatch, nLiveIn, bpBytes, G;
};

struct WParams {
  WideTables t;
  const char* blob;
  int32_t W, R, oneD;      // W: column warps per CTA (each 32/G columns)
  DevBatch b;
  const int64_t* order;
  int64_t nWork;
  unsigned long long* counter;
  double* result;
  int32_t* flag;
  double* bnd;          // per CTA: 2 buffers of bndRows * nLiveIn doubles
  int2* bndFG;          // per CTA: 2 buffers of bndRows (F, G)
  int64_t bndRows;
  unsigned char* bp;    // back-pointers, work item n at bpOff[n] (bytes), layout [o][i][s]
  const int64_t* bpOff;
};

__device__ __forceinline__ double w_ninf() { return __longlong_as_double (0xfff0000000000000LL); }
__device__ __forceinline__ double w_pow2 (int e) {   // 2^e, 0 below the normal range
  return e < -1022 ? 0. : __longlong_as_double ((long long) (e > 1023 ? 2046 : e + 1023) << 52);
}

// log(exp(a)+exp(b)): max, difference and final add in FP64, softplus in FP32 (MUFU ex2/lg2);
// <= 1.2e-7 absolute per operation (the reference's table deviates from the exact function by 4.5e-5)
__device__ __forceinline__ double w_lse (double a, double b) {
  const double mx = fmax (a, b), mn = fmin (a, b);
  const float d = (float) (mn - mx);      // <= 0; -inf or NaN when an operand is -inf
  if (!(d > -40.f)) return mx;
  return mx + (double) __logf (1.f + __expf (d));
}

struct WTab { const WEntry* ent; const uint32_t* phM; const uint32_t* phD; const uint32_t* phI; const uint16_t* live; };

// Rows [row0, row1) of one phase, reading the cell `from` (a neighbour, or the cell itself for
// silent lists).  One table pointer runs through the phase with the next entry always in flight
// (the table ends with a spare row).  SILENT: every group of the warp walks the same rows, so the
// level barriers are whole-warp; the token-selected phases differ between groups and are
// synchronised by the caller.  live == false: a group that only keeps the warp in step.
template<int OP, int G, bool SILENT>
__device__ __forceinline__ void run_rows (const WTab& T, uint32_t row0, uint32_t row1, const double* from, double* cur, uint16_t* bpS,
                                          double f, unsigned kindBits, int gl, unsigned gmask, bool live) {
  if (row0 == row1) return;
  const WEntry* e = T.ent + (size_t) row0 * G + gl;
  uint4 v = *reinterpret_cast<const uint4*> (e);      // this row's entry; the next row's is fetched while this one is worked on,
  double xn = from[v.z & 0xffffu];                    // and its source value as soon as the level barrier (if any) has passed
  double acc = OP == OP_SUM ? 0. : w_ninf();      // OP_MAX: the best candidate so far
  unsigned bp = 0xffffu;
  for (uint32_t row = row0; row < row1; ++row) {
    const uint4 u = v;
    const double x = xn;
    e += G;
    v = *reinterpret_cast<const uint4*> (e);
    const double w = __hiloint2double ((int) u.y, (int) u.x);
    if (OP == OP_MAX) {
      // (the max-plus sweep keeps one test per flag: measured 138 GCUPS on prot2dna => dnapsw against 90 with
      // the combined test below, whose special path most rows take when lists average 1.6 entries)
      if (u.z & W_FIRST) { acc = w_ninf(); bp = 0xffffu; }
      const double c = x + w;
      if (acc < c) { acc = c; bp = kindBits | ((u.z >> 16) & 0x3fffu); }      // strict: the first maximum wins (dpmatrix.defs.h:171-174)
      if (u.w & W_REDUCE) {      // the same row in every lane of the group
        const unsigned segW = 1u << ((u.w >> 16) & 7u);
        for (unsigned off = G / 2; off; off >>= 1) {      // the tree pairs lanes out of list order: a tie goes to the earlier candidate
          const double o2 = __shfl_down_sync (gmask, acc, off, G);
          const unsigned obp = __shfl_down_sync (gmask, bp, off, G);
          if (off < segW && (acc < o2 || (acc == o2 && obp < bp))) { acc = o2; bp = obp; }
        }
      }
      if ((u.z & W_LAST) && live) {
        const unsigned dst = u.w & 0xffffu;
        if (cur[dst] < acc) { cur[dst] = acc; bpS[dst] = (uint16_t) bp; }      // earlier phases keep ties
      }
      if (SILENT && (u.w & W_SYNC)) __syncwarp();
    } else {
      acc = OP == OP_SUM ? fma (w, x, acc) : w_lse (acc, x + w);
      if (u.w & W_SPECIAL) {      // one test separates the plain rows (load, multiply-add) from the rest
        if (u.w & W_REDUCE) {      // the same row in every lane of the group
          const unsigned segW = 1u << ((u.w >> 16) & 7u);
          for (unsigned off = G / 2; off; off >>= 1) {
            const double o2 = __shfl_down_sync (gmask, acc, off, G);
            if (off < segW) acc = OP == OP_SUM ? acc + o2 : w_lse (acc, o2);
          }
        }
        if ((u.w & W_STORE) && live) {
          const unsigned dst = u.w & 0xffffu;
          const double c0 = cur[dst];
          cur[dst] = OP == OP_SUM ? fma (f, acc, c0) : w_lse (c0, acc);
        }
        if (u.w & W_PEND) acc = OP == OP_SUM ? 0. : w_ninf();      // the lane's next list starts on the next row
        if (SILENT && (u.w & W_SYNC)) __syncwarp();
      }
    }
    xn = from[v.z & 0xffffu];      // within a level no list reads a state the level writes, so this may run ahead of the adds above
  }
}

// One cell per lane group, all groups of the warp in step (live == false: nothing to compute, the
// group only walks along).  up/left/diag: neighbour cells (null when outside the matrix or empty).
// Linear domain: fU/fL/fD scale the neighbour sums into this cell's frame.
template<int OP, int G>
__device__ __forceinline__ void compute_cell (const WTab& T, const WideTables& t, double* cur, uint16_t* bpS,
                                              const double* up, const double* left, const double* diag,
                                              double fU, double fL, double fD, int a, int c, bool origin, int gl, unsigned gmask, bool live) {
  const int S = t.S;
  if (live) {
    for (int d = gl; d < S; d += G) { cur[d] = OP == OP_SUM ? 0. : w_ninf(); if (OP == OP_MAX) bpS[d] = 0xffff; }
    if (origin && gl == 0) cur[0] = OP == OP_SUM ? 1. : 0.;      // written by the lane that zeroed it
  }
  __syncwarp();
  const unsigned kb = t.bpBytes == 1 ? 6 : 14;
  // reference candidate order: match, delete, insert, silent (dpmatrix.defs.h:90-103)
  if (t.hasMatch) {
    if (live && diag) { const int k = (a - 1) * t.nOut + (c - 1); run_rows<OP, G, false> (T, T.phM[k], T.phM[k + 1], diag, cur, bpS, fD, (unsigned) T_MATCH << kb, gl, gmask, true); }
    __syncwarp();
  }
  if (t.nIn) {
    if (live && left) run_rows<OP, G, false> (T, T.phD[a - 1], T.phD[a], left, cur, bpS, fL, (unsigned) T_DELETE << kb, gl, gmask, true);
    __syncwarp();
  }
  if (t.nOut) {
    if (live && up) run_rows<OP, G, false> (T, T.phI[c - 1], T.phI[c], up, cur, bpS, fU, (unsigned) T_INSERT << kb, gl, gmask, true);
    __syncwarp();
  }
  run_rows<OP, G, true> (T, t.silRow0, t.silRow1, cur, cur, bpS, 1., (unsigned) T_SILENT << kb, gl, gmask, live);
  __syncwarp();
}

template<int G> __device__ __forceinline__ int group_max (int v) {
#pragma unroll
  for (int off = G / 2; off; off >>= 1) v = max (v, __shfl_xor_sync (0xffffffffu, v, off, G));
  return v;
}

// exponent bookkeeping of a finished linear-domain cell (all groups of the warp call it together):
// returns G (W_SENT if empty); sets bad on overflow, underflow in progress, or an exponent spread beyond W_SPREAD
template<int G>
__device__ __forceinline__ int cell_frame (const double* cur, int S, int F, int gl, bool live, bool& bad) {
  int mx = 0, mnNeg = -0x7fffffff, dust = 0;
  if (live)
    for (int d = gl; d < S; d += G) {
      const double v = cur[d];
      const int hi = __double2hiint (v) & 0x7fffffff;
      mx = max (mx, hi);
      if (hi >= 0x00100000) mnNeg = max (mnNeg, -hi);
      else if (v != 0.) dust = 1;      // a denormal: something is underflowing
    }
  mx = group_max<G> (mx);
  mnNeg = group_max<G> (mnNeg);
  dust = group_max<G> (dust);
  if (!live) return W_SENT;
  if (dust) bad = true;
  if (mx < 0x00100000) return W_SENT;     // an empty cell
  const int emx = mx >> 20, emn = (-mnNeg) >> 20;
  if (emx == 0x7ff || emx - emn > W_SPREAD) bad = true;
  return F + emx - 1023;
}

struct EnvD {
  const int64_t* start; const int64_t* end;
  __device__ __forceinline__ bool contains (int64_t i, int64_t o) const { return !start || (i >= start[o] && i < end[o]); }
};

template<int OP, int G, bool TABS>
__global__ void __launch_bounds__(544) wide_kernel (const __grid_constant__ WParams p) {
  extern __shared__ __align__(16) char smem[];
  constexpr int CPW = 32 / G;      // cells (matrix columns, or pairs in the 1-D sweep) per warp
  const WideTables& t = p.t;
  const int S = t.S, R = p.R;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nWarps = blockDim.x >> 5;
  const int grp = lane / G, gl = lane % G;
  const unsigned gmask = G == 32 ? 0xffffffffu : ((1u << G) - 1u) << (grp * G);
  // ---- shared memory: [tables] [ring: column slots x R cells of S doubles] [FG] [bp stage] [work slot]
  const int nSlots = nWarps * CPW;      // column slots; in the 2-D sweep the last slot of warp 0 is the virtual column left of the strip
  size_t at = 0;
  if (TABS) {
    for (uint32_t n = threadIdx.x * 16; n < t.bytes; n += blockDim.x * 16) *reinterpret_cast<uint4*> (smem + n) = *reinterpret_cast<const uint4*> (p.blob + n);
    at = (t.bytes + 15) & ~(size_t) 15;
  }
  double* ring = reinterpret_cast<double*> (smem + at); at += (size_t) nSlots * R * S * 8;
  int2* fg = reinterpret_cast<int2*> (smem + at); at += (size_t) nSlots * R * 8;
  uint16_t* bpStage = reinterpret_cast<uint16_t*> (smem + at); at += OP == OP_MAX ? (size_t) nSlots * S * 2 : 0;
  at = (at + 7) & ~(size_t) 7;
  volatile long long* workSlot = reinterpret_cast<volatile long long*> (smem + at);
  WTab T;
  if (TABS) T = { reinterpret_cast<const WEntry*> (smem + t.oEnt), reinterpret_cast<const uint32_t*> (smem + t.oPhM), reinterpret_cast<const uint32_t*> (smem + t.oPhD),
                  reinterpret_cast<const uint32_t*> (smem + t.oPhI), reinterpret_cast<const uint16_t*> (smem + t.oLive) };
  else T = { reinterpret_cast<const WEntry*> (p.blob + t.oEnt), reinterpret_cast<const uint32_t*> (p.blob + t.oPhM), reinterpret_cast<const uint32_t*> (p.blob + t.oPhD),
             reinterpret_cast<const uint32_t*> (p.blob + t.oPhI), reinterpret_cast<const uint16_t*> (p.blob + t.oLive) };
  __syncthreads();
  const int mySlot = warp * CPW + grp;
  double* myRing = ring + (size_t) mySlot * R * S;
  int2* myFG = fg + mySlot * R;
  uint16_t* bpS = bpStage + (OP == OP_MAX ? (size_t) mySlot * S : 0);
  const double LN2 = 0.693147180559945309417232121458;

  if (p.oneD) {
    // ---- batches without input sequences: every lane group sweeps its own pair, the groups of a warp in step; no CTA barriers
    for (;;) {
      long long wk0 = 0;
      if (lane == 0) wk0 = (long long) atomicAdd (p.counter, (unsigned long long) CPW);
      wk0 = __shfl_sync (0xffffffffu, wk0, 0);
      if (wk0 >= p.nWork) break;
      const long long wk = wk0 + grp;
      const bool have = wk < p.nWork;
      const int64_t k = have ? p.order[wk] : 0;
      const uint8_t* y = p.b.y + p.b.yOff[k];
      const int64_t Lo = have ? p.b.yOff[k + 1] - p.b.yOff[k] : -1;
      const int64_t maxLo = (int64_t) group_max<32> ((int) Lo);
      EnvD env { nullptr, nullptr };
      if (have && p.b.envOff && p.b.envOff[k + 1] != p.b.envOff[k]) env = EnvD { p.b.envStart + p.b.envOff[k], p.b.envEnd + p.b.envOff[k] };
      unsigned char* bp = OP == OP_MAX && p.bp && have ? p.bp + p.bpOff[wk] : nullptr;
      bool bad = false;
      int slot = 0;
      int Fprev = 0, Gprev = W_SENT;
      double res = OP == OP_SUM ? 0. : w_ninf();
      int Fres = 0;
      for (int64_t o = 0; o <= maxLo; ++o) {
        const bool inRange = o <= Lo;
        double* cur = myRing + (size_t) slot * S;
        const double* up = o ? myRing + (size_t) (slot ^ 1) * S : nullptr;
        const bool inside = inRange && env.contains (0, o);
        int F = 0;
        double fU = 1.;
        if (OP == OP_SUM && up) { if (Gprev == W_SENT) up = nullptr; else { F = Gprev; fU = w_pow2 (Fprev - F); } }
        compute_cell<OP, G> (T, t, cur, bpS, up, nullptr, nullptr, fU, 0., 0., 0, (inRange && o) ? y[o - 1] : 1, o == 0, gl, gmask, inside);
        if (inRange && !inside) for (int d = gl; d < S; d += G) cur[d] = OP == OP_SUM ? 0. : w_ninf();
        if (OP == OP_SUM) { const int Gc = cell_frame<G> (cur, S, F, gl, inside, bad); if (inRange) { Fprev = F; Gprev = Gc; } }
        else if (bp && inside) {
          unsigned char* row = bp + (size_t) o * S * t.bpBytes;
          if (t.bpBytes == 1) for (int d = gl; d < S; d += G) row[d] = (unsigned char) bpS[d];
          else for (int d = gl; d < S; d += G) reinterpret_cast<uint16_t*> (row)[d] = bpS[d];
        }
        __syncwarp();
        if (o == Lo) { res = cur[S - 1]; Fres = F; }
        slot ^= 1;
      }
      if (gl == 0 && have) {
        if (OP == OP_SUM) { p.result[k] = res > 0. ? log (res) + Fres * LN2 : w_ninf(); p.flag[k] = bad || !(res > 0.) || !(res < 1e300); }
        else p.result[k] = res;
      }
    }
    return;
  }

  // ---- two-dimensional sweep: warp 0 streams the left boundary in, warps 1.. own CPW columns each
  const int WC = (nWarps - 1) * CPW;      // columns per strip
  double* bndBase = p.bnd + (size_t) blockIdx.x * 2 * p.bndRows * t.nLiveIn;
  int2* bndFGBase = p.bndFG + (size_t) blockIdx.x * 2 * p.bndRows;
  double* virtRing = ring + (size_t) (CPW - 1) * R * S;      // the column slot just left of warp 1's first column
  int2* virtFG = fg + (CPW - 1) * R;
  for (;;) {
    if (threadIdx.x == 0) *workSlot = (long long) atomicAdd (p.counter, 1ULL);
    __syncthreads();
    const long long wk = *workSlot;
    __syncthreads();
    if (wk >= p.nWork) break;
    const int64_t k = p.order[wk];
    const uint8_t* x = p.b.x + p.b.xOff[k];
    const uint8_t* y = p.b.y + p.b.yOff[k];
    const int64_t Li = p.b.xOff[k + 1] - p.b.xOff[k], Lo = p.b.yOff[k + 1] - p.b.yOff[k];
    EnvD env { nullptr, nullptr };
    if (p.b.envOff && p.b.envOff[k + 1] != p.b.envOff[k]) env = EnvD { p.b.envStart + p.b.envOff[k], p.b.envEnd + p.b.envOff[k] };
    unsigned char* bp = OP == OP_MAX && p.bp ? p.bp + p.bpOff[wk] : nullptr;
    bool bad = false;
    const int64_t nStrips = (Li + WC) / WC;     // ceil ((Li + 1) / WC)
    for (int64_t strip = 0; strip < nStrips; ++strip) {
      const int64_t i0 = strip * WC;
      const int nCols = (int) min ((int64_t) WC, Li + 1 - i0);
      const int col = (warp - 1) * CPW + grp;
      const bool active = warp >= 1 && col < nCols;
      const int64_t i = i0 + col;
      const int a = (active && i > 0) ? x[i - 1] : 1;
      const bool writesBnd = active && col == nCols - 1 && strip + 1 < nStrips;
      const double* bndIn = bndBase + (size_t) ((strip & 1) ^ 1) * p.bndRows * t.nLiveIn;
      double* bndOut = bndBase + (size_t) (strip & 1) * p.bndRows * t.nLiveIn;
      const int2* fgIn = bndFGBase + (size_t) ((strip & 1) ^ 1) * p.bndRows;
      int2* fgOut = bndFGBase + (size_t) (strip & 1) * p.bndRows;
      if (warp == 0 && strip > 0) {      // boundary row 0 -> the slot step 0 reads
        double* dst = virtRing + (size_t) (R - 1) * S;
        for (int q = lane; q < t.nLiveIn; q += 32) dst[T.live[q]] = bndIn[q];
        if (lane == 0 && OP == OP_SUM) virtFG[R - 1] = fgIn[0];
      }
      __syncthreads();
      const int64_t nSteps = Lo + nCols;
      const int firstCol = (warp - 1) * CPW, lastCol = min (firstCol + CPW, nCols) - 1;      // this warp's columns in the strip
      int slot = 0;      // t % R
      for (int64_t ts = 0; ts < nSteps; ++ts) {
        const int prev = slot == 0 ? R - 1 : slot - 1;            // (t-1) % R
        const int prev2 = prev == 0 ? R - 1 : prev - 1;           // (t-2) % R (only read when R == 3)
        if (warp == 0) {
          if (strip > 0 && ts + 1 <= Lo) {      // the virtual column left of the strip "computes" row t+1 at step t
            double* dst = virtRing + (size_t) slot * S;
            const double* srcRow = bndIn + (size_t) (ts + 1) * t.nLiveIn;
            for (int q = lane; q < t.nLiveIn; q += 32) dst[T.live[q]] = srcRow[q];
            if (lane == 0 && OP == OP_SUM) virtFG[slot] = fgIn[ts + 1];
          }
        } else if (lastCol >= firstCol && ts - lastCol <= Lo && ts - firstCol >= 0) {      // some column of this warp has a row to do
          const int64_t o = ts - col;
          const bool inRange = active && o >= 0 && o <= Lo;
          double* cur = myRing + (size_t) slot * S;
          const double* up = (inRange && o > 0) ? myRing + (size_t) prev * S : nullptr;
          const double* left = (inRange && i > 0) ? myRing - (size_t) R * S + (size_t) prev * S : nullptr;
          const double* diag = (inRange && i > 0 && o > 0 && t.hasMatch) ? myRing - (size_t) R * S + (size_t) prev2 * S : nullptr;
          const bool inside = inRange && env.contains (i, o);
          int F = 0;
          double fU = 1., fL = 1., fD = 1.;
          if (OP == OP_SUM) {
            const int2 gU = up ? myFG[prev] : make_int2 (0, W_SENT);
            const int2 gL = left ? myFG[prev - R] : make_int2 (0, W_SENT);
            const int2 gD = diag ? myFG[prev2 - R] : make_int2 (0, W_SENT);
            const int Gm = max (gU.y, max (gL.y, gD.y));
            F = Gm == W_SENT ? 0 : Gm;
            if (gU.y == W_SENT) up = nullptr; else { fU = w_pow2 (gU.x - F); if (F - gU.y > W_SPREAD) bad = true; }
            if (gL.y == W_SENT) left = nullptr; else { fL = w_pow2 (gL.x - F); if (F - gL.y > W_SPREAD) bad = true; }
            if (gD.y == W_SENT) diag = nullptr; else { fD = w_pow2 (gD.x - F); if (F - gD.y > W_SPREAD) bad = true; }
          }
          compute_cell<OP, G> (T, t, cur, bpS, up, left, diag, fU, fL, fD, a, (inRange && o) ? y[o - 1] : 1, i == 0 && o == 0, gl, gmask, inside);
          if (inRange && !inside) for (int d = gl; d < S; d += G) cur[d] = OP == OP_SUM ? 0. : w_ninf();
          if (OP == OP_SUM) {
            const int Gc = cell_frame<G> (cur, S, F, gl, inside, bad);
            if (inRange && gl == 0) { myFG[slot] = make_int2 (F, Gc); if (writesBnd) fgOut[o] = make_int2 (F, Gc); }
          } else if (bp && inside) {
            unsigned char* row = bp + ((size_t) o * (Li + 1) + i) * S * t.bpBytes;
            if (t.bpBytes == 1) for (int d = gl; d < S; d += G) row[d] = (unsigned char) bpS[d];
            else for (int d = gl; d < S; d += G) reinterpret_cast<uint16_t*> (row)[d] = bpS[d];
          }
          __syncwarp();
          if (inRange && writesBnd) { double* dstRow = bndOut + (size_t) o * t.nLiveIn; for (int q = gl; q < t.nLiveIn; q += G) dstRow[q] = cur[T.live[q]]; }
          if (inRange && i == Li && o == Lo && gl == 0) {
            const double res = cur[S - 1];
            if (OP == OP_SUM) { p.result[k] = res > 0. ? log (res) + F * LN2 : w_ninf(); if (!(res > 0.) || !(res < 1e300)) bad = true; }
            else p.result[k] = res;
          }
        }
        __syncthreads();
        slot = slot + 1 == R ? 0 : slot + 1;
      }
    }
    if (OP == OP_SUM && bad && gl == 0) p.flag[k] = 1;      // flag[] is cleared by the host before the launch
  }
}

// DPMatrix::traceBack (dpmatrix.defs.h:82-110) over the stored back-pointers, one thread per pair.
// lenOut only (out == nullptr) or the path written start -> end.
__global__ void wide_traceback_kernel (DevMachine m, DevBatch b, const int64_t* __restrict__ order, int64_t nWork,
                                       const unsigned char* __restrict__ bp, const int64_t* __restrict__ bpOff, int bpBytes, int laneLayout,
                                       const double* __restrict__ score, int64_t* __restrict__ lenOut, int32_t* __restrict__ out,
                                       const int64_t* __restrict__ outOff) {
  const int64_t wk = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (wk >= nWork) return;
  const int64_t k = order[wk];
  const uint8_t* x = b.x + b.xOff[k];
  const uint8_t* y = b.y + b.yOff[k];
  const int64_t Li = b.xOff[k + 1] - b.xOff[k], Lo = b.yOff[k + 1] - b.yOff[k];
  const int S = m.S;
  const unsigned char* base = bp + bpOff[wk];
  const unsigned kb = bpBytes == 1 ? 6 : 14, none = bpBytes == 1 ? 0xffu : 0xffffu;
  int64_t n = 0;
  if (score[k] > __longlong_as_double (0xfff0000000000000LL)) {      // boss.cpp:831
    const int64_t total = out ? lenOut[wk] : 0;
    int64_t i = Li, o = Lo;
    int s = S - 1;
    while (i > 0 || o > 0 || s != 0) {
      // wide engine: [o][i][s] per pair; lane engine (no input sequence): [o][s][read] per task of laneLayout reads
      const size_t cell = laneLayout ? ((size_t) o * S + s) * laneLayout + (size_t) (wk % laneLayout) : ((size_t) o * (Li + 1) + i) * S + s;
      const unsigned v = bpBytes == 1 ? base[cell] : reinterpret_cast<const uint16_t*> (base)[cell];
      if (v == none) break;      // cannot happen on a finite path
      const unsigned kind = v >> kb, idx = v & ((1u << kb) - 1);
      const int a = i ? x[i - 1] : 0, c = o ? y[o - 1] : 0;
      const int64_t ks = (int64_t) s * m.nIn1;
      const int64_t key = kind == T_MATCH ? (ks + a) * m.nOut1 + c : kind == T_DELETE ? (ks + a) * m.nOut1 : kind == T_INSERT ? ks * m.nOut1 + c : ks * m.nOut1;
      const int64_t q = m.inc.off[key] + idx;
      if (out) out[outOff[wk] + total - 1 - n] = m.inc.id[q];
      ++n;
      if (kind == T_MATCH || kind == T_DELETE) --i;
      if (kind == T_MATCH || kind == T_INSERT) --o;
      s = m.inc.other[q];
    }
  }
  if (!out) lenOut[wk] = n;
}

int wide_traceback_launch (mb_machine* m, mb_batch* b, const int64_t* dOrder, int64_t nWork, const unsigned char* dBp, const int64_t* dBpOff,
                           int bpBytes, int laneLayout, const double* dScore, int64_t* dLen, int32_t* dOut, const int64_t* dOutOff) {
  const unsigned tg = (unsigned) ((nWork + 31) / 32);
  wide_traceback_kernel<<<tg, 32, 0, b->stream>>> (m->dev, b->dev, dOrder, nWork, dBp, dBpOff, bpBytes, laneLayout, dScore, dLen, dOut, dOutOff);
  MB_CUDA (cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
struct WHost {
  WideTables t {};
  std::vector<char> blobLin, blobLog;      // identical except for the weights: exp(lw) and lw
  std::vector<int64_t> entPerm;            // table entry n is hInc entry entPerm[n] (-1: padding)
  char* dLin = nullptr;
  char* dLog = nullptr;
  bool linearOk = false;                   // every finite log-weight within +-30 ln 2
  int maxList = 0;
  int numSMs = 148;
  double estInstrPerCell = 0;
};

static WHost* wh (const mb_machine* m) { return static_cast<WHost*> (m->wide); }

template<class T> static uint32_t put_vec (std::vector<char>& blob, const std::vector<T>& v) {
  const size_t at = (blob.size() + 15) & ~(size_t) 15;
  blob.resize (at + std::max<size_t> (v.size(), 1) * sizeof (T), 0);
  if (!v.empty()) memcpy (blob.data() + at, v.data(), v.size() * sizeof (T));
  return (uint32_t) at;
}

bool wide_supported (const mb_machine* m, std::string* why) {
  if (m->S > 16000) { if (why) *why = "wide engine: more than 16000 states"; return false; }
  if (m->T > 100000000) { if (why) *why = "wide engine: too many transitions"; return false; }
  // two columns (rings of 3 cells + the back-pointer stage) must fit in shared memory
  if ((size_t) m->S * 2 * (3 * 8 + 2) + 1024 > 227 * 1024) { if (why) *why = "wide engine: a cell does not fit in shared memory"; return false; }
  return true;
}

// ---- table construction -------------------------------------------------------------------------
struct WList { int dst; int64_t p0, p1; };      // one destination's token-selected source list: hInc entries [p0, p1)

struct WBuilder {
  int G = 32;
  std::vector<WEntry> ent;       // rows of G entries
  std::vector<int64_t> perm;
  size_t rows() const { return ent.size() / (size_t) G; }
};

static int pow2ceil (int v) { int n = 1; while (n < v) n <<= 1; return n; }
static int ilog2 (int v) { int l = 0; while ((1 << l) < v) ++l; return l; }

// One dependency-free set of lists -> rows: long lists cut into 2^k pieces on adjacent lanes
// (combined by shuffles on their last row), the rest dealt longest-first to the least loaded lane.
// Returns the number of rows; the last row carries the sync flag.
static int schedule_lists (const std::vector<WList>& lists, const mb_machine* m, WBuilder& B) {
  if (lists.empty()) return 0;
  const int G = B.G;
  int64_t total = 0;
  for (auto& l: lists) total += l.p1 - l.p0;
  const int share = (int) std::max<int64_t> (3, (total + G - 1) / G);
  struct Placed { int list, lane, row, n, rows; };
  std::vector<Placed> placed;
  std::vector<int> freeRow ((size_t) G, 0);
  std::vector<int> order (lists.size());
  for (size_t j = 0; j < lists.size(); ++j) order[j] = (int) j;
  std::stable_sort (order.begin(), order.end(), [&] (int a, int b) { return lists[a].p1 - lists[a].p0 > lists[b].p1 - lists[b].p0; });
  for (int j: order) {
    const int L = (int) (lists[j].p1 - lists[j].p0);
    int n = 1;
    if (L >= 6 && L > share + share / 2) n = std::min (G, pow2ceil ((L + share - 1) / share));
    const int rows = (L + n - 1) / n;
    int bestLane = 0, bestStart = 1 << 30;
    for (int l0 = 0; l0 + n <= G; l0 += n) {
      int start = 0;
      for (int l = l0; l < l0 + n; ++l) start = std::max (start, freeRow[l]);
      if (start < bestStart) { bestStart = start; bestLane = l0; }
    }
    placed.push_back (Placed { j, bestLane, bestStart, n, rows });
    for (int l = bestLane; l < bestLane + n; ++l) freeRow[l] = bestStart + rows;
  }
  int nRows = 0;
  for (int l = 0; l < G; ++l) nRows = std::max (nRows, freeRow[l]);
  const size_t e0 = B.ent.size();
  WEntry padE; padE.w = 0; padE.z = 0; padE.d = 0;
  B.ent.resize (e0 + (size_t) nRows * G, padE);
  B.perm.resize (e0 + (size_t) nRows * G, -1);
  for (auto& pl: placed) {
    const WList& ls = lists[pl.list];
    const int L = (int) (ls.p1 - ls.p0);
    for (int j = 0; j < pl.n; ++j)
      for (int k = 0; k < pl.rows; ++k) {
        const size_t e = e0 + (size_t) (pl.row + k) * G + pl.lane + j;
        const int n = j * pl.rows + k;
        WEntry& en = B.ent[e];
        if (n < L) { en.z = (uint32_t) m->hInc.other[ls.p0 + n] | ((uint32_t) n << 16); B.perm[e] = ls.p0 + n; }
        else en.z = (uint32_t) 0 | (0x3fffu << 16);      // padding inside a piece: weight 0 / -inf
        if (k == 0) en.z |= W_FIRST;
        en.d = (uint32_t) ls.dst | ((uint32_t) ilog2 (pl.n) << 16);
        if (k == pl.rows - 1) en.d |= W_PEND;
        if (k == pl.rows - 1 && j == 0) { en.z |= W_LAST; en.d |= W_STORE; }
      }
  }
  for (auto& pl: placed)      // after every entry is in place: the reduce row is flagged in all lanes of the group
    if (pl.n > 1) for (int l = 0; l < G; ++l) B.ent[e0 + (size_t) (pl.row + pl.rows - 1) * G + l].d |= W_REDUCE;
  for (int l = 0; l < G; ++l) B.ent[e0 + (size_t) (nRows - 1) * G + l].d |= W_SYNC;
  return nRows;
}

// all tables for lane-group width G; perCell: estimated warp instructions per cell (a warp works on 32/G cells at once)
static void build_tables (const mb_machine* m, int G, WBuilder& B, std::vector<uint32_t>& phM, std::vector<uint32_t>& phD, std::vector<uint32_t>& phI,
                          uint32_t& silRow0, uint32_t& silRow1, std::vector<uint16_t>& live, bool& hasMatch, int& maxList, double& perCell) {
  const int S = m->S, nIn = m->nIn, nOut = m->nOut, nIn1 = nIn + 1, nOut1 = nOut + 1;
  const HostCsr& inc = m->hInc;
  B = WBuilder();
  B.G = G;
  maxList = 0;
  std::vector<char> isLive ((size_t) S, 0);
  auto lists_for = [&] (int a, int c, bool input) {
    std::vector<WList> ls;
    for (int d = 0; d < S; ++d) {
      const int64_t key = ((int64_t) d * nIn1 + a) * nOut1 + c;
      if (inc.off[key] == inc.off[key + 1]) continue;
      ls.push_back (WList { d, inc.off[key], inc.off[key + 1] });
      maxList = std::max<int> (maxList, (int) (inc.off[key + 1] - inc.off[key]));
      if (input) for (int64_t q = inc.off[key]; q < inc.off[key + 1]; ++q) isLive[inc.other[q]] = 1;
    }
    return ls;
  };
  hasMatch = false;
  phM.clear(); phD.clear(); phI.clear();
  for (int a = 1; a <= nIn; ++a) for (int c = 1; c <= nOut; ++c) {
    phM.push_back ((uint32_t) B.rows());
    if (schedule_lists (lists_for (a, c, true), m, B)) hasMatch = true;
  }
  phM.push_back ((uint32_t) B.rows());
  for (int a = 1; a <= nIn; ++a) { phD.push_back ((uint32_t) B.rows()); schedule_lists (lists_for (a, 0, true), m, B); }
  phD.push_back ((uint32_t) B.rows());
  for (int c = 1; c <= nOut; ++c) { phI.push_back ((uint32_t) B.rows()); schedule_lists (lists_for (0, c, false), m, B); }
  phI.push_back ((uint32_t) B.rows());
  const double rowsM = nIn && nOut ? (double) (phM.back() - phM.front()) / ((double) nIn * nOut) : 0;
  const double rowsD = nIn ? (double) (phD.back() - phD.front()) / nIn : 0, rowsI = nOut ? (double) (phI.back() - phI.front()) / nOut : 0;
  silRow0 = (uint32_t) B.rows();
  const int nLevels = (int) m->fwdLevelOff.size() - 1;
  for (int l = 1; l < nLevels; ++l) {      // level 0 has no silent sources
    std::vector<WList> ls;
    for (int n = m->fwdLevelOff[l]; n < m->fwdLevelOff[l + 1]; ++n) {
      const int d = m->fwdLevelStates[n];
      if (d == 0) continue;      // state 0's only possible silent source is its own self-loop, which contributes nothing
      const int64_t key = (int64_t) d * nIn1 * nOut1;
      if (inc.off[key] == inc.off[key + 1]) continue;
      ls.push_back (WList { d, inc.off[key], inc.off[key + 1] });
      maxList = std::max<int> (maxList, (int) (inc.off[key + 1] - inc.off[key]));
    }
    schedule_lists (ls, m, B);
  }
  silRow1 = (uint32_t) B.rows();
  live.clear();
  for (int s = 0; s < S; ++s) if (isLive[s]) live.push_back ((uint16_t) s);
  const double perWarp = 13.0 * ((double) (silRow1 - silRow0) + rowsM + rowsD + rowsI) + 4.0 * std::max (nLevels - 1, 0)
    + 10.0 * ((S + G - 1) / G) + 150;      // rows, level barriers, zero + frame / back-pointer passes, step overhead
  perCell = perWarp / (32 / G);
}

static void wide_fill_weights (const mb_machine* m, WHost* h) {
  WEntry* lin = reinterpret_cast<WEntry*> (h->blobLin.data() + h->t.oEnt);
  WEntry* lg = reinterpret_cast<WEntry*> (h->blobLog.data() + h->t.oEnt);
  bool ok = true;
  const double lim = 30. * 0.6931471805599453;
  for (size_t n = 0; n < h->entPerm.size(); ++n) {
    if (h->entPerm[n] < 0) { lin[n].w = 0.; lg[n].w = -INFINITY; continue; }
    const double lw = m->hInc.lw[h->entPerm[n]];
    lg[n].w = lw;
    lin[n].w = exp (lw);
    if (std::isnan (lw) || (std::isfinite (lw) && fabs (lw) > lim) || lw == INFINITY) ok = false;
  }
  h->linearOk = ok;
}

void wide_destroy (mb_machine* m) {
  WHost* h = wh (m);
  if (!h) return;
  if (h->dLin) cudaFree (h->dLin);
  if (h->dLog) cudaFree (h->dLog);
  delete h;
  m->wide = nullptr;
}

int wide_update_weights (mb_machine* m) {
  WHost* h = wh (m);
  if (!h) return 0;
  wide_fill_weights (m, h);
  const size_t eBytes = std::max<size_t> (h->entPerm.size(), 1) * sizeof (WEntry);
  MB_CUDA (cudaMemcpy (h->dLin + h->t.oEnt, h->blobLin.data() + h->t.oEnt, eBytes, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (h->dLog + h->t.oEnt, h->blobLog.data() + h->t.oEnt, eBytes, cudaMemcpyHostToDevice));
  return 0;
}

int wide_prepare (mb_machine* m) {
  WHost* h = new WHost;
  m->wide = h;
  WBuilder B, best;
  std::vector<uint32_t> phM, phD, phI, bM, bD, bI;
  std::vector<uint16_t> live, bLive;
  uint32_t s0 = 0, s1 = 0, b0 = 0, b1 = 0;
  bool hasMatch = false, bestMatch = false;
  int maxList = 0;
  double bestCost = 1e300, bestInstr = 0;
  int forceG = 0;
  forceG = m->opt.get ("wide_g", 0);
  for (int G: { 32, 16, 8 }) {
    if (forceG && G != forceG) continue;
    double perCell = 0;
    build_tables (m, G, B, phM, phD, phI, s0, s1, live, hasMatch, maxList, perCell);
    // the sweep is latency-bound below ~16 warps per SM: weigh the instruction estimate by the warps that fit
    const size_t tabBytes = B.ent.size() * sizeof (WEntry) + 4096;
    const size_t perWarp = (size_t) (32 / G) * ((hasMatch ? 3 : 2) * ((size_t) m->S * 8 + 8) + (size_t) m->S * 2);
    const size_t kSmem = 227 * 1024;
    const bool tabsFit = tabBytes + 2 * perWarp <= kSmem;      // tables in shared memory when two warps still fit
    const size_t room = tabsFit ? kSmem - tabBytes : kSmem;
    const int warps = (int) std::min<size_t> (17, room / perWarp);
    if (warps < 2 && !(forceG && G == forceG)) continue;
    const double cost = perCell * std::max (1.0, 16.0 / std::max (warps, 1)) * (tabsFit ? 1.0 : 1.5);
    if (cost < bestCost) { bestCost = cost; bestInstr = perCell; best = B; bM = phM; bD = phD; bI = phI; bLive = live; b0 = s0; b1 = s1; bestMatch = hasMatch; }
  }
  if (bestCost >= 1e300) { set_error ("wide engine: a cell does not fit in shared memory"); return 1; }
  if (maxList > 16382) { set_error ("wide engine: a transition list has more than 16382 entries"); return 1; }
  if (best.rows() > 0xfffffff0u) { set_error ("wide engine: tables too large"); return 1; }
  {      // spare row: the sweep keeps one entry in flight
    WEntry padE; padE.w = 0; padE.z = 0; padE.d = 0;
    best.ent.resize (best.ent.size() + best.G, padE);
    best.perm.resize (best.perm.size() + best.G, -1);
  }
  WideTables& t = h->t;
  std::vector<char>& blob = h->blobLin;
  t.oEnt = put_vec (blob, best.ent);
  t.oPhM = put_vec (blob, bM); t.oPhD = put_vec (blob, bD); t.oPhI = put_vec (blob, bI); t.oLive = put_vec (blob, bLive);
  blob.resize ((blob.size() + 15) & ~(size_t) 15, 0);
  t.bytes = (uint32_t) blob.size();
  t.silRow0 = b0; t.silRow1 = b1;
  t.S = m->S; t.nIn = m->nIn; t.nOut = m->nOut; t.hasMatch = bestMatch ? 1 : 0;
  t.nLiveIn = (int32_t) bLive.size(); t.bpBytes = maxList <= 63 ? 1 : 2; t.G = best.G;
  h->maxList = maxList;
  h->estInstrPerCell = bestInstr;
  h->entPerm = best.perm;
  h->blobLog = h->blobLin;
  wide_fill_weights (m, h);
  MB_CUDA (cudaSetDevice (m->device));
  MB_CUDA (cudaMalloc (&h->dLin, t.bytes));
  MB_CUDA (cudaMalloc (&h->dLog, t.bytes));
  MB_CUDA (cudaMemcpy (h->dLin, h->blobLin.data(), t.bytes, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (h->dLog, h->blobLog.data(), t.bytes, cudaMemcpyHostToDevice));
  MB_CUDA (cudaDeviceGetAttribute (&h->numSMs, cudaDevAttrMultiProcessorCount, m->device));
  if (m->opt.get ("verbose", 0))
    fprintf (stderr, "wide engine: S=%d G=%d rows=%zu (silent %u) tables=%u bytes, est. %.0f warp-instructions per cell, live-in %d, bp %d bytes\n",
             m->S, best.G, best.rows(), b1 - b0, t.bytes, bestInstr, t.nLiveIn, t.bpBytes);
  return 0;
}

// launch shape: column warps per CTA (W), ring depth, where the tables live, CTAs per SM
struct WShape { int W = 0, R = 2, tabInSmem = 0, ctasPerSM = 0; size_t smem = 0; bool oneD = false; const void* fn = nullptr; };

template<int OP> static const void* kernel_for (int G, bool tabs) {
  if (G == 32) return tabs ? (const void*) wide_kernel<OP, 32, true> : (const void*) wide_kernel<OP, 32, false>;
  if (G == 16) return tabs ? (const void*) wide_kernel<OP, 16, true> : (const void*) wide_kernel<OP, 16, false>;
  return tabs ? (const void*) wide_kernel<OP, 8, true> : (const void*) wide_kernel<OP, 8, false>;
}

template<int OP>
static int choose_shape (const WHost* h, bool oneD, int forceW, WShape& best) {
  const WideTables& t = h->t;
  const int R = t.hasMatch ? 3 : 2, CPW = 32 / t.G;
  const size_t kMaxSmem = 227 * 1024;
  double bestScore = -1;
  static const int cand[] = { 16, 12, 8, 6, 4, 3, 2, 1, 0 };
  for (int tabIn = 1; tabIn >= 0; --tabIn) {
    const void* fn = kernel_for<OP> (t.G, tabIn != 0);
    MB_CUDA (cudaFuncSetAttribute (fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) kMaxSmem));
    for (int W: cand) {
      if (forceW && W != forceW) continue;
      if (W == 0 && !oneD) continue;      // the 2-D sweep needs the loader warp and at least one column warp
      const int nWarps = W + 1, nSlots = nWarps * CPW;
      const size_t smem = (tabIn ? ((size_t) t.bytes + 15) & ~(size_t) 15 : 0) + (size_t) nSlots * R * t.S * 8 + (size_t) nSlots * R * 8
        + (OP == OP_MAX ? (size_t) nSlots * t.S * 2 : 0) + 32;
      if (smem > kMaxSmem) continue;
      int ctas = 0;
      MB_CUDA (cudaOccupancyMaxActiveBlocksPerMultiprocessor (&ctas, fn, nWarps * 32, smem));
      if (ctas < 1) continue;
      const double score = (double) (oneD ? nWarps : W) * ctas * (tabIn ? 1.0 : 0.4);
      if (score > bestScore) { bestScore = score; best.W = W; best.R = R; best.tabInSmem = tabIn; best.ctasPerSM = ctas; best.smem = smem; best.oneD = oneD; best.fn = fn; }
    }
  }
  if (bestScore < 0) { set_error ("wide engine: no launch shape fits in shared memory"); return 1; }
  return 0;
}


static std::vector<int64_t> cost_order (const mb_batch* b, const std::vector<int64_t>* subset) {
  std::vector<int64_t> order;
  if (subset) order = *subset;
  else { order.resize ((size_t) b->nPairs); for (int64_t k = 0; k < b->nPairs; ++k) order[k] = k; }
  auto cost = [&] (int64_t k) { return (double) (b->xOff[k + 1] - b->xOff[k] + 1) * (double) (b->yOff[k + 1] - b->yOff[k] + 1); };
  std::stable_sort (order.begin(), order.end(), [&] (int64_t a, int64_t c) { return cost (a) > cost (c); });
  return order;
}

// one launch of wide_kernel<OP> over `order`; bp / bpOff only for OP_MAX with traceback
template<int OP>
static int wide_launch (mb_machine* m, mb_batch* b, const std::vector<int64_t>& order, double* dResult, int32_t* dFlag,
                        unsigned char* dBp, const int64_t* dBpOff) {
  WHost* h = wh (m);
  bool oneD = true;
  int64_t maxLo = 0;
  for (int64_t k: order) { if (b->xOff[k + 1] != b->xOff[k]) oneD = false; maxLo = std::max (maxLo, b->yOff[k + 1] - b->yOff[k]); }
  WShape sh;
  if (choose_shape<OP> (h, oneD, m->opt.get ("wide_w", 0), sh)) return 1;
  const int nWarps = sh.W + 1, CPW = 32 / h->t.G;
  const int64_t nWork = (int64_t) order.size();
  const int64_t wantCtas = oneD ? (nWork + nWarps * CPW - 1) / (nWarps * CPW) : nWork;
  const int grid = (int) std::max<int64_t> (1, std::min<int64_t> (wantCtas, (int64_t) sh.ctasPerSM * h->numSMs));
  DevBuf dOrder, dCounter, dBnd, dBndFG;
  if (dOrder.alloc (order.size() * 8) || dCounter.alloc (8)) return 1;
  MB_CUDA (cudaMemcpyAsync (dOrder.p, order.data(), order.size() * 8, cudaMemcpyHostToDevice, b->stream));
  MB_CUDA (cudaMemsetAsync (dCounter.p, 0, 8, b->stream));
  const int64_t bndRows = maxLo + 1;
  if (!oneD) {
    if (dBnd.alloc ((size_t) grid * 2 * bndRows * std::max (h->t.nLiveIn, 1) * 8) || dBndFG.alloc ((size_t) grid * 2 * bndRows * 8)) return 1;
  }
  WParams p {};
  p.t = h->t;
  p.blob = OP == OP_SUM ? h->dLin : h->dLog;
  p.W = sh.W; p.R = sh.R; p.oneD = oneD ? 1 : 0;
  p.b = b->dev;
  p.order = dOrder.as<int64_t>(); p.nWork = nWork; p.counter = dCounter.as<unsigned long long>();
  p.result = dResult; p.flag = dFlag;
  p.bnd = dBnd.as<double>(); p.bndFG = dBndFG.as<int2>(); p.bndRows = bndRows;
  p.bp = dBp; p.bpOff = dBpOff;
  void* args[] = { &p };
  MB_CUDA (cudaLaunchKernel (sh.fn, dim3 ((unsigned) grid), dim3 ((unsigned) (nWarps * 32)), args, sh.smem, b->stream));
  MB_CUDA (cudaGetLastError());
  MB_CUDA (cudaStreamSynchronize (b->stream));      // the scratch buffers above die with this scope
  return 0;
}

// the log-domain sweep over a subset of the batch, results into dResult[pair] (device): where the big engine sends the pairs it flags
int wide_forward_log_subset (mb_machine* m, mb_batch* b, const std::vector<int64_t>& pairs, double* dResult) {
  if (!m->wide) { set_error ("wide engine not prepared for this machine"); return 1; }
  DevBuf dFlag;
  if (dFlag.alloc ((size_t) b->nPairs * 4)) return 1;
  return wide_launch<OP_LSE> (m, b, cost_order (b, &pairs), dResult, dFlag.as<int32_t>(), nullptr, nullptr);
}

int wide_forward (mb_machine* m, mb_batch* b, double* loglike) {
  b->lastRedo = 0;
  if (b->nPairs == 0) return 0;
  WHost* h = wh (m);
  const std::vector<int64_t> order = cost_order (b, nullptr);
  DevBuf dRes, dFlag;
  if (dRes.alloc ((size_t) b->nPairs * 8) || dFlag.alloc ((size_t) b->nPairs * 4)) return 1;
  MB_CUDA (cudaMemsetAsync (dFlag.p, 0, (size_t) b->nPairs * 4, b->stream));
  if (timing_begin (b)) return 1;
  int64_t launches = 1;
  if (h->linearOk) { if (wide_launch<OP_SUM> (m, b, order, dRes.as<double>(), dFlag.as<int32_t>(), nullptr, nullptr)) return 1; }
  else { if (wide_launch<OP_LSE> (m, b, order, dRes.as<double>(), dFlag.as<int32_t>(), nullptr, nullptr)) return 1; }
  if (h->linearOk) {
    // pairs whose dynamic range the scaled sweep could not hold (or that came out as -inf) go through the log-domain sweep
    std::vector<int32_t> flag ((size_t) b->nPairs);
    MB_CUDA (cudaMemcpy (flag.data(), dFlag.p, flag.size() * 4, cudaMemcpyDeviceToHost));
    std::vector<int64_t> redo;
    for (int64_t k = 0; k < b->nPairs; ++k) if (flag[k]) redo.push_back (k);
    if (!redo.empty()) {
      if (wide_launch<OP_LSE> (m, b, cost_order (b, &redo), dRes.as<double>(), dFlag.as<int32_t>(), nullptr, nullptr)) return 1;
      ++launches;
    }
    b->lastRedo = (int64_t) redo.size();
  }
  if (timing_end (b, launches)) return 1;
  MB_CUDA (cudaMemcpy (loglike, dRes.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  return 0;
}

int wide_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen) {
  if (b->nPairs == 0) return 0;
  WHost* h = wh (m);
  const bool trace = pathLen != nullptr;
  const std::vector<int64_t> order = cost_order (b, nullptr);
  DevBuf dRes;
  if (dRes.alloc ((size_t) b->nPairs * 8)) return 1;
  if (!trace) {
    if (timing_begin (b)) return 1;
    if (wide_launch<OP_MAX> (m, b, order, dRes.as<double>(), nullptr, nullptr, nullptr)) return 1;
    if (timing_end (b, 1)) return 1;
    MB_CUDA (cudaMemcpy (score, dRes.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
    return 0;
  }
  // chunks of pairs whose back-pointers ((Li+1)(Lo+1) S bytes or half-words) fit in free memory
  size_t freeB = 0, totalB = 0;
  MB_CUDA (cudaMemGetInfo (&freeB, &totalB));
  const double budget = 0.75 * (double) freeB;
  int64_t launches = 0;
  double ms = 0;
  for (size_t c0 = 0; c0 < order.size();) {
    std::vector<int64_t> chunk, bpOff;
    double bytes = 0;
    size_t c1 = c0;
    for (; c1 < order.size(); ++c1) {
      const int64_t k = order[c1];
      const double need = (double) (b->xOff[k + 1] - b->xOff[k] + 1) * (double) (b->yOff[k + 1] - b->yOff[k] + 1) * m->S * h->t.bpBytes;
      if (need > budget) { set_error ("pair " + std::to_string (k) + " needs more device memory for its back-pointers than is free (" + std::to_string (need) + " bytes)"); return 1; }
      if (!chunk.empty() && bytes + need > budget) break;
      chunk.push_back (k);
      bpOff.push_back ((int64_t) bytes);
      bytes += (need + 15) - fmod (need + 15, 16);
    }
    c0 = c1;
    DevBuf dBp, dBpOff, dOrder, dLen, dOutOff;
    if (dBp.alloc ((size_t) bytes) || dBpOff.alloc (bpOff.size() * 8) || dOrder.alloc (chunk.size() * 8) || dLen.alloc (chunk.size() * 8)
        || dOutOff.alloc (chunk.size() * 8)) return 1;
    MB_CUDA (cudaMemcpyAsync (dBpOff.p, bpOff.data(), bpOff.size() * 8, cudaMemcpyHostToDevice, b->stream));
    MB_CUDA (cudaMemcpyAsync (dOrder.p, chunk.data(), chunk.size() * 8, cudaMemcpyHostToDevice, b->stream));
    if (timing_begin (b)) return 1;
    if (wide_launch<OP_MAX> (m, b, chunk, dRes.as<double>(), nullptr, dBp.as<unsigned char>(), dBpOff.as<int64_t>())) return 1;
    const int64_t nWork = (int64_t) chunk.size();
    const unsigned tg = (unsigned) ((nWork + 31) / 32);
    wide_traceback_kernel<<<tg, 32, 0, b->stream>>> (m->dev, b->dev, dOrder.as<int64_t>(), nWork, dBp.as<unsigned char>(), dBpOff.as<int64_t>(), h->t.bpBytes, 0,
                                                      dRes.as<double>(), dLen.as<int64_t>(), nullptr, nullptr);
    MB_CUDA (cudaGetLastError());
    if (paths_place (b, b->viterbiPaths, chunk.data(), nWork, dLen.as<int64_t>(), dOutOff.as<int64_t>())) return 1;
    wide_traceback_kernel<<<tg, 32, 0, b->stream>>> (m->dev, b->dev, dOrder.as<int64_t>(), nWork, dBp.as<unsigned char>(), dBpOff.as<int64_t>(), h->t.bpBytes, 0,
                                                      dRes.as<double>(), dLen.as<int64_t>(), b->viterbiPaths.dPaths, dOutOff.as<int64_t>());
    MB_CUDA (cudaGetLastError());
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
