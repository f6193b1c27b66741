// mb_generic.cu -- the generic engine: anti-diagonal wavefront Forward / Backward / Viterbi / counts
// over the token-indexed CSR machine.  Works for any machine size (it is what runs the large
// composed machines, SURVEY.md section 8 configs 4-5) and is the reference-order engine: every
// cell-state is accumulated by one thread in the reference's candidate order (match, delete,
// insert, silent; each by ascending source state then transition index, src/dpmatrix.h:106-115),
// so its values differ from the reference's only through the log-sum-exp table.
//
// One CTA per sequence pair.  Cells on anti-diagonal d = inPos + outPos are independent; within a
// cell, states are swept in silent-dependency levels (a level's states have no silent transitions
// among them), with a CTA barrier between levels.
//
//   reference                                   here
//   MappedForwardMatrix::fill  forward.defs.h:22-49   fill_kernel<OP_SUM, false>
//   ViterbiMatrix::fill        viterbi.cpp:18-43      fill_kernel<OP_MAX, false>
//   BackwardMatrix::fill       backward.cpp:18-46     fill_kernel<OP_SUM, true>
//   DPMatrix::traceBack        dpmatrix.defs.h:82-110 traceback_kernel
//   ForwardMatrix::samplePath  forward.cpp:17-23      sample_kernel
//   BackwardMatrix::getCounts  backward.cpp:62-87     counts_kernel
//   postTransQueue / traceFrom backward.cpp:52-56,89-108  posterior decoding over stored Forward and Backward matrices:
//                                                     mea_fill_kernel (the MEA DP), mea_traceback_kernel (its path and each
//                                                     step's posterior), path_post_kernel (the posterior of each step of a given path)
#include <algorithm>
#include <cmath>
#include <cstdio>

#include "mb_internal.h"

namespace mb {

__device__ __forceinline__ double neg_inf() { return __longlong_as_double (0xfff0000000000000LL); }

// log(exp(a)+exp(b)); exact softplus truncated like the reference's table (logsumexp.h:48-90)
__device__ __forceinline__ double lse2 (double a, double b) {
  const double mx = fmax (a, b), mn = fmin (a, b);
  const double d = mx - mn;               // NaN when both are -inf, +inf when one is
  if (!(d < MB_LSE_CUTOFF)) return mx;
  return mx + log1p (exp (-d));
}

enum { OP_SUM = 0, OP_MAX = 1 };

// Cell storage: full = the reference's [outPos][inPos][state] order (dpmatrix.h:38-40,89-95);
// rolling = three anti-diagonals, indexed by inPos.
struct Cells {
  double* base;
  int64_t Li;
  int32_t S;
  int32_t rolling;
  __device__ __forceinline__ double* at (int64_t i, int64_t o) const {
    return rolling ? base + (((i + o) % 3) * (Li + 1) + i) * S : base + (o * (Li + 1) + i) * S;
  }
};

// Envelope of one pair (null rows = full matrix).
struct Env {
  const int64_t* start;
  const int64_t* end;
  __device__ __forceinline__ bool contains (int64_t i, int64_t o) const { return !start || (i >= start[o] && i < end[o]); }
};
__device__ __forceinline__ Env pair_env (const DevBatch& b, int64_t k) {
  if (!b.envOff || b.envOff[k + 1] == b.envOff[k]) return Env { nullptr, nullptr };
  return Env { b.envStart + b.envOff[k], b.envEnd + b.envOff[k] };
}

template<int OP>
__device__ __forceinline__ double accumulate (double acc, const DevCsr& c, int64_t key, const double* cell) {
  for (int64_t p = c.off[key], e = c.off[key + 1]; p < e; ++p) {
    const double t = cell[c.other[p]] + c.lw[p];
    acc = OP == OP_SUM ? lse2 (acc, t) : (acc < t ? t : acc);
  }
  return acc;
}

// grid: one CTA per pair in `pairs`; ws + wsOff[blockIdx.x] is that pair's cell storage.
template<int OP, bool BACKWARD>
__global__ void __launch_bounds__(256) fill_kernel (DevMachine m, DevBatch b, const int64_t* __restrict__ pairs,
                                                    const int64_t* __restrict__ wsOff, double* __restrict__ ws, int rolling,
                                                    double* __restrict__ result) {
  const int64_t k = pairs[blockIdx.x];
  const uint8_t* x = b.x + b.xOff[k];
  const uint8_t* y = b.y + b.yOff[k];
  const int64_t Li = b.xOff[k + 1] - b.xOff[k], Lo = b.yOff[k + 1] - b.yOff[k];
  const int S = m.S;
  const Cells C = { ws + wsOff[blockIdx.x], Li, S, rolling };
  const int nLevels = BACKWARD ? m.nBwdLevels : m.nFwdLevels;
  const int32_t* levelOff = BACKWARD ? m.bwdLevelOff : m.fwdLevelOff;
  const int32_t* levelStates = BACKWARD ? m.bwdLevelStates : m.fwdLevelStates;
  const DevCsr& csr = BACKWARD ? m.out : m.inc;
  const double ninf = neg_inf();
  const Env env = pair_env (b, k);

  for (int64_t step = 0; step <= Li + Lo; ++step) {
    const int64_t d = BACKWARD ? Li + Lo - step : step;
    const int64_t lo = d > Lo ? d - Lo : 0, hi = d < Li ? d : Li;
    const int64_t nc = hi - lo + 1;
    for (int l = 0; l < nLevels; ++l) {
      const int l0 = levelOff[l], ns = levelOff[l + 1] - l0;
      for (int64_t item = threadIdx.x; item < nc * ns; item += blockDim.x) {
        const int64_t i = lo + item / ns, o = d - i;
        const int s = levelStates[l0 + (int) (item % ns)];
        double* cur = C.at (i, o);
        double acc;
        // cells outside the envelope are never filled and read as -inf (dpmatrix.h:142-144, dpmatrix.defs.h:36)
        if (!env.contains (i, o)) { cur[s] = ninf; continue; }
        if (!BACKWARD) {
          // forward.defs.h:36-45 / viterbi.cpp:30-39
          const int a = i ? x[i - 1] : 0, c = o ? y[o - 1] : 0;
          acc = (i || o || s) ? ninf : 0.;
          const int64_t ks = (int64_t) s * m.nIn1;
          if (i && o) acc = accumulate<OP> (acc, csr, (ks + a) * m.nOut1 + c, C.at (i - 1, o - 1));
          if (i) acc = accumulate<OP> (acc, csr, (ks + a) * m.nOut1, C.at (i - 1, o));
          if (o) acc = accumulate<OP> (acc, csr, ks * m.nOut1 + c, C.at (i, o - 1));
          acc = accumulate<OP> (acc, csr, ks * m.nOut1, cur);
        } else {
          // backward.cpp:32-41
          const bool endI = (i == Li), endO = (o == Lo);
          const int a = endI ? 0 : x[i], c = endO ? 0 : y[o];
          acc = (endI && endO && s == S - 1) ? 0. : ninf;
          const int64_t ks = (int64_t) s * m.nIn1;
          if (!endI && !endO) acc = accumulate<OP> (acc, csr, (ks + a) * m.nOut1 + c, C.at (i + 1, o + 1));
          if (!endI) acc = accumulate<OP> (acc, csr, (ks + a) * m.nOut1, C.at (i + 1, o));
          if (!endO) acc = accumulate<OP> (acc, csr, ks * m.nOut1 + c, C.at (i, o + 1));
          acc = accumulate<OP> (acc, csr, ks * m.nOut1, cur);
        }
        cur[s] = acc;
      }
      __syncthreads();
    }
  }
  if (threadIdx.x == 0)
    result[k] = BACKWARD ? (env.contains (0, 0) ? C.at (0, 0)[0] : ninf) : (env.contains (Li, Lo) ? C.at (Li, Lo)[S - 1] : ninf);
}

// DPMatrix::traceBack (dpmatrix.defs.h:82-110) over a stored Viterbi matrix, one thread per pair.
// Candidates are rebuilt per step in the reference's order and the FIRST maximum wins
// (std::max_element, dpmatrix.defs.h:171-174).  With out == nullptr only the length is computed;
// otherwise the path is written start -> end into out[outOff[blockIdx.x] ..).
__global__ void traceback_kernel (DevMachine m, DevBatch b, const int64_t* __restrict__ pairs, const int64_t* __restrict__ wsOff,
                                  const double* __restrict__ ws, const double* __restrict__ score,
                                  int64_t* __restrict__ lenOut, int32_t* __restrict__ out, const int64_t* __restrict__ outOff) {
  const int64_t slot = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= b.nPairs) return;   // nPairs here = number of pairs in this chunk
  const int64_t k = pairs[slot];
  const uint8_t* x = b.x + b.xOff[k];
  const uint8_t* y = b.y + b.yOff[k];
  const int64_t Li = b.xOff[k + 1] - b.xOff[k], Lo = b.yOff[k + 1] - b.yOff[k];
  const int S = m.S;
  const Cells C = { const_cast<double*> (ws) + wsOff[slot], Li, S, 0 };
  int64_t n = 0;
  if (score[k] > neg_inf()) {    // boss.cpp:831: only finite scores are traced
    const int64_t total = out ? lenOut[slot] : 0;
    int64_t i = Li, o = Lo;
    int s = S - 1;
    while (i > 0 || o > 0 || s != 0) {
      const int a = i ? x[i - 1] : 0, c = o ? y[o - 1] : 0;
      const int64_t ks = (int64_t) s * m.nIn1;
      double best = 0;
      int64_t bestP = -1;
      int bestType = 0;
      auto scan = [&] (int64_t key, const double* cell, int type) {
        for (int64_t p = m.inc.off[key], e = m.inc.off[key + 1]; p < e; ++p) {
          const double t = cell[m.inc.other[p]] + m.inc.lw[p];
          if (bestP < 0 || best < t) { best = t; bestP = p; bestType = type; }
        }
      };
      if (i && o) scan ((ks + a) * m.nOut1 + c, C.at (i - 1, o - 1), T_MATCH);
      if (i) scan ((ks + a) * m.nOut1, C.at (i - 1, o), T_DELETE);
      if (o) scan (ks * m.nOut1 + c, C.at (i, o - 1), T_INSERT);
      scan (ks * m.nOut1, C.at (i, o), T_SILENT);
      if (bestP < 0) break;   // cannot happen for a finite score
      if (out) out[outOff[slot] + total - 1 - n] = m.inc.id[bestP];
      ++n;
      if (bestType == T_MATCH || bestType == T_DELETE) --i;
      if (bestType == T_MATCH || bestType == T_INSERT) --o;
      s = m.inc.other[bestP];
    }
  }
  if (!out) lenOut[slot] = n;
}

// Philox4x32-10 (Salmon, Moraes, Dror and Shaw, SC'11), as Random123's philox4x32 with 10 rounds: the counter-based generator
// of sample_kernel.  Written out here, not taken from cuRAND, so that a host replay reproduces every draw bit for bit.
__device__ __forceinline__ uint4 philox4x32_10 (uint4 c, uint2 key) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r) { key.x += 0x9E3779B9u; key.y += 0xBB67AE85u; }
    const uint32_t lo0 = 0xD2511F53u * c.x, hi0 = __umulhi (0xD2511F53u, c.x);
    const uint32_t lo1 = 0xCD9E8D57u * c.z, hi1 = __umulhi (0xCD9E8D57u, c.z);
    c = make_uint4 (hi1 ^ c.y ^ key.x, lo1, hi0 ^ c.w ^ key.y, lo0);
  }
  return c;
}

// ForwardMatrix::samplePath (forward.cpp:17-23, dpmatrix.defs.h:176-186) over stored Forward matrices: one thread per
// (pair of the chunk, sample), thread q = slot * nSamples + j.  Each step rebuilds the candidates as traceback_kernel does
// (match, delete, insert, silent; each by source state then transition index), weighs candidate n by
// w_n = exp (v_n - max v), v_n = F(previous cell)[source] + log-weight (the reference's exp (v_n) underflows to all zeros once
// Forward values fall below about -745), and takes the first candidate with w_n > 0 whose running sum exceeds u * sum w, or
// failing that, after rounding, the last one with w_n > 0.  u is drawn with Philox4x32-10, key = seed, counter = (step, j, k):
// a path depends only on (seed, pair index k, sample j) and the pair, never on the chunking.  With out == nullptr only the
// length is computed; otherwise path q is written start -> end into out[outOff[q] ..).
__global__ void sample_kernel (DevMachine m, DevBatch b, const int64_t* __restrict__ pairs, int64_t nSlots, int32_t nSamples, uint64_t seed,
                               const int64_t* __restrict__ wsOff, const double* __restrict__ ws, const double* __restrict__ loglike,
                               int64_t* __restrict__ lenOut, int32_t* __restrict__ out, const int64_t* __restrict__ outOff) {
  const int64_t q = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nSlots * nSamples) return;
  const int64_t slot = q / nSamples;
  const uint32_t j = (uint32_t) (q - slot * nSamples);
  const int64_t k = pairs[slot];
  const uint8_t* x = b.x + b.xOff[k];
  const uint8_t* y = b.y + b.yOff[k];
  const int64_t Li = b.xOff[k + 1] - b.xOff[k], Lo = b.yOff[k + 1] - b.yOff[k];
  const int S = m.S;
  const Cells C = { const_cast<double*> (ws) + wsOff[slot], Li, S, 0 };
  const uint2 key = make_uint2 ((uint32_t) seed, (uint32_t) (seed >> 32));
  int64_t n = 0;
  if (loglike[k] > neg_inf()) {
    const int64_t total = out ? lenOut[q] : 0;
    int64_t i = Li, o = Lo;
    int s = S - 1;
    while (i > 0 || o > 0 || s != 0) {
      const int a = i ? x[i - 1] : 0, c = o ? y[o - 1] : 0;
      const int64_t ks = (int64_t) s * m.nIn1;
      auto visit = [&] (auto&& f) {      // f (list entry, value, type) over the candidates in order
        auto list = [&] (int64_t listKey, const double* cell, int type) {
          for (int64_t p = m.inc.off[listKey], e = m.inc.off[listKey + 1]; p < e; ++p) f (p, cell[m.inc.other[p]] + m.inc.lw[p], type);
        };
        if (i && o) list ((ks + a) * m.nOut1 + c, C.at (i - 1, o - 1), T_MATCH);
        if (i) list ((ks + a) * m.nOut1, C.at (i - 1, o), T_DELETE);
        if (o) list (ks * m.nOut1 + c, C.at (i, o - 1), T_INSERT);
        list (ks * m.nOut1, C.at (i, o), T_SILENT);
      };
      double mx = neg_inf();
      visit ([&] (int64_t, double v, int) { mx = fmax (mx, v); });
      if (!(mx > neg_inf())) break;   // cannot happen on a path through finite cells
      double norm = 0;
      visit ([&] (int64_t, double v, int) { norm += exp (v - mx); });
      const uint4 r = philox4x32_10 (make_uint4 ((uint32_t) n, j, (uint32_t) k, (uint32_t) ((uint64_t) k >> 32)), key);
      const double thr = (double) (((uint64_t) r.x << 21) | (r.y >> 11)) * 0x1p-53 * norm;
      double run = 0;
      int64_t pick = -1, last = -1;
      int pickType = 0, lastType = 0;
      visit ([&] (int64_t p, double v, int type) {
        if (pick >= 0) return;
        const double w = exp (v - mx);
        if (!(w > 0)) return;
        run += w;
        last = p; lastType = type;
        if (run > thr) { pick = p; pickType = type; }
      });
      if (pick < 0) { pick = last; pickType = lastType; }
      if (out) {
        if (n >= total) break;   // cannot happen: the walk replays the length pass's
        out[outOff[q] + total - 1 - n] = m.inc.id[pick];
      }
      ++n;
      if (pickType == T_MATCH || pickType == T_DELETE) --i;
      if (pickType == T_MATCH || pickType == T_INSERT) --o;
      s = m.inc.other[pick];
    }
  }
  if (!out) lenOut[q] = n;
}

// BackwardMatrix::getCounts (backward.cpp:62-87): count[t] += exp(F(src cell) - ll + w_t + B(dest cell)).
// One CTA per pair; the CTA walks the transitions, each thread sums the cells where the
// transition's labels match the tokens, then a block reduction and one atomic per transition.
// ROWS: the CTA of the chunk's pair blockIdx.x adds into that pair's own row, counts + blockIdx.x * rowStride.
template<bool ROWS>
__global__ void __launch_bounds__(256) counts_kernel (DevMachine m, DevBatch b, const int64_t* __restrict__ pairs,
                                                      const int64_t* __restrict__ wsOff, const double* __restrict__ wsF,
                                                      const double* __restrict__ wsB, const double* __restrict__ backLL,
                                                      double* __restrict__ counts, int64_t rowStride) {
  __shared__ double red[256];
  const int64_t k = pairs[blockIdx.x];
  const double ll = backLL[k];   // backward.cpp:66 uses the Backward log-likelihood
  if (!(ll > neg_inf())) return;
  const uint8_t* x = b.x + b.xOff[k];
  const uint8_t* y = b.y + b.yOff[k];
  const int64_t Li = b.xOff[k + 1] - b.xOff[k], Lo = b.yOff[k + 1] - b.yOff[k];
  const int S = m.S;
  const Cells F = { const_cast<double*> (wsF) + wsOff[blockIdx.x], Li, S, 0 }, B = { const_cast<double*> (wsB) + wsOff[blockIdx.x], Li, S, 0 };
  const int64_t nKeys = (int64_t) S * m.nIn1 * m.nOut1;
  const Env env = pair_env (b, k);
  if (ROWS) counts += (int64_t) blockIdx.x * rowStride;
  for (int64_t key = 0; key < nKeys; ++key) {
    const int64_t p0 = m.out.off[key], p1 = m.out.off[key + 1];
    if (p0 == p1) continue;
    const int c = (int) (key % m.nOut1), a = (int) ((key / m.nOut1) % m.nIn1), s = (int) (key / ((int64_t) m.nOut1 * m.nIn1));
    const int di = a ? 1 : 0, dO = c ? 1 : 0;
    const int64_t ni = Li + 1 - di, no = Lo + 1 - dO;
    for (int64_t p = p0; p < p1; ++p) {
      const int dest = m.out.other[p];
      const double lw = m.out.lw[p];
      double sum = 0;
      for (int64_t cell = threadIdx.x; cell < ni * no; cell += blockDim.x) {
        const int64_t i = cell % ni, o = cell / ni;
        if ((a && x[i] != a) || (c && y[o] != c)) continue;
        if (!env.contains (i, o)) continue;   // getCounts walks the envelope's cells (backward.cpp:70); outside reads are -inf
        sum += exp ((F.at (i, o)[s] - ll) + (B.at (i + di, o + dO)[dest] + lw));
      }
      red[threadIdx.x] = sum;
      __syncthreads();
      for (int w = blockDim.x / 2; w > 0; w >>= 1) {
        if ((int) threadIdx.x < w) red[threadIdx.x] += red[threadIdx.x + w];
        __syncthreads();
      }
      if (threadIdx.x == 0 && red[0] != 0) atomicAdd (&counts[m.out.id[p]], red[0]);
      __syncthreads();
    }
  }
}

// ---------------------------------------------------------------------------------------------
// posterior decoding (definitions: include/machineboss_b200.h, mb_mea)
// ---------------------------------------------------------------------------------------------
// The candidates into state s at cell (i, o), a = x[i-1] (0 at i == 0), c = y[o-1] (0 at o == 0): f (incoming list entry p,
// source inPos, source outPos, tokens consumed) in the reference's order (match, delete, insert, silent; each by source state
// then transition index), as traceback_kernel and sample_kernel walk them.
template<class Fn>
__device__ __forceinline__ void for_each_incoming (const DevMachine& m, int64_t i, int64_t o, int s, int a, int c, Fn&& f) {
  const int64_t ks = (int64_t) s * m.nIn1;
  auto list = [&] (int64_t key, int64_t si, int64_t so, int tokens) {
    for (int64_t p = m.inc.off[key], e = m.inc.off[key + 1]; p < e; ++p) f (p, si, so, tokens);
  };
  if (i && o) list ((ks + a) * m.nOut1 + c, i - 1, o - 1, 2);
  if (i) list ((ks + a) * m.nOut1, i - 1, o, 1);
  if (o) list (ks * m.nOut1 + c, i, o - 1, 1);
  list (ks * m.nOut1, i, o, 0);
}

// A step's posterior gamma = exp ((F - ll) + (B + w)) from f = F(source cell)[src] and bw = B(destination cell)[dst] + w: the
// bracketing of counts_kernel, so that gamma is bit for bit the term it adds.  Returns whether the step is admissible.
__device__ __forceinline__ bool step_post (double f, double ll, double bw, double& gamma) {
  const double e = (f - ll) + bw;
  gamma = exp (e);
  return e > neg_inf();
}

// The MEA DP over a chunk's stored Forward (wsF) and Backward (wsB) matrices, A into wsA: fill_kernel's forward wavefront and
// silent-level sweep, one CTA per pair, cells outside the envelope -inf.  gain[k] = A(Li, Lo)[end state].
__global__ void __launch_bounds__(256) mea_fill_kernel (DevMachine m, DevBatch b, const int64_t* __restrict__ pairs,
                                                        const int64_t* __restrict__ wsOff, const double* __restrict__ wsF,
                                                        const double* __restrict__ wsB, const double* __restrict__ backLL,
                                                        double* __restrict__ wsA, double* __restrict__ gain) {
  const int64_t k = pairs[blockIdx.x];
  const uint8_t* x = b.x + b.xOff[k];
  const uint8_t* y = b.y + b.yOff[k];
  const int64_t Li = b.xOff[k + 1] - b.xOff[k], Lo = b.yOff[k + 1] - b.yOff[k];
  const int S = m.S;
  const Cells F = { const_cast<double*> (wsF) + wsOff[blockIdx.x], Li, S, 0 }, B = { const_cast<double*> (wsB) + wsOff[blockIdx.x], Li, S, 0 },
              A = { wsA + wsOff[blockIdx.x], Li, S, 0 };
  const double ninf = neg_inf(), ll = backLL[k];
  const Env env = pair_env (b, k);
  for (int64_t d = 0; d <= Li + Lo; ++d) {
    const int64_t lo = d > Lo ? d - Lo : 0, hi = d < Li ? d : Li;
    const int64_t nc = hi - lo + 1;
    for (int l = 0; l < m.nFwdLevels; ++l) {
      const int l0 = m.fwdLevelOff[l], ns = m.fwdLevelOff[l + 1] - l0;
      for (int64_t item = threadIdx.x; item < nc * ns; item += blockDim.x) {
        const int64_t i = lo + item / ns, o = d - i;
        const int s = m.fwdLevelStates[l0 + (int) (item % ns)];
        double acc = (i || o || s) ? ninf : 0.;
        const double bs = B.at (i, o)[s];
        if (env.contains (i, o) && ll > ninf && bs > ninf)
          for_each_incoming (m, i, o, s, i ? x[i - 1] : 0, o ? y[o - 1] : 0, [&] (int64_t p, int64_t si, int64_t so, int tokens) {
            const int src = m.inc.other[p];
            double g;
            if (!step_post (F.at (si, so)[src], ll, bs + m.inc.lw[p], g)) return;
            const double v = A.at (si, so)[src] + tokens * g;
            if (acc < v) acc = v;
          });
        A.at (i, o)[s] = env.contains (i, o) ? acc : ninf;
      }
      __syncthreads();
    }
  }
  if (threadIdx.x == 0) gain[k] = env.contains (Li, Lo) ? A.at (Li, Lo)[S - 1] : ninf;
}

// The MEA path over the stored A, F and B matrices, one thread per pair of the chunk: each step rebuilds the candidates with the
// fill's arithmetic and takes the first maximum, as the fill did.  With out == nullptr only the length is computed; otherwise the
// path is written start -> end into out[outOff[slot] ..) and each step's gamma into outPost at the same place.
__global__ void mea_traceback_kernel (DevMachine m, DevBatch b, const int64_t* __restrict__ pairs, int64_t nSlots, const int64_t* __restrict__ wsOff,
                                      const double* __restrict__ wsF, const double* __restrict__ wsB, const double* __restrict__ wsA,
                                      const double* __restrict__ backLL, const double* __restrict__ gain, int64_t* __restrict__ lenOut,
                                      int32_t* __restrict__ out, double* __restrict__ outPost, const int64_t* __restrict__ outOff) {
  const int64_t slot = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= nSlots) return;
  const int64_t k = pairs[slot];
  const uint8_t* x = b.x + b.xOff[k];
  const uint8_t* y = b.y + b.yOff[k];
  const int64_t Li = b.xOff[k + 1] - b.xOff[k], Lo = b.yOff[k + 1] - b.yOff[k];
  const int S = m.S;
  const Cells F = { const_cast<double*> (wsF) + wsOff[slot], Li, S, 0 }, B = { const_cast<double*> (wsB) + wsOff[slot], Li, S, 0 },
              A = { const_cast<double*> (wsA) + wsOff[slot], Li, S, 0 };
  const double ninf = neg_inf(), ll = backLL[k];
  int64_t n = 0;
  if (gain[k] > ninf) {
    const int64_t total = out ? lenOut[slot] : 0;
    int64_t i = Li, o = Lo;
    int s = S - 1;
    while (i > 0 || o > 0 || s != 0) {
      const double bs = B.at (i, o)[s];
      double best = ninf, bestG = 0;
      int64_t bestP = -1, bi = 0, bo = 0;
      for_each_incoming (m, i, o, s, i ? x[i - 1] : 0, o ? y[o - 1] : 0, [&] (int64_t p, int64_t si, int64_t so, int tokens) {
        const int src = m.inc.other[p];
        double g;
        if (!step_post (F.at (si, so)[src], ll, bs + m.inc.lw[p], g)) return;
        const double v = A.at (si, so)[src] + tokens * g;
        if (best < v) { best = v; bestG = g; bestP = p; bi = si; bo = so; }
      });
      if (bestP < 0) break;   // cannot happen for a finite gain
      if (out) {
        if (n >= total) break;   // cannot happen: the walk replays the length pass's
        out[outOff[slot] + total - 1 - n] = m.inc.id[bestP];
        outPost[outOff[slot] + total - 1 - n] = bestG;
      }
      ++n;
      i = bi; o = bo; s = m.inc.other[bestP];
    }
  }
  if (!out) lenOut[slot] = n;
}

// per-path outcome of path_post_kernel (the first check a step fails)
enum { PP_OK = 0, PP_SOURCE, PP_INPUT, PP_OUTPUT, PP_ENVELOPE, PP_END };

// The posterior of each step of given paths, one thread per path of the chunk: path r (pair pairOfPath[r], the chunk's pair
// slotOfPath[r]) is ids[off[r] .. off[r + 1]), its gammas go to post at the same places.  The walk checks each step and records
// the first one that is not a step of the pair (err[r], errStep[r]; PP_END with errStep = length when the path stops early).
__global__ void path_post_kernel (DevMachine m, DevBatch b, const int64_t* __restrict__ chunkPaths, int64_t nChunkPaths,
                                  const int64_t* __restrict__ slotOfPath, const int64_t* __restrict__ pairOfPath,
                                  const int32_t* __restrict__ ids, const int64_t* __restrict__ off, const int64_t* __restrict__ wsOff,
                                  const double* __restrict__ wsF, const double* __restrict__ wsB, const double* __restrict__ backLL,
                                  double* __restrict__ post, int32_t* __restrict__ err, int64_t* __restrict__ errStep) {
  const int64_t q = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= nChunkPaths) return;
  const int64_t r = chunkPaths[q], slot = slotOfPath[r], k = pairOfPath[r];
  const uint8_t* x = b.x + b.xOff[k];
  const uint8_t* y = b.y + b.yOff[k];
  const int64_t Li = b.xOff[k + 1] - b.xOff[k], Lo = b.yOff[k + 1] - b.yOff[k];
  const int S = m.S;
  const Cells F = { const_cast<double*> (wsF) + wsOff[slot], Li, S, 0 }, B = { const_cast<double*> (wsB) + wsOff[slot], Li, S, 0 };
  const double ninf = neg_inf(), ll = backLL[k];
  const Env env = pair_env (b, k);
  int64_t i = 0, o = 0, n = off[r];
  int s = 0, code = PP_OK;
  for (; n < off[r + 1]; ++n) {
    const int t = ids[n], a = m.tIn[t], c = m.tOut[t], dst = m.tDst[t];
    if (m.tSrc[t] != s) { code = PP_SOURCE; break; }
    if (a && (i >= Li || x[i] != a)) { code = PP_INPUT; break; }
    if (c && (o >= Lo || y[o] != c)) { code = PP_OUTPUT; break; }
    const int64_t ni = i + (a ? 1 : 0), no = o + (c ? 1 : 0);
    if (!env.contains (ni, no)) { code = PP_ENVELOPE; break; }
    // a silent transition that does not advance (only possible on state 0) never contributes to the DP (build_csr): gamma 0
    double g = 0;
    if (ll > ninf && (a || c || dst > s)) step_post (F.at (i, o)[s], ll, B.at (ni, no)[dst] + m.tLw[t], g);
    post[n] = g;
    i = ni; o = no; s = dst;
  }
  if (code == PP_OK && !(i == Li && o == Lo && s == S - 1)) code = PP_END;
  err[r] = code;
  errStep[r] = n - off[r];
}

// ---------------------------------------------------------------------------------------------
// host side: chunk the batch so that the cell storage of a chunk fits in free device memory
// ---------------------------------------------------------------------------------------------
struct Chunk {
  std::vector<int64_t> pairs, wsOff;
  int64_t doubles = 0;
};

// rowDoubles: a further buffer of that many doubles per pair of a chunk (per-pair counts), which shares the budget
static int plan_chunks (const mb_batch* b, int S, bool rolling, int copies, std::vector<Chunk>& chunks, int64_t rowDoubles = 0) {
  size_t freeB = 0, totalB = 0;
  MB_CUDA (cudaMemGetInfo (&freeB, &totalB));
  const double budget = 0.80 * (double) freeB / 8.0 / copies;   // doubles per copy
  const double rowShare = (double) rowDoubles / copies;
  Chunk cur;
  for (int64_t k = 0; k < b->nPairs; ++k) {
    const int64_t Li = b->xOff[k + 1] - b->xOff[k], Lo = b->yOff[k + 1] - b->yOff[k];
    const double need = rolling ? 3.0 * (double) (Li + 1) * S : (double) (Li + 1) * (double) (Lo + 1) * S;
    if (need + rowShare > budget) { set_error ("pair " + std::to_string (k) + " needs more device memory than is free (" + std::to_string ((need + rowShare) * 8 * copies) + " bytes)"); return 1; }
    if (!cur.pairs.empty() && ((double) cur.doubles + need + rowShare * (double) (cur.pairs.size() + 1) > budget || cur.pairs.size() >= 65535 * 16)) { chunks.push_back (cur); cur = Chunk(); }
    cur.pairs.push_back (k);
    cur.wsOff.push_back (cur.doubles);
    cur.doubles += (int64_t) need;
  }
  if (!cur.pairs.empty()) chunks.push_back (cur);
  return 0;
}

static int upload (DevBuf& d, const std::vector<int64_t>& v, cudaStream_t st) {
  if (d.alloc (v.size() * 8)) return 1;
  MB_CUDA (cudaMemcpyAsync (d.p, v.data(), v.size() * 8, cudaMemcpyHostToDevice, st));
  return 0;
}

int generic_forward (mb_machine* m, mb_batch* b, double* loglike, bool backward) {
  if (b->nPairs == 0) return 0;
  std::vector<Chunk> chunks;
  if (plan_chunks (b, m->S, true, 1, chunks)) return 1;
  DevBuf dRes;
  if (dRes.alloc ((size_t) b->nPairs * 8)) return 1;
  if (timing_begin (b)) return 1;
  int64_t launches = 0;
  for (auto& ch: chunks) {
    DevBuf dPairs, dOff, dWs;
    if (upload (dPairs, ch.pairs, b->stream) || upload (dOff, ch.wsOff, b->stream) || dWs.alloc ((size_t) ch.doubles * 8)) return 1;
    const unsigned grid = (unsigned) ch.pairs.size();
    if (backward) fill_kernel<OP_SUM, true><<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWs.as<double>(), 1, dRes.as<double>());
    else fill_kernel<OP_SUM, false><<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWs.as<double>(), 1, dRes.as<double>());
    MB_CUDA (cudaGetLastError());
    ++launches;
    MB_CUDA (cudaStreamSynchronize (b->stream));
  }
  if (timing_end (b, launches)) return 1;
  MB_CUDA (cudaMemcpy (loglike, dRes.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  return 0;
}


// DPMatrix::cell (dpmatrix.h:128-146): the whole matrix of one pair, [o][i][s] as the reference stores it
// (state fastest, then input position, then output position), -inf outside the envelope.
int generic_matrix (mb_machine* m, mb_batch* b, int64_t pair, int kind, double* cells) {
  if (pair < 0 || pair >= b->nPairs) { set_error ("mb_matrix: no such pair"); return 1; }
  if (kind < 0 || kind > 2) { set_error ("mb_matrix: kind must be 0 (Forward), 1 (Backward) or 2 (Viterbi)"); return 1; }
  const int64_t Li = b->xOff[pair + 1] - b->xOff[pair], Lo = b->yOff[pair + 1] - b->yOff[pair];
  const size_t n = (size_t) (Li + 1) * (size_t) (Lo + 1) * m->S;
  std::vector<int64_t> one (1, pair), zero (1, 0);
  DevBuf dPairs, dOff, dWs, dRes;
  if (upload (dPairs, one, b->stream) || upload (dOff, zero, b->stream) || dWs.alloc (n * 8) || dRes.alloc ((size_t) b->nPairs * 8)) return 1;
  if (timing_begin (b)) return 1;
  if (kind == 0) fill_kernel<OP_SUM, false><<<1, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWs.as<double>(), 0, dRes.as<double>());
  else if (kind == 1) fill_kernel<OP_SUM, true><<<1, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWs.as<double>(), 0, dRes.as<double>());
  else fill_kernel<OP_MAX, false><<<1, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWs.as<double>(), 0, dRes.as<double>());
  MB_CUDA (cudaGetLastError());
  if (timing_end (b, 1)) return 1;
  MB_CUDA (cudaMemcpy (cells, dWs.p, n * 8, cudaMemcpyDeviceToHost));
  return 0;
}

int generic_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen) {
  if (b->nPairs == 0) return 0;
  const bool trace = pathLen != nullptr;
  std::vector<Chunk> chunks;
  if (plan_chunks (b, m->S, !trace, 1, chunks)) return 1;
  DevBuf dRes;
  if (dRes.alloc ((size_t) b->nPairs * 8)) return 1;
  int64_t launches = 0;
  double ms = 0;
  for (auto& ch: chunks) {
    DevBuf dPairs, dOff, dWs, dLen, dOutOff;
    if (upload (dPairs, ch.pairs, b->stream) || upload (dOff, ch.wsOff, b->stream) || dWs.alloc ((size_t) ch.doubles * 8)) return 1;
    const unsigned grid = (unsigned) ch.pairs.size();
    if (timing_begin (b)) return 1;
    fill_kernel<OP_MAX, false><<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWs.as<double>(), trace ? 0 : 1, dRes.as<double>());
    MB_CUDA (cudaGetLastError());
    ++launches;
    if (trace) {
      DevBatch cb = b->dev;
      cb.nPairs = (int64_t) ch.pairs.size();
      if (dLen.alloc (ch.pairs.size() * 8) || dOutOff.alloc (ch.pairs.size() * 8)) return 1;
      const unsigned tg = (unsigned) ((ch.pairs.size() + 63) / 64);
      traceback_kernel<<<tg, 64, 0, b->stream>>> (m->dev, cb, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWs.as<double>(), dRes.as<double>(), dLen.as<int64_t>(), nullptr, nullptr);
      MB_CUDA (cudaGetLastError());
      if (paths_place (b, b->viterbiPaths, ch.pairs.data(), (int64_t) ch.pairs.size(), dLen.as<int64_t>(), dOutOff.as<int64_t>())) return 1;
      traceback_kernel<<<tg, 64, 0, b->stream>>> (m->dev, cb, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWs.as<double>(), dRes.as<double>(), dLen.as<int64_t>(), b->viterbiPaths.dPaths, dOutOff.as<int64_t>());
      MB_CUDA (cudaGetLastError());
      launches += 2;
    }
    if (timing_end (b, launches)) return 1;
    ms += b->lastMs;
  }
  b->lastMs = ms;
  b->lastLaunches = launches;
  MB_CUDA (cudaMemcpy (score, dRes.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  return 0;
}

// Per chunk: the full-storage Forward fill, the sampler's length pass, placement, the id pass (generic_viterbi's scheme).
int generic_sample_paths (mb_machine* m, mb_batch* b, int32_t nSamples, uint64_t seed, double* loglike) {
  b->lastMs = 0;
  b->lastLaunches = 0;
  if (b->nPairs == 0) return 0;
  std::vector<Chunk> chunks;
  if (plan_chunks (b, m->S, false, 1, chunks)) return 1;
  DevBuf dRes;
  if (dRes.alloc ((size_t) b->nPairs * 8)) return 1;
  int64_t launches = 0;
  double ms = 0;
  for (auto& ch: chunks) {
    const int64_t nSlots = (int64_t) ch.pairs.size(), nPaths = nSlots * nSamples;
    std::vector<int64_t> rows ((size_t) nPaths);      // path q of the chunk is path k * nSamples + j of the batch
    for (int64_t q = 0; q < nPaths; ++q) rows[q] = ch.pairs[q / nSamples] * nSamples + q % nSamples;
    DevBuf dPairs, dOff, dWs, dLen, dOutOff;
    if (upload (dPairs, ch.pairs, b->stream) || upload (dOff, ch.wsOff, b->stream) || dWs.alloc ((size_t) ch.doubles * 8)
        || dLen.alloc ((size_t) nPaths * 8) || dOutOff.alloc ((size_t) nPaths * 8)) return 1;
    if (timing_begin (b)) return 1;
    fill_kernel<OP_SUM, false><<<(unsigned) nSlots, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWs.as<double>(), 0, dRes.as<double>());
    MB_CUDA (cudaGetLastError());
    const unsigned sg = (unsigned) ((nPaths + 63) / 64);
    sample_kernel<<<sg, 64, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), nSlots, nSamples, seed, dOff.as<int64_t>(), dWs.as<double>(), dRes.as<double>(),
                                             dLen.as<int64_t>(), nullptr, nullptr);
    MB_CUDA (cudaGetLastError());
    if (paths_place (b, b->sampledPaths, rows.data(), nPaths, dLen.as<int64_t>(), dOutOff.as<int64_t>())) return 1;
    sample_kernel<<<sg, 64, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), nSlots, nSamples, seed, dOff.as<int64_t>(), dWs.as<double>(), dRes.as<double>(),
                                             dLen.as<int64_t>(), b->sampledPaths.dPaths, dOutOff.as<int64_t>());
    MB_CUDA (cudaGetLastError());
    launches += 3;
    if (timing_end (b, launches)) return 1;
    ms += b->lastMs;
  }
  b->lastMs = ms;
  b->lastLaunches = launches;
  if (loglike) MB_CUDA (cudaMemcpy (loglike, dRes.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  return 0;
}

int generic_counts (mb_machine* m, mb_batch* b, double* counts, double* loglike, double* rows) {
  if (b->nPairs == 0) { if (counts) for (int64_t t = 0; t < m->T; ++t) counts[t] = 0; return 0; }
  std::vector<Chunk> chunks;
  if (plan_chunks (b, m->S, false, 2, chunks, rows ? m->T : 0)) return 1;
  size_t maxPairs = 0;
  for (auto& ch: chunks) maxPairs = std::max (maxPairs, ch.pairs.size());
  const size_t T = (size_t) std::max<int64_t> (m->T, 1), countDoubles = rows ? maxPairs * T : T;      // rows: [chunk pairs][nTrans]
  DevBuf dF, dB, dCounts;
  if (dF.alloc ((size_t) b->nPairs * 8) || dB.alloc ((size_t) b->nPairs * 8) || dCounts.alloc (countDoubles * 8)) return 1;
  MB_CUDA (cudaMemsetAsync (dCounts.p, 0, T * 8, b->stream));
  int64_t launches = 0;
  double ms = 0;
  for (auto& ch: chunks) {
    DevBuf dPairs, dOff, dWsF, dWsB;
    if (upload (dPairs, ch.pairs, b->stream) || upload (dOff, ch.wsOff, b->stream) || dWsF.alloc ((size_t) ch.doubles * 8) || dWsB.alloc ((size_t) ch.doubles * 8)) return 1;
    const unsigned grid = (unsigned) ch.pairs.size();
    if (timing_begin (b)) return 1;
    if (rows) MB_CUDA (cudaMemsetAsync (dCounts.p, 0, ch.pairs.size() * T * 8, b->stream));
    fill_kernel<OP_SUM, false><<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWsF.as<double>(), 0, dF.as<double>());
    fill_kernel<OP_SUM, true><<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWsB.as<double>(), 0, dB.as<double>());
    if (rows)
      counts_kernel<true><<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWsF.as<double>(), dWsB.as<double>(), dB.as<double>(), dCounts.as<double>(), (int64_t) T);
    else if (counts)
      counts_kernel<false><<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWsF.as<double>(), dWsB.as<double>(), dB.as<double>(), dCounts.as<double>(), 0);
    MB_CUDA (cudaGetLastError());
    launches += counts || rows ? 3 : 2;
    if (timing_end (b, launches)) return 1;
    ms += b->lastMs;
    // a chunk's pairs are consecutive in the batch, so its rows are one block of the caller's array
    if (rows && m->T) MB_CUDA (cudaMemcpy (rows + ch.pairs[0] * m->T, dCounts.p, ch.pairs.size() * T * 8, cudaMemcpyDeviceToHost));
  }
  b->lastMs = ms;
  b->lastLaunches = launches;
  if (loglike) MB_CUDA (cudaMemcpy (loglike, dF.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  if (counts && !rows) MB_CUDA (cudaMemcpy (counts, dCounts.p, (size_t) m->T * 8, cudaMemcpyDeviceToHost));
  return 0;
}

// Per chunk: the Forward and Backward fills into full storage, the MEA fill into a third matrix, then generic_viterbi's length
// pass / placement / id pass, the id pass also writing each step's gamma into b->dMeaPost.
int generic_mea (mb_machine* m, mb_batch* b, double* gain, double* loglike) {
  b->lastMs = 0;
  b->lastLaunches = 0;
  if (b->nPairs == 0) return 0;
  std::vector<Chunk> chunks;
  if (plan_chunks (b, m->S, false, 3, chunks)) return 1;
  DevBuf dF, dB, dGain;
  if (dF.alloc ((size_t) b->nPairs * 8) || dB.alloc ((size_t) b->nPairs * 8) || dGain.alloc ((size_t) b->nPairs * 8)) return 1;
  int64_t launches = 0;
  double ms = 0;
  for (auto& ch: chunks) {
    const int64_t nSlots = (int64_t) ch.pairs.size();
    DevBuf dPairs, dOff, dWsF, dWsB, dWsA, dLen, dOutOff;
    if (upload (dPairs, ch.pairs, b->stream) || upload (dOff, ch.wsOff, b->stream) || dWsF.alloc ((size_t) ch.doubles * 8)
        || dWsB.alloc ((size_t) ch.doubles * 8) || dWsA.alloc ((size_t) ch.doubles * 8) || dLen.alloc ((size_t) nSlots * 8)
        || dOutOff.alloc ((size_t) nSlots * 8)) return 1;
    const unsigned grid = (unsigned) nSlots, tg = (unsigned) ((nSlots + 63) / 64);
    if (timing_begin (b)) return 1;
    fill_kernel<OP_SUM, false><<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWsF.as<double>(), 0, dF.as<double>());
    fill_kernel<OP_SUM, true><<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWsB.as<double>(), 0, dB.as<double>());
    mea_fill_kernel<<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWsF.as<double>(), dWsB.as<double>(), dB.as<double>(),
                                                  dWsA.as<double>(), dGain.as<double>());
    mea_traceback_kernel<<<tg, 64, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), nSlots, dOff.as<int64_t>(), dWsF.as<double>(), dWsB.as<double>(),
                                                    dWsA.as<double>(), dB.as<double>(), dGain.as<double>(), dLen.as<int64_t>(), nullptr, nullptr, nullptr);
    MB_CUDA (cudaGetLastError());
    if (paths_place (b, b->meaPaths, ch.pairs.data(), nSlots, dLen.as<int64_t>(), dOutOff.as<int64_t>()) || mea_post_reserve (b, b->meaPaths.pathsPacked)) return 1;
    mea_traceback_kernel<<<tg, 64, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), nSlots, dOff.as<int64_t>(), dWsF.as<double>(), dWsB.as<double>(),
                                                    dWsA.as<double>(), dB.as<double>(), dGain.as<double>(), dLen.as<int64_t>(), b->meaPaths.dPaths, b->dMeaPost,
                                                    dOutOff.as<int64_t>());
    MB_CUDA (cudaGetLastError());
    launches += 5;
    if (timing_end (b, launches)) return 1;
    ms += b->lastMs;
  }
  b->lastMs = ms;
  b->lastLaunches = launches;
  MB_CUDA (cudaMemcpy (gain, dGain.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  if (loglike) MB_CUDA (cudaMemcpy (loglike, dF.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  return 0;
}

// Per chunk that holds the pair of some path: the Forward and Backward fills into full storage, then path_post_kernel over that
// chunk's paths.
int generic_path_posteriors (mb_machine* m, mb_batch* b, int64_t nPaths, const int64_t* pairOfPath, const std::vector<int32_t>& ids,
                             const std::vector<int64_t>& off, std::vector<double>& post) {
  b->lastMs = 0;
  b->lastLaunches = 0;
  post.assign ((size_t) off[nPaths], 0.);
  if (nPaths == 0) return 0;
  std::vector<Chunk> chunks;
  if (plan_chunks (b, m->S, false, 2, chunks)) return 1;
  std::vector<int64_t> chunkOf ((size_t) b->nPairs), slotOf ((size_t) b->nPairs), slotOfPath ((size_t) nPaths), pairs (pairOfPath, pairOfPath + nPaths);
  for (size_t c = 0; c < chunks.size(); ++c)
    for (size_t q = 0; q < chunks[c].pairs.size(); ++q) { chunkOf[chunks[c].pairs[q]] = (int64_t) c; slotOf[chunks[c].pairs[q]] = (int64_t) q; }
  std::vector<std::vector<int64_t>> pathsOf (chunks.size());
  for (int64_t r = 0; r < nPaths; ++r) { pathsOf[chunkOf[pairs[r]]].push_back (r); slotOfPath[r] = slotOf[pairs[r]]; }
  DevBuf dLL, dFLL, dSlotOfPath, dPairOfPath, dIds, dPathOff, dPost, dErr, dErrStep;
  if (dLL.alloc ((size_t) b->nPairs * 8) || dFLL.alloc ((size_t) b->nPairs * 8) || upload (dSlotOfPath, slotOfPath, b->stream)
      || upload (dPairOfPath, pairs, b->stream) || upload (dPathOff, off, b->stream) || dIds.alloc (ids.size() * 4)
      || dPost.alloc (post.size() * 8) || dErr.alloc ((size_t) nPaths * 4) || dErrStep.alloc ((size_t) nPaths * 8)) return 1;
  if (!ids.empty()) MB_CUDA (cudaMemcpyAsync (dIds.p, ids.data(), ids.size() * 4, cudaMemcpyHostToDevice, b->stream));
  int64_t launches = 0;
  double ms = 0;
  for (size_t c = 0; c < chunks.size(); ++c) {
    if (pathsOf[c].empty()) continue;
    const Chunk& ch = chunks[c];
    const int64_t nChunkPaths = (int64_t) pathsOf[c].size();
    DevBuf dPairs, dOff, dWsF, dWsB, dChunkPaths;
    if (upload (dPairs, ch.pairs, b->stream) || upload (dOff, ch.wsOff, b->stream) || upload (dChunkPaths, pathsOf[c], b->stream)
        || dWsF.alloc ((size_t) ch.doubles * 8) || dWsB.alloc ((size_t) ch.doubles * 8)) return 1;
    const unsigned grid = (unsigned) ch.pairs.size();
    if (timing_begin (b)) return 1;
    fill_kernel<OP_SUM, false><<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWsF.as<double>(), 0, dFLL.as<double>());
    fill_kernel<OP_SUM, true><<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWsB.as<double>(), 0, dLL.as<double>());
    path_post_kernel<<<(unsigned) ((nChunkPaths + 63) / 64), 64, 0, b->stream>>> (m->dev, b->dev, dChunkPaths.as<int64_t>(), nChunkPaths, dSlotOfPath.as<int64_t>(),
                                                                                 dPairOfPath.as<int64_t>(), dIds.as<int32_t>(), dPathOff.as<int64_t>(), dOff.as<int64_t>(),
                                                                                 dWsF.as<double>(), dWsB.as<double>(), dLL.as<double>(), dPost.as<double>(),
                                                                                 dErr.as<int32_t>(), dErrStep.as<int64_t>());
    MB_CUDA (cudaGetLastError());
    launches += 3;
    if (timing_end (b, launches)) return 1;
    ms += b->lastMs;
  }
  b->lastMs = ms;
  b->lastLaunches = launches;
  std::vector<int32_t> err ((size_t) nPaths);
  std::vector<int64_t> errStep ((size_t) nPaths);
  MB_CUDA (cudaMemcpy (err.data(), dErr.p, (size_t) nPaths * 4, cudaMemcpyDeviceToHost));
  MB_CUDA (cudaMemcpy (errStep.data(), dErrStep.p, (size_t) nPaths * 8, cudaMemcpyDeviceToHost));
  for (int64_t r = 0; r < nPaths; ++r) {
    if (err[r] == PP_OK) continue;
    static const char* const what[] = { "", "transition %d does not leave the state the path is in", "transition %d does not read the pair's next input token",
                                        "transition %d does not write the pair's next output token", "transition %d leaves the pair's envelope",
                                        "the path ends before the end state at the end of both sequences" };
    char msg[160];
    snprintf (msg, sizeof msg, what[err[r]], err[r] == PP_END ? 0 : ids[off[r] + errStep[r]]);
    set_error ("mb_path_posteriors: path " + std::to_string (r) + " (pair " + std::to_string (pairs[r]) + "), step " + std::to_string (errStep[r]) + ": " + msg);
    return 1;
  }
  if (!post.empty()) MB_CUDA (cudaMemcpy (post.data(), dPost.p, post.size() * 8, cudaMemcpyDeviceToHost));
  return 0;
}

}  // namespace mb
