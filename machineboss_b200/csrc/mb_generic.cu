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
//   BackwardMatrix::getCounts  backward.cpp:62-87     counts_kernel
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

// BackwardMatrix::getCounts (backward.cpp:62-87): count[t] += exp(F(src cell) - ll + w_t + B(dest cell)).
// One CTA per pair; the CTA walks the transitions, each thread sums the cells where the
// transition's labels match the tokens, then a block reduction and one atomic per transition.
__global__ void __launch_bounds__(256) counts_kernel (DevMachine m, DevBatch b, const int64_t* __restrict__ pairs,
                                                      const int64_t* __restrict__ wsOff, const double* __restrict__ wsF,
                                                      const double* __restrict__ wsB, const double* __restrict__ backLL,
                                                      double* __restrict__ counts) {
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
// host side: chunk the batch so that the cell storage of a chunk fits in free device memory
// ---------------------------------------------------------------------------------------------
struct Chunk {
  std::vector<int64_t> pairs, wsOff;
  int64_t doubles = 0;
};

static int plan_chunks (const mb_batch* b, int S, bool rolling, int copies, std::vector<Chunk>& chunks) {
  size_t freeB = 0, totalB = 0;
  MB_CUDA (cudaMemGetInfo (&freeB, &totalB));
  const double budget = 0.80 * (double) freeB / 8.0 / copies;   // doubles per copy
  Chunk cur;
  for (int64_t k = 0; k < b->nPairs; ++k) {
    const int64_t Li = b->xOff[k + 1] - b->xOff[k], Lo = b->yOff[k + 1] - b->yOff[k];
    const double need = rolling ? 3.0 * (double) (Li + 1) * S : (double) (Li + 1) * (double) (Lo + 1) * S;
    if (need > budget) { set_error ("pair " + std::to_string (k) + " needs more device memory than is free (" + std::to_string (need * 8 * copies) + " bytes)"); return 1; }
    if (!cur.pairs.empty() && ((double) cur.doubles + need > budget || cur.pairs.size() >= 65535 * 16)) { chunks.push_back (cur); cur = Chunk(); }
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
      if (paths_place (b, ch.pairs.data(), (int64_t) ch.pairs.size(), dLen.as<int64_t>(), dOutOff.as<int64_t>())) return 1;
      traceback_kernel<<<tg, 64, 0, b->stream>>> (m->dev, cb, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWs.as<double>(), dRes.as<double>(), dLen.as<int64_t>(), b->dPaths, dOutOff.as<int64_t>());
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

int generic_counts (mb_machine* m, mb_batch* b, double* counts, double* loglike) {
  if (b->nPairs == 0) { if (counts) for (int64_t t = 0; t < m->T; ++t) counts[t] = 0; return 0; }
  std::vector<Chunk> chunks;
  if (plan_chunks (b, m->S, false, 2, chunks)) return 1;
  DevBuf dF, dB, dCounts;
  if (dF.alloc ((size_t) b->nPairs * 8) || dB.alloc ((size_t) b->nPairs * 8) || dCounts.alloc ((size_t) std::max<int64_t> (m->T, 1) * 8)) return 1;
  MB_CUDA (cudaMemsetAsync (dCounts.p, 0, (size_t) std::max<int64_t> (m->T, 1) * 8, b->stream));
  int64_t launches = 0;
  double ms = 0;
  for (auto& ch: chunks) {
    DevBuf dPairs, dOff, dWsF, dWsB;
    if (upload (dPairs, ch.pairs, b->stream) || upload (dOff, ch.wsOff, b->stream) || dWsF.alloc ((size_t) ch.doubles * 8) || dWsB.alloc ((size_t) ch.doubles * 8)) return 1;
    const unsigned grid = (unsigned) ch.pairs.size();
    if (timing_begin (b)) return 1;
    fill_kernel<OP_SUM, false><<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWsF.as<double>(), 0, dF.as<double>());
    fill_kernel<OP_SUM, true><<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWsB.as<double>(), 0, dB.as<double>());
    if (counts)
      counts_kernel<<<grid, 256, 0, b->stream>>> (m->dev, b->dev, dPairs.as<int64_t>(), dOff.as<int64_t>(), dWsF.as<double>(), dWsB.as<double>(), dB.as<double>(), dCounts.as<double>());
    MB_CUDA (cudaGetLastError());
    launches += counts ? 3 : 2;
    if (timing_end (b, launches)) return 1;
    ms += b->lastMs;
  }
  b->lastMs = ms;
  b->lastLaunches = launches;
  if (loglike) MB_CUDA (cudaMemcpy (loglike, dF.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  if (counts) MB_CUDA (cudaMemcpy (counts, dCounts.p, (size_t) m->T * 8, cudaMemcpyDeviceToHost));
  return 0;
}

}  // namespace mb
