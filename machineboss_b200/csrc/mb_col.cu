// mb_col.cu -- the column engine: generators without input whose states repeat with a period (profile HMMs and their
// compositions with an error model: SURVEY.md section 8 config 5; the reference builds them in src/hmmer.cpp and
// runs them through the same ForwardMatrix / ViterbiMatrix, forward.cpp:5-56, viterbi.cpp:5-47), swept as a
// two-dimensional recurrence -- column = period of the machine, row = read position -- by a machine-specialised strip
// kernel (mb_col_skeleton.h).  Reached through the lane engine (mb_lane.cu), which keeps the reads the linear sweep
// flags, the traceback, and every machine this file declines.
//
// The analysis (col_analyse).  States [0, a0) are the PREFIX, [a0, a0 + K P) the K PERIODS of P states, the rest the
// SUFFIX.  Accepted when every transition is one of
//     period k -> period k (silent: to a later state of the period; or consuming a token)      SILENT / UP   group
//     period k -> period k+1 (silent, or consuming a token)                                    LEFT / DIAG   group
//     prefix -> prefix, suffix -> suffix                                                       the small programs below
//     prefix -> period k  (any k: "hub" sources such as a profile's begin state)               the prefix state is CARRIED
//     period k -> suffix  (any k: "hub" destinations such as a profile's end state)            an ACCUMULATOR collects it
//     prefix -> suffix                                                                         carried all the way
// A carried state is a state of the cell whose only group is a copy from the column to the left; an accumulator
// is one with that copy plus what its column sends to the suffix state.  The period P is the smallest shift under
// which the (number of transitions, number that consume a token) profile of the middle half of the states repeats;
// the phase a0 is the one that classifies with the fewest groups.  The weights of a group differ from column to
// column (-inf where a column lacks the transition): one table row per column, nSlots = silent groups + nOut per
// token-consuming group.
//
// Three kernels per chunk of reads: col_prefix_kernel (a thread per read: the prefix states over the rows, written as
// the first strip's left boundary), the strip kernel, col_suffix_kernel (a thread per read: the suffix states from
// the last column's accumulators; the end state at the last row is the result).  The two small kernels are
// table-driven and work in the log domain with an exact log-sum-exp (a few dozen states: no time to speak of).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <set>
#include <sstream>
#include <string>
#include <tuple>
#include <vector>

#include "mb_internal.h"
#include "mb_col_skeleton.h"

namespace mb {

enum { CG_SILENT = 0, CG_LEFT = 1, CG_UP = 2, CG_DIAG = 3 };
enum { CE_SILENT = 0, CE_EMIT = 1, CE_EXT_CUR = 2, CE_EXT_PREV = 3 };

struct ColGroup { int type, dst, src, slot; bool emit; };      // cell-state indices; slot < 0: a copy (weight one)
struct ColEntry { int dst, src, tok, kind; int64_t trans; int ord; };   // trans < 0: weight one; ord: rank among the destination's candidates

struct ColProg {
  bool ok = false;
  std::string why;
  int P = 0, a0 = 0, K = 0, nPre = 0, nSuf = 0, nC = 0, nA = 0, nCell = 0;
  int nSlots = 0, nSilSlots = 0, nLU = 0, nLL = 0, nLD = 0, nStrips = 0, nOut = 0;
  int C = 1, Kpad = 0;                           // columns per lane; K rounded up to a multiple of it (empty columns pass the carried states and accumulators on)
  std::vector<int> carried;                      // prefix state behind carried state c
  std::vector<std::pair<int, int>> acc;          // (suffix-local state, consumes a token)
  std::vector<ColGroup> groups;                  // in order of destination
  std::vector<int> upIdx, leftIdx, diagIdx;      // per cell state: index in U[] / the left-going set / Lprev[], or -1
  std::vector<int64_t> slotTrans;                // [K][nSlots] -> transition, or -1
  // Viterbi pointers: cell state d's field is ptrBits[d] wide at (ptrWord[d], ptrShift[d]) of the cell's nPtrWords 32-bit words and
  // holds the index of the winning candidate among the state's groups [groupStart[d], groupStart[d+1]); bpBytes bytes per cell
  std::vector<int> ptrWord, ptrShift, ptrBits, groupStart;
  int nPtrWords = 1, bpBytes = 4;
  std::vector<ColEntry> pre, suf;
};

struct ColEngine {
  ColProg prog;
  std::string source;
  int threads = 256, minBlocks = 2, R = 1;
  bool silInRegs = false;
  bool linearOK = false;
  void* mod = nullptr; void* kSum = nullptr; void* kMax = nullptr;
  int blocksPerSMSum = 1, blocksPerSMMax = 1, numSMs = 148;
  size_t smemBytes = 0;
  std::vector<double> tabLin, tabLog, preW, sufW;
  double* dTabLin = nullptr; double* dTabLog = nullptr;
  int32_t* dPre = nullptr; double* dPreW = nullptr; int32_t* dSuf = nullptr; double* dSufW = nullptr;
  int32_t* dCarriedSlot = nullptr;      // [nC] left-going slot of carried c | [nC] prefix state
  void* kMaxP = nullptr;                // max-plus with pointers
  int blocksPerSMMaxP = 1;
  int32_t* dTbPlan = nullptr;           // the traceback's tables, one array (see ColTbPlan)
  size_t tbOff[12] = { 0 };
};

static ColEngine* ce (const mb_machine* m) { return static_cast<ColEngine*> (m->col); }

// ---------------------------------------------------------------------------------------------
// analysis
// ---------------------------------------------------------------------------------------------
static bool col_classify (const mb_machine* m, int a0, int P, int K, ColProg& out, bool build) {
  const int S = m->S, end = a0 + K * P;
  typedef std::tuple<int, int, int, int> Key;      // (source kind/state, relation, destination, emit)
  std::map<Key, int> keyGroup;
  std::set<int> carriedSet;
  std::set<std::pair<int, int>> accSet;
  struct Raw { int64_t t; int kind; int src, dst; int col; bool emit; };      // kind 0 per->per dk 0, 1 per->per dk 1, 2 pre->per, 3 per->suf
  std::vector<Raw> raws;
  for (int64_t t = 0; t < m->T; ++t) {
    const int s = m->src[t], d = m->dst[t];
    const bool emit = m->out[t] != 0;
    if (m->in[t] != 0) return false;
    if (s == 0 && d == 0 && !emit) continue;      // the start state's silent self-loop contributes nothing (machine.cpp:759)
    const int ws = s < a0 ? 0 : s >= end ? 2 : 1, wd = d < a0 ? 0 : d >= end ? 2 : 1;
    if (ws == 1 && wd == 1) {
      const int ks = (s - a0) / P, kd = (d - a0) / P, js = (s - a0) % P, jd = (d - a0) % P;
      if (kd - ks != 0 && kd - ks != 1) return false;
      if (!emit && kd == ks && jd <= js) return false;
      raws.push_back (Raw { t, kd - ks, js, jd, kd, emit });
    } else if (ws == 0 && wd == 1) { carriedSet.insert (s); raws.push_back (Raw { t, 2, s, (d - a0) % P, (d - a0) / P, emit }); }
    else if (ws == 1 && wd == 2) { accSet.insert (std::make_pair (d - end, emit ? 1 : 0)); raws.push_back (Raw { t, 3, (s - a0) % P, d - end, (s - a0) / P, emit }); }
    else if (ws == 0 && wd == 0) { if (!emit && d <= s) return false; }
    else if (ws == 2 && wd == 2) { if (!emit && d <= s) return false; }
    else if (ws == 0 && wd == 2) carriedSet.insert (s);
    else return false;
  }
  for (auto& r: raws) {
    keyGroup[Key (r.kind == 2 ? -1 - r.src : r.src, r.kind, r.dst, r.emit ? 1 : 0)] = 0;
    if (keyGroup.size() > 640) return false;      // (a phase that needs this many groups is no periodic reading of the machine: give up on it early)
  }
  out.P = P; out.a0 = a0; out.K = K; out.nPre = a0; out.nSuf = S - end;
  out.nC = (int) carriedSet.size(); out.nA = (int) accSet.size();
  out.nCell = out.nC + P + out.nA;
  if (!build) { out.groups.resize (keyGroup.size()); return true; }

  out.nOut = m->nOut;
  out.carried.assign (carriedSet.begin(), carriedSet.end());
  out.acc.assign (accSet.begin(), accSet.end());
  std::map<int, int> carriedIdx;
  for (int c = 0; c < out.nC; ++c) carriedIdx[out.carried[c]] = c;
  std::map<std::pair<int, int>, int> accIdx;
  for (int a = 0; a < out.nA; ++a) accIdx[out.acc[a]] = a;
  auto cellOfPeriod = [&] (int j) { return out.nC + j; };
  // groups, with their cell-state indices
  std::vector<ColGroup> gs;
  for (auto& kv: keyGroup) {
    const int srcKey = std::get<0> (kv.first), kind = std::get<1> (kv.first), dst = std::get<2> (kv.first);
    const bool emit = std::get<3> (kv.first) != 0;
    ColGroup g;
    g.emit = emit; g.slot = 0;
    if (kind == 0) { g.type = emit ? CG_UP : CG_SILENT; g.src = cellOfPeriod (srcKey); g.dst = cellOfPeriod (dst); }
    else if (kind == 1) { g.type = emit ? CG_DIAG : CG_LEFT; g.src = cellOfPeriod (srcKey); g.dst = cellOfPeriod (dst); }
    else if (kind == 2) { g.type = emit ? CG_UP : CG_SILENT; g.src = carriedIdx[-1 - srcKey]; g.dst = cellOfPeriod (dst); }
    else { g.type = emit ? CG_UP : CG_SILENT; g.src = cellOfPeriod (srcKey); g.dst = out.nC + P + accIdx[std::make_pair (dst, emit ? 1 : 0)]; }
    gs.push_back (g);
  }
  for (int c = 0; c < out.nC; ++c) gs.push_back (ColGroup { CG_LEFT, c, c, -1, false });
  for (int a = 0; a < out.nA; ++a) gs.push_back (ColGroup { CG_LEFT, out.nC + P + a, out.nC + P + a, -1, false });
  // Candidates of a state in the reference's order (viterbi.cpp:30-39: token-consuming sources before silent ones, each by
  // source state): the copy from the left stands for sources in earlier columns, carried states are prefix states (lowest
  // index), then the column to the left, then this column.  Strict '<' in the max-plus cell then keeps the same first maximum.
  auto rank = [&] (const ColGroup& g) {
    if (g.slot < 0) return -1;
    const int cls = g.src < out.nC ? 0 : (g.type == CG_LEFT || g.type == CG_DIAG) ? 1 : 2;
    return ((g.emit ? 0 : 1) * 3 + cls) * 4096 + g.src;
  };
  std::stable_sort (gs.begin(), gs.end(), [&] (const ColGroup& p, const ColGroup& q) { return p.dst != q.dst ? p.dst < q.dst : rank (p) < rank (q); });
  int slot = 0;
  for (auto& g: gs) if (g.slot >= 0 && !g.emit) g.slot = slot++;
  out.nSilSlots = slot;
  for (auto& g: gs) if (g.slot >= 0 && g.emit) { g.slot = slot; slot += m->nOut; }
  out.nSlots = std::max (slot, 1);
  out.groups = gs;
  out.upIdx.assign ((size_t) out.nCell, -1); out.leftIdx.assign ((size_t) out.nCell, -1); out.diagIdx.assign ((size_t) out.nCell, -1);
  std::vector<char> isU ((size_t) out.nCell, 0), isL ((size_t) out.nCell, 0), isD ((size_t) out.nCell, 0);
  for (auto& g: gs) { if (g.type == CG_UP) isU[g.src] = 1; if (g.type == CG_LEFT || g.type == CG_DIAG) isL[g.src] = 1; if (g.type == CG_DIAG) isD[g.src] = 1; }
  for (int c = 0; c < out.nC; ++c) isL[c] = 1;      // carried all the way to the suffix kernel
  out.nLU = out.nLL = out.nLD = 0;
  for (int s = 0; s < out.nCell; ++s) { if (isU[s]) out.upIdx[s] = out.nLU++; if (isL[s]) out.leftIdx[s] = out.nLL++; if (isD[s]) out.diagIdx[s] = out.nLD++; }
  // two columns per lane halve the per-cell share of the shuffles, the boundary traffic and the loop (measured on B200:
  // PF00516 812 -> 1332 GCUPS, PF00516 => protpsw 564 -> 685; three and four lose to register pressure)
  out.groupStart.assign ((size_t) out.nCell + 1, 0);
  for (auto& g: gs) out.groupStart[g.dst + 1]++;
  for (int d = 0; d < out.nCell; ++d) out.groupStart[d + 1] += out.groupStart[d];
  out.ptrWord.assign ((size_t) out.nCell, 0); out.ptrShift.assign ((size_t) out.nCell, 0); out.ptrBits.assign ((size_t) out.nCell, 0);
  {
    int word = 0, used = 0;
    for (int d = 0; d < out.nCell; ++d) {
      const int n = out.groupStart[d + 1] - out.groupStart[d];
      int bt = 0; while ((1 << bt) < n) ++bt;
      if (bt == 0) continue;
      if (used + bt > 32) { ++word; used = 0; }
      out.ptrWord[d] = word; out.ptrShift[d] = used; out.ptrBits[d] = bt;
      used += bt;
    }
    out.nPtrWords = word + 1;
    out.bpBytes = word == 0 ? (used <= 8 ? 1 : used <= 16 ? 2 : 4) : 4 * out.nPtrWords;
  }
  out.C = std::max (1, std::min (4, m->opt.get ("col_c", (size_t) out.nSlots * 64 * 8 <= 112 * 1024 ? 2 : 1)));
  out.Kpad = (K + out.C - 1) / out.C * out.C;
  out.nStrips = (out.Kpad + 32 * out.C - 1) / (32 * out.C);
  // per column: which transition fills which slot
  std::map<std::tuple<int, int, int, int>, int> groupOf;      // (type, src, dst, emit) -> index in gs
  for (size_t n = 0; n < gs.size(); ++n) if (gs[n].slot >= 0) groupOf[std::make_tuple (gs[n].type, gs[n].src, gs[n].dst, gs[n].emit ? 1 : 0)] = (int) n;
  out.slotTrans.assign ((size_t) K * out.nSlots, -1);
  for (auto& r: raws) {
    int type, src, dst;
    if (r.kind == 0) { type = r.emit ? CG_UP : CG_SILENT; src = cellOfPeriod (r.src); dst = cellOfPeriod (r.dst); }
    else if (r.kind == 1) { type = r.emit ? CG_DIAG : CG_LEFT; src = cellOfPeriod (r.src); dst = cellOfPeriod (r.dst); }
    else if (r.kind == 2) { type = r.emit ? CG_UP : CG_SILENT; src = carriedIdx[r.src]; dst = cellOfPeriod (r.dst); }
    else { type = r.emit ? CG_UP : CG_SILENT; src = cellOfPeriod (r.src); dst = out.nC + P + accIdx[std::make_pair (r.dst, r.emit ? 1 : 0)]; }
    const ColGroup& g = gs[groupOf[std::make_tuple (type, src, dst, r.emit ? 1 : 0)]];
    int64_t& cell = out.slotTrans[(size_t) r.col * out.nSlots + g.slot + (r.emit ? m->out[r.t] - 1 : 0)];
    if (cell >= 0) { out.why = "parallel transitions with the same label"; return false; }
    cell = r.t;
  }
  // the prefix and suffix programs, by destination (a silent source is an earlier state, so it is final when read)
  for (int64_t t = 0; t < m->T; ++t) {
    const int s = m->src[t], d = m->dst[t];
    const bool emit = m->out[t] != 0;
    if (s == 0 && d == 0 && !emit) continue;
    const int ord = (emit ? 0 : 1) * (S + 1) + s;      // token-consuming candidates first, each class by source state
    if (s < a0 && d < a0) out.pre.push_back (ColEntry { d, s, m->out[t], emit ? CE_EMIT : CE_SILENT, t, ord });
    else if (s >= end && d >= end) out.suf.push_back (ColEntry { d - end, s - end, m->out[t], emit ? CE_EMIT : CE_SILENT, t, ord });
    else if (s < a0 && d >= end) out.suf.push_back (ColEntry { d - end, out.leftIdx[carriedIdx[s]], m->out[t], emit ? CE_EXT_PREV : CE_EXT_CUR, t, ord });
  }
  for (int a = 0; a < out.nA; ++a)      // an accumulator stands for the period states that send to the suffix state: between the prefix and the suffix
    out.suf.push_back (ColEntry { out.acc[a].first, out.leftIdx[out.nC + P + a], 0, CE_EXT_CUR, -1, (out.acc[a].second ? 0 : 1) * (S + 1) + a0 });
  auto byDst = [] (const ColEntry& p, const ColEntry& q) { return p.dst != q.dst ? p.dst < q.dst : p.ord < q.ord; };
  std::stable_sort (out.pre.begin(), out.pre.end(), byDst);
  std::stable_sort (out.suf.begin(), out.suf.end(), byDst);
  return true;
}

static void col_analyse (const mb_machine* m, ColProg& best) {
  best = ColProg();
  const int S = m->S;
  if (m->nIn != 0) { best.why = "the machine reads an input sequence"; return; }
  if (S < 200) { best.why = "fewer than 200 states"; return; }
  if (m->T > 2000000) { best.why = "more than 2 000 000 transitions"; return; }
  std::vector<std::pair<int, int>> sig ((size_t) S, std::make_pair (0, 0));
  for (int64_t t = 0; t < m->T; ++t) { ++sig[m->src[t]].first; if (m->out[t]) ++sig[m->src[t]].second; }
  const int lo = S / 4, hi = 3 * S / 4;
  int P = 0;
  for (int p = 1; p <= 128 && !P; ++p) {
    bool same = true;
    for (int s = lo; s < hi && same; ++s) same = sig[s] == sig[s + p];
    if (same) P = p;
  }
  if (!P) { best.why = "no period of up to 128 states in the transition profile"; return; }
  double bestScore = 1e300;
  int bestA0 = -1, bestK = 0;
  for (int phase = 0; phase < P; ++phase) {
    int a0 = lo - (lo % P) + phase;
    while (a0 - P >= 1) a0 -= P;
    int K = (S - 1 - a0) / P;
    ColProg trial;
    bool ok = false;
    for (int tries = 0; tries < 8 && K >= 32; ++tries) {      // irregular periods at either end go to the prefix / suffix
      if (col_classify (m, a0, P, K, trial, false)) { ok = true; break; }
      if (tries % 2 == 0) --K; else { a0 += P; --K; }
    }
    if (!ok) continue;
    const double score = (double) trial.groups.size() + 4. * (trial.nC + trial.nA) + trial.nPre + trial.nSuf;
    if (score < bestScore) { bestScore = score; bestA0 = a0; bestK = K; }
  }
  if (bestA0 < 0) { best.why = "period " + std::to_string (P) + ": no phase classifies (transitions that skip a period, or run backwards)"; return; }
  if (!col_classify (m, bestA0, P, bestK, best, true)) { if (best.why.empty()) best.why = "classification failed"; return; }
  if (best.nLL < 1 || best.nLL > 40) { best.why = "left-going states: " + std::to_string (best.nLL); return; }
  if (best.nLU > 40) { best.why = "too many states consumed from the row above"; return; }
  if (best.nPre > 64 || best.nSuf > 64) { best.why = "prefix / suffix of more than 64 states"; return; }
  if ((size_t) best.nSlots * 32 * best.C * 8 > 160 * 1024) { best.why = "a strip's weight table exceeds 160 KB"; return; }
  if (best.groups.size() > 600) { best.why = "more than 600 transition groups per cell"; return; }
  if (m->nOut > 250) { best.why = "alphabet too large"; return; }
  best.ok = true;
}

// ---------------------------------------------------------------------------------------------
// code generation
// ---------------------------------------------------------------------------------------------
static void col_generate (const mb_machine* m, ColEngine& E) {
  const ColProg& p = E.prog;
  E.silInRegs = p.nSilSlots * p.C <= m->opt.get ("col_sil_regs", 40);
  E.threads = std::max (32, std::min (1024, m->opt.get ("col_threads", 256) / 32 * 32));
  E.minBlocks = std::max (1, std::min (8, m->opt.get ("col_minblocks", p.nCell <= 12 ? 2 : 1)));
  E.R = std::max (1, std::min (16, m->opt.get ("col_r", 1)));
  std::ostringstream o;
  o << "// generated by machineboss_b200 (mb_col.cu): period " << p.P << ", " << p.K << " columns from state " << p.a0 << ", " << p.nC << " carried, " << p.nA << " accumulators\n";
  o << "typedef unsigned char uint8_t;\ntypedef int int32_t;\ntypedef long long int64_t;\ntypedef unsigned long long uint64_t;\n";
  const int C = p.C;
  o << "#define MB_COL_C " << C << "\n#define MB_NLL " << p.nLL << "\n#define MB_NUREG " << p.nLU * C << "\n#define MB_NDREG " << p.nLD * C << "\n#define MB_NSLOTS " << p.nSlots << "\n";
  o << "#define MB_COL_THREADS " << E.threads << "\n#define MB_COL_MINBLOCKS " << E.minBlocks << "\n";
  o << "#define MB_NPW " << p.nPtrWords << "\n#define MB_BPBYTES " << p.bpBytes << "\n";
  o << "#define MB_COL_DECLW";
  if (E.silInRegs) for (int c = 0; c < C; ++c) for (int q = 0; q < p.nSilSlots; ++q) o << " const double w" << c << "_" << q << " = W[" << q * C + c << " * 32];";
  o << "\n";
  // column c of the lane: its weights sit at W[(slot * C + c) * 32]; what it reads from the column to its left is the
  // shuffled Lin / Lprev for c = 0 and the lane's own previous column otherwise
  auto weight = [&] (const ColGroup& g, int c) {
    std::ostringstream w;
    if (g.emit) w << "W[((" << g.slot << " + tokb) * " << C << " + " << c << ") * 32]";
    else if (E.silInRegs) w << "w" << c << "_" << g.slot;
    else w << "W[" << g.slot * C + c << " * 32]";
    return w.str();
  };
  auto source = [&] (const ColGroup& g, int c) {
    std::ostringstream s;
    if (g.type == CG_SILENT) s << "n" << c << "_" << g.src;
    else if (g.type == CG_LEFT) { if (c) s << "n" << c - 1 << "_" << g.src; else s << "Lin[" << p.leftIdx[g.src] << "]"; }
    else if (g.type == CG_UP) s << "U[" << c * p.nLU + p.upIdx[g.src] << "]";
    else s << "Lprev[" << c * p.nLD + p.diagIdx[g.src] << "]";
    return s.str();
  };
  for (int pass = 0; pass < 3; ++pass) {      // sums; max-plus; max-plus with the winners' indices
    const int lin = pass == 0;
    const bool wp = pass == 2;
    o << "#define MB_COL_CELL_" << (lin ? "LIN" : wp ? "MAXP" : "MAX") << " \\\n";
    for (int c = 0; c < C; ++c) {
      size_t gi = 0;
      for (int d = 0; d < p.nCell; ++d) {
        bool first = true;
        std::ostringstream nm;
        nm << "n" << c << "_" << d;
        const std::string n = nm.str();
        o << "  double " << n;
        std::ostringstream rest;
        const size_t g0 = gi;
        if (wp && p.ptrBits[d]) rest << " unsigned p" << c << "_" << d << " = 0u;";
        for (; gi < p.groups.size() && p.groups[gi].dst == d; ++gi) {
          const ColGroup& g = p.groups[gi];
          if (g.slot < 0) { o << " = " << source (g, c) << ";"; first = false; continue; }      // the copy comes first
          if (lin) {
            if (first) rest << " " << n << " = " << source (g, c) << " * " << weight (g, c) << ";";
            else rest << " " << n << " = fma (" << source (g, c) << ", " << weight (g, c) << ", " << n << ");";
          } else {
            if (first) rest << " " << n << " = " << source (g, c) << " + " << weight (g, c) << ";";
            else if (wp) rest << " { const double cand = " << source (g, c) << " + " << weight (g, c) << "; if (" << n << " < cand) { " << n << " = cand; p" << c << "_" << d << " = " << gi - g0 << "u; } }";
            else rest << " { const double cand = " << source (g, c) << " + " << weight (g, c) << "; if (" << n << " < cand) " << n << " = cand; }";
          }
          if (first) { o << ";"; first = false; }
        }
        if (first) o << " = ZERO;";
        o << rest.str() << " \\\n";
      }
    }
    for (int c = 0; c < C; ++c) for (int s = 0; s < p.nCell; ++s) if (p.upIdx[s] >= 0) o << "  U[" << c * p.nLU + p.upIdx[s] << "] = n" << c << "_" << s << "; \\\n";
    for (int c = 0; c + 1 < C; ++c) for (int s = 0; s < p.nCell; ++s) if (p.diagIdx[s] >= 0) o << "  Lprev[" << (c + 1) * p.nLD + p.diagIdx[s] << "] = n" << c << "_" << s << "; \\\n";
    for (int s = 0; s < p.nCell; ++s) if (p.leftIdx[s] >= 0) o << "  Lown[" << p.leftIdx[s] << "] = n" << C - 1 << "_" << s << "; \\\n";
    if (wp)
      for (int c = 0; c < C; ++c)
        for (int wd = 0; wd < p.nPtrWords; ++wd) {
          o << "  pk[" << c * p.nPtrWords + wd << "] = 0u";
          for (int d = 0; d < p.nCell; ++d) if (p.ptrBits[d] && p.ptrWord[d] == wd) o << " | (p" << c << "_" << d << " << " << p.ptrShift[d] << ")";
          o << "; \\\n";
        }
    o << "\n";
  }
  o << "#define MB_COL_KEEPDIAG";
  for (int s = 0; s < p.nCell; ++s) if (p.diagIdx[s] >= 0) o << " Lprev[" << p.diagIdx[s] << "] = Lin[" << p.leftIdx[s] << "];";
  o << "\n";
  o << kColSkeleton;
  E.source = o.str();
}

// ---------------------------------------------------------------------------------------------
// the prefix and suffix programs on the device (a thread per read, log domain)
// ---------------------------------------------------------------------------------------------
#define COL_MAXSIDE 64
#define COL_MAXLL 40
struct ColSideArgs {
  const uint8_t* y; const int64_t* yOff; const int64_t* order; int64_t nWork;
  double* bnd; const int64_t* bndOff;
  const int32_t* ent; const double* w; int32_t nEnt;      // entries: dst, src, tok, kind
  int32_t nStates, nLL, nC;
  const int32_t* carried;      // [nC] left-going slot | [nC] prefix state
  double* result;
  unsigned short* ptr;      // max-plus with traceback: the winning entry of (row o, work item n, state s) at ptr[(o * nWork + n) * nStates + s] (threads of a warp write neighbours); 0xffff: none
};

__device__ __forceinline__ double col_ninf() { return __longlong_as_double (0xfff0000000000000LL); }
__device__ __forceinline__ double col_lse (double a, double b) {
  const double mx = fmax (a, b), mn = fmin (a, b);
  if (!(mn > col_ninf())) return mx;
  return mx + log1p (exp (mn - mx));
}

template<bool SUM>
__global__ void __launch_bounds__(128) col_prefix_kernel (ColSideArgs A) {
  const int64_t n = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= A.nWork) return;
  const int64_t k = A.order[n];
  const uint8_t* y = A.y + A.yOff[k];
  const int Lo = (int) (A.yOff[k + 1] - A.yOff[k]);
  double* bnd = A.bnd + A.bndOff[n];
  double cur[COL_MAXSIDE], prev[COL_MAXSIDE];
  for (int s = 0; s < A.nStates; ++s) prev[s] = col_ninf();
  const int brow = A.nLL + 1;
  for (int o = 0; o <= Lo; ++o) {
    for (int s = 0; s < A.nStates; ++s) cur[s] = col_ninf();
    if (o == 0) cur[0] = 0.;
    const int tok = o ? y[o - 1] : -1;
    unsigned short* won = (!SUM && A.ptr) ? A.ptr + ((int64_t) o * A.nWork + n) * A.nStates : (unsigned short*) 0;
    if (won) for (int s = 0; s < A.nStates; ++s) won[s] = 0xffff;
    for (int e = 0; e < A.nEnt; ++e) {
      const int dst = A.ent[4 * e], src = A.ent[4 * e + 1], etok = A.ent[4 * e + 2], kind = A.ent[4 * e + 3];
      double v;
      if (kind == CE_SILENT) v = cur[src] + A.w[e];
      else if (etok == tok) v = prev[src] + A.w[e];
      else continue;
      if (SUM) cur[dst] = col_lse (cur[dst], v);
      else if (cur[dst] < v) { cur[dst] = v; if (won) won[dst] = (unsigned short) e; }      // strict '<': the first maximum stays (dpmatrix.defs.h:171-174)
    }
    double* row = bnd + (int64_t) o * brow;
    if (SUM) {      // linear values under a power-of-two frame
      double mx = col_ninf();
      for (int c = 0; c < A.nC; ++c) mx = fmax (mx, cur[A.carried[A.nC + c]]);
      const int fr = mx > col_ninf() ? (int) floor (mx * 1.4426950408889634) : 0;
      for (int j = 0; j < A.nLL; ++j) row[j] = 0.;
      for (int c = 0; c < A.nC; ++c) { const double v = cur[A.carried[A.nC + c]]; row[A.carried[c]] = v > col_ninf() ? exp (v - (double) fr * 0.6931471805599453094) : 0.; }
      row[A.nLL] = (double) fr;
    } else {
      for (int j = 0; j < A.nLL; ++j) row[j] = col_ninf();
      for (int c = 0; c < A.nC; ++c) row[A.carried[c]] = cur[A.carried[A.nC + c]];
      row[A.nLL] = 0.;
    }
    for (int s = 0; s < A.nStates; ++s) prev[s] = cur[s];
  }
}

template<bool SUM>
__global__ void __launch_bounds__(128) col_suffix_kernel (ColSideArgs A) {
  const int64_t n = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= A.nWork) return;
  const int64_t k = A.order[n];
  const uint8_t* y = A.y + A.yOff[k];
  const int Lo = (int) (A.yOff[k + 1] - A.yOff[k]);
  const double* bnd = A.bnd + A.bndOff[n];
  double cur[COL_MAXSIDE], prev[COL_MAXSIDE], X[COL_MAXLL], Xprev[COL_MAXLL];
  for (int s = 0; s < A.nStates; ++s) prev[s] = col_ninf();
  for (int j = 0; j < A.nLL; ++j) Xprev[j] = col_ninf();
  const int brow = A.nLL + 1;
  for (int o = 0; o <= Lo; ++o) {
    const double* row = bnd + (int64_t) o * brow;
    const double fr = SUM ? row[A.nLL] * 0.6931471805599453094 : 0.;
    for (int j = 0; j < A.nLL; ++j) { const double v = row[j]; X[j] = SUM ? (v > 0. ? log (v) + fr : col_ninf()) : v; }
    for (int s = 0; s < A.nStates; ++s) cur[s] = col_ninf();
    const int tok = o ? y[o - 1] : -1;
    unsigned short* won = (!SUM && A.ptr) ? A.ptr + ((int64_t) o * A.nWork + n) * A.nStates : (unsigned short*) 0;
    if (won) for (int s = 0; s < A.nStates; ++s) won[s] = 0xffff;
    for (int e = 0; e < A.nEnt; ++e) {
      const int dst = A.ent[4 * e], src = A.ent[4 * e + 1], etok = A.ent[4 * e + 2], kind = A.ent[4 * e + 3];
      double v;
      if (kind == CE_SILENT) v = cur[src] + A.w[e];
      else if (kind == CE_EXT_CUR) v = X[src] + A.w[e];
      else if (etok != tok) continue;
      else v = (kind == CE_EMIT ? prev[src] : Xprev[src]) + A.w[e];
      if (SUM) cur[dst] = col_lse (cur[dst], v);
      else if (cur[dst] < v) { cur[dst] = v; if (won) won[dst] = (unsigned short) e; }
    }
    for (int s = 0; s < A.nStates; ++s) prev[s] = cur[s];
    for (int j = 0; j < A.nLL; ++j) Xprev[j] = X[j];
  }
  A.result[k] = prev[A.nStates - 1];
}

// ---------------------------------------------------------------------------------------------
// weights, preparation
// ---------------------------------------------------------------------------------------------
// column k = (strip * 32 + lane) * C + c; its weight of slot q sits at [strip][q][c][lane]
static size_t col_tab_index (const ColProg& p, int k, int q) {
  const int strip = k / (32 * p.C), lane = (k / p.C) % 32, c = k % p.C;
  return (((size_t) strip * p.nSlots + q) * p.C + c) * 32 + lane;
}

static void col_fill_weights (const mb_machine* m, ColEngine& E) {
  const ColProg& p = E.prog;
  E.tabLin.assign ((size_t) p.nStrips * p.nSlots * 32 * p.C, 0.);
  E.tabLog.assign ((size_t) p.nStrips * p.nSlots * 32 * p.C, -INFINITY);
  bool ok = true;
  const double lim = 40. * 0.6931471805599453;
  for (int k = 0; k < p.K; ++k)
    for (int q = 0; q < p.nSlots; ++q) {
      const int64_t t = p.slotTrans[(size_t) k * p.nSlots + q];
      if (t < 0) continue;
      const double lw = m->lw[t];
      if (std::isnan (lw) || lw == INFINITY || (std::isfinite (lw) && std::fabs (lw) > lim)) ok = false;
      const size_t at = col_tab_index (p, k, q);
      E.tabLog[at] = lw;
      E.tabLin[at] = std::exp (lw);
    }
  E.preW.assign (std::max<size_t> (p.pre.size(), 1), 0.);
  E.sufW.assign (std::max<size_t> (p.suf.size(), 1), 0.);
  for (size_t e = 0; e < p.pre.size(); ++e) E.preW[e] = p.pre[e].trans >= 0 ? m->lw[p.pre[e].trans] : 0.;
  for (size_t e = 0; e < p.suf.size(); ++e) E.sufW[e] = p.suf[e].trans >= 0 ? m->lw[p.suf[e].trans] : 0.;
  for (double w: E.preW) if (std::isnan (w) || w == INFINITY) ok = false;
  for (double w: E.sufW) if (std::isnan (w) || w == INFINITY) ok = false;
  E.linearOK = ok;
}

int col_update_weights (mb_machine* m) {
  ColEngine* E = ce (m);
  if (!E) return 0;
  col_fill_weights (m, *E);
  if (!E->dTabLin) return 0;      // host only
  MB_CUDA (cudaSetDevice (m->device));
  MB_CUDA (cudaMemcpy (E->dTabLin, E->tabLin.data(), E->tabLin.size() * 8, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (E->dTabLog, E->tabLog.data(), E->tabLog.size() * 8, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (E->dPreW, E->preW.data(), E->preW.size() * 8, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (E->dSufW, E->sufW.data(), E->sufW.size() * 8, cudaMemcpyHostToDevice));
  return 0;
}

void col_destroy (mb_machine* m) {
  ColEngine* E = ce (m);
  if (!E) return;
  if (E->mod) rt_unload (E->mod);
  for (void* p: { (void*) E->dTabLin, (void*) E->dTabLog, (void*) E->dPre, (void*) E->dPreW, (void*) E->dSuf, (void*) E->dSufW, (void*) E->dCarriedSlot, (void*) E->dTbPlan }) if (p) cudaFree (p);
  delete E;
  m->col = nullptr;
}

// Analysis, code generation and (unless hostOnly) compilation + upload.  A machine without the structure is not an
// error: m->col stays null and the lane engine's own sweep runs.
int col_prepare (mb_machine* m, bool hostOnly) {
  if (m->opt.get ("no_col", 0)) return 0;
  ColEngine* E = new ColEngine;
  col_analyse (m, E->prog);
  if (m->opt.get ("verbose", 0)) {
    const ColProg& p = E->prog;
    if (p.ok) fprintf (stderr, "column engine: period %d, %d columns from state %d (prefix %d, suffix %d states), %d carried, %d accumulators, %zu groups, %d weight slots (%d silent), %d up, %d left-going, %d diagonal\n",
                       p.P, p.K, p.a0, p.nPre, p.nSuf, p.nC, p.nA, p.groups.size(), p.nSlots, p.nSilSlots, p.nLU, p.nLL, p.nLD);
    else fprintf (stderr, "column engine: not for this machine (%s)\n", p.why.c_str());
  }
  if (!E->prog.ok) { delete E; return 0; }
  m->col = E;
  col_generate (m, *E);
  col_fill_weights (m, *E);
  if (hostOnly) return 0;
  const ColProg& p = E->prog;
  std::vector<char> cubin;
  if (rt_compile (E->source, ".col.cu", cubin, nullptr)) return 1;
  MB_CUDA (cudaSetDevice (m->device));
  if (rt_load (cubin, &E->mod) || rt_function (E->mod, "mb_k_col_sum", &E->kSum) || rt_function (E->mod, "mb_k_col_max", &E->kMax)
      || rt_function (E->mod, "mb_k_col_maxp", &E->kMaxP)) return 1;
  MB_CUDA (cudaDeviceGetAttribute (&E->numSMs, cudaDevAttrMultiProcessorCount, m->device));
  E->smemBytes = (size_t) (p.nSlots * 32 * p.C + (E->threads / 32) * 16 * p.nLL) * 8;
  if (rt_prepare (E->kSum, E->threads, E->smemBytes, &E->blocksPerSMSum) || rt_prepare (E->kMax, E->threads, E->smemBytes, &E->blocksPerSMMax)
      || rt_prepare (E->kMaxP, E->threads, E->smemBytes, &E->blocksPerSMMaxP)) return 1;
  if (E->blocksPerSMSum < 1 || E->blocksPerSMMax < 1 || E->blocksPerSMMaxP < 1) { set_error ("column engine: a kernel does not fit on an SM"); return 1; }
  {      // the traceback's tables: groupStart | ptrWord | ptrShift | ptrBits | group type | source | slot | left slot -> cell state | carried -> prefix state | slotTrans | prefix entries | suffix entries
    std::vector<int32_t> plan;
    auto section = [&] (int q, const std::vector<int32_t>& v) { E->tbOff[q] = plan.size(); plan.insert (plan.end(), v.begin(), v.end()); };
    std::vector<int32_t> gt, gsrc, gslot, leftCell ((size_t) p.nLL, -1), st ((size_t) p.K * p.nSlots), pe, se;
    for (auto& g: p.groups) { gt.push_back (g.type); gsrc.push_back (g.src); gslot.push_back (g.slot); }
    for (int c = 0; c < p.nCell; ++c) if (p.leftIdx[c] >= 0) leftCell[p.leftIdx[c]] = c;
    for (size_t q = 0; q < st.size(); ++q) st[q] = (int32_t) p.slotTrans[q];
    for (auto& e: p.pre) { pe.push_back (e.src); pe.push_back (e.kind); pe.push_back ((int32_t) e.trans); }
    for (auto& e: p.suf) { se.push_back (e.src); se.push_back (e.kind); se.push_back ((int32_t) e.trans); }
    section (0, std::vector<int32_t> (p.groupStart.begin(), p.groupStart.end()));
    section (1, std::vector<int32_t> (p.ptrWord.begin(), p.ptrWord.end()));
    section (2, std::vector<int32_t> (p.ptrShift.begin(), p.ptrShift.end()));
    section (3, std::vector<int32_t> (p.ptrBits.begin(), p.ptrBits.end()));
    section (4, gt); section (5, gsrc); section (6, gslot); section (7, leftCell);
    section (8, std::vector<int32_t> (p.carried.begin(), p.carried.end()));
    section (9, st); section (10, pe); section (11, se);
    MB_CUDA (cudaMalloc (&E->dTbPlan, std::max<size_t> (plan.size(), 1) * 4));
    MB_CUDA (cudaMemcpy (E->dTbPlan, plan.data(), plan.size() * 4, cudaMemcpyHostToDevice));
  }
  MB_CUDA (cudaMalloc (&E->dTabLin, E->tabLin.size() * 8));
  MB_CUDA (cudaMalloc (&E->dTabLog, E->tabLog.size() * 8));
  std::vector<int32_t> pre, suf, car;
  for (auto& e: p.pre) { pre.push_back (e.dst); pre.push_back (e.src); pre.push_back (e.tok); pre.push_back (e.kind); }
  for (auto& e: p.suf) { suf.push_back (e.dst); suf.push_back (e.src); suf.push_back (e.tok); suf.push_back (e.kind); }
  for (int c = 0; c < p.nC; ++c) car.push_back (p.leftIdx[c]);
  for (int c = 0; c < p.nC; ++c) car.push_back (p.carried[c]);
  MB_CUDA (cudaMalloc (&E->dPre, std::max<size_t> (pre.size(), 1) * 4));
  MB_CUDA (cudaMalloc (&E->dSuf, std::max<size_t> (suf.size(), 1) * 4));
  MB_CUDA (cudaMalloc (&E->dCarriedSlot, std::max<size_t> (car.size(), 1) * 4));
  MB_CUDA (cudaMalloc (&E->dPreW, E->preW.size() * 8));
  MB_CUDA (cudaMalloc (&E->dSufW, E->sufW.size() * 8));
  if (!pre.empty()) MB_CUDA (cudaMemcpy (E->dPre, pre.data(), pre.size() * 4, cudaMemcpyHostToDevice));
  if (!suf.empty()) MB_CUDA (cudaMemcpy (E->dSuf, suf.data(), suf.size() * 4, cudaMemcpyHostToDevice));
  if (!car.empty()) MB_CUDA (cudaMemcpy (E->dCarriedSlot, car.data(), car.size() * 4, cudaMemcpyHostToDevice));
  if (m->opt.get ("verbose", 0))
    fprintf (stderr, "column engine: %d column(s) per lane, %d threads per CTA, %zu B smem, %d / %d CTAs per SM (sums / max), silent weights in %s\n", p.C, E->threads, E->smemBytes, E->blocksPerSMSum, E->blocksPerSMMax, E->silInRegs ? "registers" : "shared memory");
  return col_update_weights (m);
}

int col_compile_check (const mb_machine* m, std::string* log) {
  ColEngine E;
  col_analyse (m, E.prog);
  if (!E.prog.ok) { set_error ("machine not eligible for the column engine: " + E.prog.why); return 1; }
  col_generate (m, E);
  std::vector<char> cubin;
  return rt_compile (E.source, ".col.cu", cubin, log);
}

bool col_usable (const mb_machine* m, bool sums) {
  const ColEngine* E = ce (m);
  return E && E->mod && (!sums || E->linearOK) && !m->opt.get ("no_col", 0);
}

int col_info (const mb_machine* m, int32_t* info) {
  const ColEngine* E = ce (m);
  for (int q = 0; q < 12; ++q) info[q] = 0;
  if (!E) return 0;
  const ColProg& p = E->prog;
  const int v[12] = { 1, p.P, p.a0, p.K, p.nPre, p.nSuf, p.nC, p.nA, (int) p.groups.size(), p.nSlots, p.nLL, p.nLU };
  for (int q = 0; q < 12; ++q) info[q] = v[q];
  return 0;
}

// ---------------------------------------------------------------------------------------------
// launch: chunks of reads whose boundary buffers fit the budget; three kernels per chunk
// ---------------------------------------------------------------------------------------------
struct MBColArgsHost {      // must match struct MBColArgs in the skeleton
  const uint8_t* y; const int64_t* yOff;
  const int64_t* order; int64_t nWork; unsigned long long* counter;
  double* bnd; const int64_t* bndOff;
  const double* tab;
  int32_t* flag;
  int nStrips, K, R, pad;
  unsigned char* bp; const int64_t* bpOff;
};

// order: reads, longest first.  sums: Forward (flags set for the reads whose result must not be trusted); else Viterbi scores.
static int col_launch (mb_machine* m, mb_batch* b, const std::vector<int64_t>& order, bool sums, double* dResult, int32_t* dFlag, int64_t* launches) {
  ColEngine& E = *ce (m);
  const ColProg& p = E.prog;
  const int brow = p.nLL + 1;
  size_t freeB = 0, totalB = 0;
  MB_CUDA (cudaMemGetInfo (&freeB, &totalB));
  const double budget = std::min (0.5 * (double) freeB, (double) m->opt.get ("col_bnd_budget_mb", 4096) * 1048576.);
  const int warps = E.threads / 32;
  for (size_t c0 = 0; c0 < order.size();) {
    std::vector<int64_t> off;
    double doubles = 0;
    size_t c1 = c0;
    while (c1 < order.size()) {
      const int64_t k = order[c1];
      const double need = (double) (b->yOff[k + 1] - b->yOff[k] + 1) * brow;
      if (c1 > c0 && (doubles + need) * 8 > budget) break;
      off.push_back ((int64_t) doubles);
      doubles += need;
      ++c1;
    }
    const int64_t nWork = (int64_t) (c1 - c0);
    int64_t* dOrder = (int64_t*) ws_reserve (b, WS_ORDER, (size_t) nWork * 8);
    int64_t* dOff = (int64_t*) ws_reserve (b, WS_ITEMBND, (size_t) nWork * 8);
    double* dBnd = (double*) ws_reserve (b, WS_BND, (size_t) doubles * 8);
    unsigned long long* dCounter = (unsigned long long*) ws_reserve (b, WS_COUNTER, 8);
    if (!dOrder || !dOff || !dBnd || !dCounter) return 1;
    b->wsOrderHoldsFull = false;
    MB_CUDA (cudaMemcpyAsync (dOrder, order.data() + c0, (size_t) nWork * 8, cudaMemcpyHostToDevice, b->stream));
    MB_CUDA (cudaMemcpyAsync (dOff, off.data(), (size_t) nWork * 8, cudaMemcpyHostToDevice, b->stream));
    MB_CUDA (cudaMemsetAsync (dCounter, 0, 8, b->stream));
    ColSideArgs S;
    S.y = b->dY; S.yOff = b->dYOff; S.order = dOrder; S.nWork = nWork; S.bnd = dBnd; S.bndOff = dOff;
    S.ent = E.dPre; S.w = E.dPreW; S.nEnt = (int32_t) p.pre.size(); S.nStates = p.nPre; S.nLL = p.nLL; S.nC = p.nC; S.carried = E.dCarriedSlot; S.result = dResult;
    S.ptr = nullptr;
    const unsigned sideGrid = (unsigned) ((nWork + 127) / 128);
    if (sums) col_prefix_kernel<true><<<sideGrid, 128, 0, b->stream>>> (S); else col_prefix_kernel<false><<<sideGrid, 128, 0, b->stream>>> (S);
    MB_CUDA (cudaGetLastError());
    MBColArgsHost A;
    A.y = b->dY; A.yOff = b->dYOff; A.order = dOrder; A.nWork = nWork; A.counter = dCounter;
    A.bnd = dBnd; A.bndOff = dOff; A.tab = sums ? E.dTabLin : E.dTabLog; A.flag = dFlag;
    A.nStrips = p.nStrips; A.K = p.Kpad; A.R = E.R; A.pad = 0; A.bp = nullptr; A.bpOff = nullptr;
    const int64_t groups = (nWork + (int64_t) warps * E.R - 1) / ((int64_t) warps * E.R);
    const int64_t grid = std::max<int64_t> (1, std::min<int64_t> ((int64_t) E.numSMs * (sums ? E.blocksPerSMSum : E.blocksPerSMMax), groups));
    void* params[1] = { &A };
    if (rt_launch (sums ? E.kSum : E.kMax, (unsigned) grid, (unsigned) E.threads, E.smemBytes, b->stream, params)) return 1;
    S.ent = E.dSuf; S.w = E.dSufW; S.nEnt = (int32_t) p.suf.size(); S.nStates = p.nSuf;
    if (sums) col_suffix_kernel<true><<<sideGrid, 128, 0, b->stream>>> (S); else col_suffix_kernel<false><<<sideGrid, 128, 0, b->stream>>> (S);
    MB_CUDA (cudaGetLastError());
    if (launches) *launches += 3;
    if (m->opt.get ("verbose", 0))
      fprintf (stderr, "column engine: %lld reads, grid %lld x %d threads, %d read(s) per warp and strip, boundary rows %.1f MB\n", (long long) nWork, (long long) grid, E.threads, E.R, doubles * 8 / 1e6);
    c0 = c1;
    if (c0 < order.size()) MB_CUDA (cudaStreamSynchronize (b->stream));      // the next chunk reuses the workspace
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Viterbi with traceback: the max-plus sweep storing every cell's pointers, then a thread per read walking them back
// (col_walk below is the same walk on the host).  Chunks of reads whose pointers fit in memory.
// ---------------------------------------------------------------------------------------------
struct ColTbPlan {
  const int32_t *groupStart, *ptrWord, *ptrShift, *ptrBits, *gType, *gSrc, *gSlot, *leftCell, *carried, *slotTrans, *preEnt, *sufEnt;
  int32_t nCell, nC, K, nPre, nSuf, nSlots, bpBytes, C;      // C: columns per lane of the sweep that stored the pointers
};

// out == nullptr: lengths only; otherwise the path is written start -> end at out[outOff[n] ..) (lenOut[n] from the first pass)
__global__ void __launch_bounds__(64) col_traceback_kernel (ColTbPlan p, const uint8_t* __restrict__ yAll, const int64_t* __restrict__ yOff, const int64_t* __restrict__ order, int64_t nWork,
                                      const unsigned char* __restrict__ bp, const int64_t* __restrict__ bpOff,
                                      const unsigned short* __restrict__ prePtr, const unsigned short* __restrict__ sufPtr,
                                      const double* __restrict__ score, int64_t* __restrict__ lenOut, int32_t* __restrict__ out, const int64_t* __restrict__ outOff) {
  const int64_t n = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= nWork) return;
  const int64_t kr = order[n];
  const uint8_t* y = yAll + yOff[kr];
  const int64_t Lo = yOff[kr + 1] - yOff[kr];
  const unsigned char* cells = bp + bpOff[n];
  const unsigned short* preP = prePtr + n * p.nPre;      // row o: + o * nWork * nPre
  const unsigned short* sufP = sufPtr + n * p.nSuf;
  int64_t len = 0;
  if (score[kr] > -INFINITY) {      // boss.cpp:831
    const int64_t total = out ? lenOut[n] : 0;
    int32_t* dst = out ? out + outOff[n] : nullptr;
    int where = 2, k = p.K - 1, s = p.nSuf - 1;
    int64_t o = Lo;
    const int64_t limit = (Lo + 2) * ((int64_t) p.K * 4 + p.nPre + p.nSuf + p.nCell + 4);
    for (int64_t guard = 0; guard < limit; ++guard) {
      if (where == 0 && o == 0 && s == 0) break;
      int32_t tr = -1;
      if (where == 2) {
        const int e = sufP[o * nWork * p.nSuf + s];
        if (e == 0xffff) break;
        const int src = p.sufEnt[3 * e], kind = p.sufEnt[3 * e + 1];
        tr = p.sufEnt[3 * e + 2];
        if (kind == CE_SILENT) s = src;
        else if (kind == CE_EMIT) { s = src; --o; }
        else { where = 1; k = p.K - 1; s = p.leftCell[src]; if (kind == CE_EXT_PREV) --o; }
      } else if (where == 1) {
        const int bits = p.ptrBits[s];
        int idx = 0;
        if (bits) {
          // sweep order (see MBColArgs::bp): column k is column k % C of lane (k / C) % 32 in strip k / (32 C), stored at step o + lane
          const int strip = k / (32 * p.C), lane = (k / p.C) & 31;
          const unsigned char* c = cells + ((((int64_t) strip * (Lo + 32) + o + lane) * 32 + lane) * p.C + k % p.C) * p.bpBytes;
          const unsigned v = p.bpBytes == 1 ? (unsigned) c[0] : p.bpBytes == 2 ? (unsigned) *(const unsigned short*) c : ((const unsigned*) c)[p.ptrWord[s]];
          idx = (int) ((v >> p.ptrShift[s]) & ((1u << bits) - 1u));
        }
        const int g = p.groupStart[s] + idx;
        if (g >= p.groupStart[s + 1]) break;
        const int slot = p.gSlot[g], type = p.gType[g];
        if (slot < 0) {      // the copy from the left: no transition
          if (k == 0) { if (s >= p.nC) break; where = 0; s = p.carried[s]; }
          else if (!bits) k = 0;      // nothing else ever enters this state (a carried state): straight to the first column
          else --k;
          continue;
        }
        const bool emit = type == CG_UP || type == CG_DIAG;
        tr = p.slotTrans[(int64_t) k * p.nSlots + slot + (emit ? y[o - 1] - 1 : 0)];
        if (tr < 0) break;
        s = p.gSrc[g];
        if (type == CG_LEFT || type == CG_DIAG) { if (k == 0) break; --k; }
        if (emit) --o;
      } else {
        const int e = preP[o * nWork * p.nPre + s];
        if (e == 0xffff) break;
        tr = p.preEnt[3 * e + 2];
        s = p.preEnt[3 * e];
        if (p.preEnt[3 * e + 1] == CE_EMIT) --o;
      }
      if (tr >= 0) { if (dst && len < total) dst[total - 1 - len] = tr; ++len; }
    }
  }
  if (!out) lenOut[n] = len;
}

// scores (dResult, by read) and paths (b->viterbiPaths) of every read in `order`; *ms receives the device time
static int col_viterbi_paths (mb_machine* m, mb_batch* b, const std::vector<int64_t>& order, double* dResult, int64_t* launches, double* msOut) {
  ColEngine& E = *ce (m);
  const ColProg& p = E.prog;
  const int brow = p.nLL + 1;
  const int64_t stepBytes = (int64_t) 32 * p.C * p.bpBytes;      // one (strip, step) block of pointers
  size_t freeB = 0, totalB = 0;
  MB_CUDA (cudaMemGetInfo (&freeB, &totalB));
  const double budget = std::min (0.6 * (double) freeB, (double) m->opt.get ("col_bp_budget_mb", 1 << 20) * 1048576.);
  const int warps = E.threads / 32;
  double ms = 0;
  ColTbPlan T;
  const int32_t* base = E.dTbPlan;
  T.groupStart = base + E.tbOff[0]; T.ptrWord = base + E.tbOff[1]; T.ptrShift = base + E.tbOff[2]; T.ptrBits = base + E.tbOff[3];
  T.gType = base + E.tbOff[4]; T.gSrc = base + E.tbOff[5]; T.gSlot = base + E.tbOff[6]; T.leftCell = base + E.tbOff[7]; T.carried = base + E.tbOff[8];
  T.slotTrans = base + E.tbOff[9]; T.preEnt = base + E.tbOff[10]; T.sufEnt = base + E.tbOff[11];
  T.nCell = p.nCell; T.nC = p.nC; T.K = p.K; T.nPre = p.nPre; T.nSuf = p.nSuf; T.nSlots = p.nSlots; T.bpBytes = p.bpBytes; T.C = p.C;
  for (size_t c0 = 0; c0 < order.size();) {
    std::vector<int64_t> off, bpOff;
    double doubles = 0, bpBytes = 0, sideShorts = 0;
    size_t c1 = c0;
    const double rowsMax = (double) (b->yOff[order[c0] + 1] - b->yOff[order[c0]] + 1);      // the chunk's longest read comes first
    while (c1 < order.size()) {
      const int64_t k = order[c1];
      const double rows = (double) (b->yOff[k + 1] - b->yOff[k] + 1);
      const double bpNeed = (double) (((int64_t) p.nStrips * (int64_t) (rows + 31) * stepBytes + 15) / 16 * 16);
      const double need = rows * (brow * 8 + 16) + rowsMax * (p.nPre + p.nSuf) * 2 + bpNeed;      // (the prefix / suffix pointers are [row][read][state]: every read pays for the longest one's rows)
      if (need > budget) { set_error ("column engine: one read's Viterbi pointers need more device memory than is free"); return 1; }
      if (c1 > c0 && doubles * 8 + bpBytes + sideShorts * 2 + need > budget) break;
      off.push_back ((int64_t) doubles); bpOff.push_back ((int64_t) bpBytes);
      doubles += rows * brow; bpBytes += bpNeed; sideShorts += rowsMax * (p.nPre + p.nSuf);
      ++c1;
    }
    const int64_t nWork = (int64_t) (c1 - c0);
    b->wsOrderHoldsFull = false;
    int64_t* dOrder = (int64_t*) ws_reserve (b, WS_ORDER, (size_t) nWork * 8);
    int64_t* dOffs = (int64_t*) ws_reserve (b, WS_ITEMBND, (size_t) nWork * 8 * 2);      // bnd | bp offsets
    double* dBnd = (double*) ws_reserve (b, WS_BND, (size_t) doubles * 8);
    unsigned char* dBp = (unsigned char*) ws_reserve (b, WS_TB, (size_t) bpBytes + 8);
    unsigned short* dSide = (unsigned short*) ws_reserve (b, WS_PATHTMP, (size_t) sideShorts * 2 + 8);
    unsigned long long* dCounter = (unsigned long long*) ws_reserve (b, WS_COUNTER, 8);
    int64_t* dLen = (int64_t*) ws_reserve (b, WS_LEN, (size_t) nWork * 8);
    int64_t* dOutOff = (int64_t*) ws_reserve (b, WS_OUTOFF, (size_t) nWork * 8);
    if (!dOrder || !dOffs || !dBnd || !dBp || !dSide || !dCounter || !dLen || !dOutOff) return 1;
    MB_CUDA (cudaMemcpyAsync (dOrder, order.data() + c0, (size_t) nWork * 8, cudaMemcpyHostToDevice, b->stream));
    MB_CUDA (cudaMemcpyAsync (dOffs, off.data(), (size_t) nWork * 8, cudaMemcpyHostToDevice, b->stream));
    MB_CUDA (cudaMemcpyAsync (dOffs + nWork, bpOff.data(), (size_t) nWork * 8, cudaMemcpyHostToDevice, b->stream));
    unsigned short* dPreP = dSide;
    unsigned short* dSufP = dSide + (int64_t) rowsMax * nWork * p.nPre;
    MB_CUDA (cudaMemsetAsync (dCounter, 0, 8, b->stream));
    if (timing_begin (b)) return 1;
    ColSideArgs S;
    S.y = b->dY; S.yOff = b->dYOff; S.order = dOrder; S.nWork = nWork; S.bnd = dBnd; S.bndOff = dOffs;
    S.ent = E.dPre; S.w = E.dPreW; S.nEnt = (int32_t) p.pre.size(); S.nStates = p.nPre; S.nLL = p.nLL; S.nC = p.nC; S.carried = E.dCarriedSlot; S.result = dResult;
    S.ptr = dPreP;
    const unsigned sideGrid = (unsigned) ((nWork + 127) / 128);
    col_prefix_kernel<false><<<sideGrid, 128, 0, b->stream>>> (S);
    MB_CUDA (cudaGetLastError());
    MBColArgsHost A;
    A.y = b->dY; A.yOff = b->dYOff; A.order = dOrder; A.nWork = nWork; A.counter = dCounter;
    A.bnd = dBnd; A.bndOff = dOffs; A.tab = E.dTabLog; A.flag = nullptr;
    A.nStrips = p.nStrips; A.K = p.Kpad; A.R = E.R; A.pad = 0; A.bp = dBp; A.bpOff = dOffs + nWork;
    const int64_t groups = (nWork + (int64_t) warps * E.R - 1) / ((int64_t) warps * E.R);
    const int64_t grid = std::max<int64_t> (1, std::min<int64_t> ((int64_t) E.numSMs * E.blocksPerSMMaxP, groups));
    void* params[1] = { &A };
    if (rt_launch (E.kMaxP, (unsigned) grid, (unsigned) E.threads, E.smemBytes, b->stream, params)) return 1;
    S.ent = E.dSuf; S.w = E.dSufW; S.nEnt = (int32_t) p.suf.size(); S.nStates = p.nSuf; S.ptr = dSufP;
    col_suffix_kernel<false><<<sideGrid, 128, 0, b->stream>>> (S);
    MB_CUDA (cudaGetLastError());
    const unsigned tbGrid = (unsigned) ((nWork + 63) / 64);
    col_traceback_kernel<<<tbGrid, 64, 0, b->stream>>> (T, b->dY, b->dYOff, dOrder, nWork, dBp, dOffs + nWork, dPreP, dSufP, dResult, dLen, nullptr, nullptr);
    MB_CUDA (cudaGetLastError());
    if (paths_place (b, b->viterbiPaths, order.data() + c0, nWork, dLen, dOutOff)) return 1;
    col_traceback_kernel<<<tbGrid, 64, 0, b->stream>>> (T, b->dY, b->dYOff, dOrder, nWork, dBp, dOffs + nWork, dPreP, dSufP, dResult, dLen, b->viterbiPaths.dPaths, dOutOff);
    MB_CUDA (cudaGetLastError());
    if (launches) *launches += 5;
    if (timing_end (b, 5)) return 1;
    ms += b->lastMs;
    if (m->opt.get ("verbose", 0))
      fprintf (stderr, "column engine: Viterbi with traceback, %lld reads, %d B of pointers per cell, %.1f MB of pointers, %.1f MB of boundary rows\n", (long long) nWork, p.bpBytes, bpBytes / 1e6, doubles * 8 / 1e6);
    c0 = c1;
  }
  if (msOut) *msOut = ms;
  return 0;
}

int col_forward (mb_machine* m, mb_batch* b, double* loglike) {
  b->lastRedo = 0;
  if (b->nPairs == 0) return 0;
  const std::vector<int64_t> order = lane_order (b, nullptr);
  DevBuf dRes, dFlag;
  if (dRes.alloc ((size_t) b->nPairs * 8) || dFlag.alloc ((size_t) b->nPairs * 4)) return 1;
  MB_CUDA (cudaMemsetAsync (dFlag.p, 0, (size_t) b->nPairs * 4, b->stream));
  if (timing_begin (b)) return 1;
  // the linear sweep; reads it flags, or that come out without any path, are decided by the lane engine's log-domain sweep
  int64_t launches = 0;
  if (col_launch (m, b, order, true, dRes.as<double>(), dFlag.as<int32_t>(), &launches)) return 1;
  std::vector<int32_t> flag ((size_t) b->nPairs);
  std::vector<double> res ((size_t) b->nPairs);
  MB_CUDA (cudaMemcpyAsync (flag.data(), dFlag.p, flag.size() * 4, cudaMemcpyDeviceToHost, b->stream));
  MB_CUDA (cudaMemcpyAsync (res.data(), dRes.p, res.size() * 8, cudaMemcpyDeviceToHost, b->stream));
  MB_CUDA (cudaStreamSynchronize (b->stream));
  std::vector<int64_t> redo;
  for (int64_t k = 0; k < b->nPairs; ++k) if (flag[k] || !(res[k] > -INFINITY)) redo.push_back (k);
  if (!redo.empty()) {
    if (lane_forward_log_subset (m, b, redo, dRes.as<double>(), dFlag.as<int32_t>())) return 1;
    ++launches;
  }
  b->lastRedo = (int64_t) redo.size();
  if (timing_end (b, launches)) return 1;
  MB_CUDA (cudaMemcpy (loglike, dRes.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  return 0;
}

// scores only: the max-plus sweep; with pathLen: the sweep with pointers and the column engine's own walk back
int col_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen) {
  if (b->nPairs == 0) return 0;
  const std::vector<int64_t> order = lane_order (b, nullptr);
  DevBuf dRes;
  if (dRes.alloc ((size_t) b->nPairs * 8)) return 1;
  if (!pathLen) {
    if (timing_begin (b)) return 1;
    int64_t launches = 0;
    if (col_launch (m, b, order, false, dRes.as<double>(), nullptr, &launches)) return 1;
    if (timing_end (b, launches)) return 1;
  } else {
    int64_t launches = 0;
    double ms = 0;
    if (col_viterbi_paths (m, b, order, dRes.as<double>(), &launches, &ms)) return 1;
    b->lastMs = ms;
    b->lastLaunches = launches;
  }
  MB_CUDA (cudaMemcpy (score, dRes.p, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  return 0;
}

// ---------------------------------------------------------------------------------------------
// the column program executed on the host for one read (diagnostic: pins the analysis and the tables without a device)
// op 0: log-sum-exp (exact), 1: max
// ---------------------------------------------------------------------------------------------
// The walk back over the pointers of the max-plus sweep (DPMatrix::traceBack, dpmatrix.defs.h:82-110, in the column
// program's coordinates), shared by the host emulation and -- through the same tables -- the device kernel.  A position is
// (where, k, o, s): where 2 = suffix state s, 1 = cell state s of column k, 0 = prefix state s, at row o.
//   suffix entry won: silent / token-consuming inside the suffix, or an external one -- an accumulator or a carried state
//     of the last column (row o, or o - 1 when the entry consumes the token);
//   cell group won: a copy from the left moves one column left without a transition (from column 0 into the prefix: a
//     carried state IS its prefix state); SILENT stays, LEFT moves a column, UP a row, DIAG both;
//   prefix entry won: as in the suffix; the walk ends at (row 0, state 0).
struct ColPtrs {      // what col_emulate records for the walk
  std::vector<int32_t> pre, cell, suf;      // [o][state] entry index; [o][k][cell state] group index; -1: nothing won
};

static int col_walk (const ColProg& p, const uint8_t* y, int64_t Lo, const ColPtrs& P, std::vector<int64_t>& path) {
  path.clear();
  int where = 2, k = p.K - 1, s = p.nSuf - 1;
  int64_t o = Lo;
  auto cellOfLeft = [&] (int leftSlot) { for (int c = 0; c < p.nCell; ++c) if (p.leftIdx[c] == leftSlot) return c; return -1; };
  for (int64_t guard = 0; guard < (Lo + 2) * ((int64_t) p.K * p.nCell + p.nPre + p.nSuf + 2); ++guard) {
    if (where == 0 && o == 0 && s == 0) { std::reverse (path.begin(), path.end()); return 0; }
    if (where == 2) {
      const int e = P.suf[(size_t) o * p.nSuf + s];
      if (e < 0) break;
      const ColEntry& en = p.suf[e];
      if (en.trans >= 0) path.push_back (en.trans);
      if (en.kind == CE_SILENT) s = en.src;
      else if (en.kind == CE_EMIT) { s = en.src; --o; }
      else { where = 1; k = p.K - 1; s = cellOfLeft (en.src); if (en.kind == CE_EXT_PREV) --o; }
    } else if (where == 1) {
      const int gi = P.cell[((size_t) o * p.K + k) * p.nCell + s];
      if (gi < 0) break;
      const ColGroup& g = p.groups[gi];
      if (g.slot < 0) {      // the copy from the left
        if (k == 0) { if (s >= p.nC) break; where = 0; s = p.carried[s]; } else --k;
        continue;
      }
      const int64_t t = p.slotTrans[(size_t) k * p.nSlots + g.slot + (g.emit ? y[o - 1] - 1 : 0)];
      if (t < 0) break;
      path.push_back (t);
      s = g.src;
      if (g.type == CG_LEFT || g.type == CG_DIAG) { if (k == 0) break; --k; }
      if (g.type == CG_UP || g.type == CG_DIAG) --o;
    } else {
      const int e = P.pre[(size_t) o * p.nPre + s];
      if (e < 0) break;
      const ColEntry& en = p.pre[e];
      path.push_back (en.trans);
      s = en.src;
      if (en.kind == CE_EMIT) --o;
    }
  }
  set_error ("column engine: the walk back over the pointers did not reach the start state");
  return 1;
}

int col_emulate (const mb_machine* m, const uint8_t* y, int64_t Lo, int op, double* result, std::vector<int64_t>* path) {
  const ColEngine* E = ce (m);
  if (!E) { set_error ("column engine: no program for this machine"); return 1; }
  const ColProg& p = E->prog;
  const double NINF = -INFINITY;
  const bool ptrs = op == 1 && path;
  ColPtrs P;
  if (ptrs) {
    P.pre.assign ((size_t) (Lo + 1) * p.nPre, -1);
    P.cell.assign ((size_t) (Lo + 1) * p.K * p.nCell, -1);
    P.suf.assign ((size_t) (Lo + 1) * p.nSuf, -1);
  }
  // a <- a (+) v; max-plus keeps the FIRST maximum (strict '<', dpmatrix.defs.h:171-174) and notes who won
  auto comb = [&] (double& a, double v, int32_t* ptr, int who) {
    if (op == 1) { if (a < v) { a = v; if (ptr) *ptr = who; } return; }
    const double mx = std::max (a, v), mn = std::min (a, v);
    a = mn > NINF ? mx + std::log1p (std::exp (mn - mx)) : mx;
  };
  auto tabw = [&] (int k, int slot) { return E->tabLog[col_tab_index (p, k, slot)]; };
  std::vector<double> preCur ((size_t) std::max (p.nPre, 1), NINF), prePrev = preCur, sufCur ((size_t) std::max (p.nSuf, 1), NINF), sufPrev = sufCur;
  std::vector<double> cur ((size_t) p.K * p.nCell, NINF), prev = cur;
  std::vector<double> bCur ((size_t) p.nCell, NINF), bPrev = bCur, xPrev ((size_t) p.nCell, NINF);      // the boundary column (column -1) at this row and the row above
  for (int64_t o = 0; o <= Lo; ++o) {
    const int tok = o ? y[o - 1] : -1;
    std::fill (preCur.begin(), preCur.end(), NINF);
    if (o == 0) preCur[0] = 0.;
    for (size_t e = 0; e < p.pre.size(); ++e) {
      const ColEntry& en = p.pre[e];
      int32_t* ptr = ptrs ? &P.pre[(size_t) o * p.nPre + en.dst] : nullptr;
      if (en.kind == CE_SILENT) comb (preCur[en.dst], preCur[en.src] + E->preW[e], ptr, (int) e);
      else if (en.tok == tok) comb (preCur[en.dst], prePrev[en.src] + E->preW[e], ptr, (int) e);
    }
    std::fill (bCur.begin(), bCur.end(), NINF);
    for (int c = 0; c < p.nC; ++c) bCur[c] = preCur[p.carried[c]];
    for (int k = 0; k < p.K; ++k) {
      double* n = &cur[(size_t) k * p.nCell];
      const double* left = k ? &cur[(size_t) (k - 1) * p.nCell] : bCur.data();
      const double* diag = k ? &prev[(size_t) (k - 1) * p.nCell] : bPrev.data();
      const double* up = &prev[(size_t) k * p.nCell];
      for (int s = 0; s < p.nCell; ++s) n[s] = NINF;
      for (size_t gi = 0; gi < p.groups.size(); ++gi) {
        const ColGroup& g = p.groups[gi];
        const double src = g.type == CG_SILENT ? n[g.src] : g.type == CG_LEFT ? left[g.src] : g.type == CG_UP ? up[g.src] : diag[g.src];
        double w = 0.;
        if (g.slot >= 0) { if (g.emit) { if (tok < 1) continue; w = tabw (k, g.slot + tok - 1); } else w = tabw (k, g.slot); }
        comb (n[g.dst], src + w, ptrs ? &P.cell[((size_t) o * p.K + k) * p.nCell + g.dst] : nullptr, (int) gi);
      }
    }
    const double* X = &cur[(size_t) (p.K - 1) * p.nCell];
    std::fill (sufCur.begin(), sufCur.end(), NINF);
    auto ext = [&] (const double* cell, int leftSlot) { for (int s = 0; s < p.nCell; ++s) if (p.leftIdx[s] == leftSlot) return cell[s]; return NINF; };
    for (size_t e = 0; e < p.suf.size(); ++e) {
      const ColEntry& en = p.suf[e];
      double v;
      if (en.kind == CE_SILENT) v = sufCur[en.src] + E->sufW[e];
      else if (en.kind == CE_EXT_CUR) v = ext (X, en.src) + E->sufW[e];
      else if (en.tok != tok) continue;
      else v = (en.kind == CE_EMIT ? sufPrev[en.src] : ext (xPrev.data(), en.src)) + E->sufW[e];
      comb (sufCur[en.dst], v, ptrs ? &P.suf[(size_t) o * p.nSuf + en.dst] : nullptr, (int) e);
    }
    for (int s = 0; s < p.nCell; ++s) xPrev[s] = X[s];
    prev.swap (cur); bPrev = bCur; prePrev = preCur; sufPrev = sufCur;
  }
  *result = sufPrev[p.nSuf - 1];
  if (ptrs) { path->clear(); if (*result > NINF) return col_walk (p, y, Lo, P, *path); }
  return 0;
}

}  // namespace mb
