// mb_big.cu -- the big engine: machine-specialised Forward sweep (scaled linear domain) for MID-SIZE machines,
// tens to hundreds of states -- composed transducers such as prot2dna => dnapsw (308 states, 716 transition
// groups), SURVEY.md section 8 config 4 -- over full two-dimensional matrices.
//
//   reference                                              here
//   MappedForwardMatrix::fill / logLike  forward.defs.h:22-55   mb_k_big_forward (generated, NVRTC, sm_100a)
//
// The wide engine (mb_wide.cu) interprets such a machine from tables with a group of lanes per cell and
// spends ~75 thread-instructions per transition on decode, flags, gathers and level barriers (150 GCUPS on
// prot2dna => dnapsw, FP64 pipe 6 % busy).  Here the machine is written out the way mb_jit.cu does for small
// machines -- one multiply-add per transition group, straight-line, in state order -- but with a THREAD PER
// CELL (lane = matrix column, mb_big_skeleton.h) and the cell's long-lived states in shared memory instead
// of registers: the states insert groups read from the cell above sit in the lane's column of a
// shared-memory array, the few that delete / match groups read from the cell to the left arrive by shuffle,
// silent weights are constant-memory operands, emission weights token-indexed shared-memory tables.
// Transition groups = all transitions between one (source, destination) of one kind, weight looked up by
// token (0 where no transition carries that label), as in mb_jit.cu.
//
// Reached through the wide engine (wide_forward) for batches of full matrices; envelopes, Viterbi, and pairs
// the scaled sweep flags stay with the wide engine.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <sstream>
#include <tuple>

#include "mb_internal.h"
#include "mb_big_skeleton.h"

namespace mb {

struct BigGroup { int self, type, other, rank; int emitOff = -1, silIdx = -1, tableSize = 1; std::vector<std::pair<int, int64_t>> entries; };      // (label, transition)

struct BigEngine {
  std::vector<BigGroup> groups;      // by (destination, kind, source, rank): the reference's candidate order
  std::vector<int> liveU, liveL;     // sources of insert groups; sources of delete / match groups
  // Linear-domain normalisation, as in mb_jit.cu (Program::unitSlot): value'(d) = value(d) / sigma_d with sigma_d = w_u sigma_src(u)
  // for the state's first silent group u makes that group a plain copy (prot2dna => dnapsw: 716 multiply-adds per cell become
  // ~450); every other weight is scaled by sigma_src / sigma_self on the host, the result carries log sigma of the end state.
  std::vector<int> unitGroup;        // per state: index into groups, or -1
  double resLog = 0;
  // FOLDED live-up values (linear sweep only).  The insert groups u -> d of one destination are usually PROPORTIONAL:
  // w(u -> d, b) = c_u e(b) for every token b -- in a composed machine the emission belongs to the destination, the factor to
  // the transition (prot2dna => dnapsw: 144 insert groups into 74 destinations, every destination's groups proportional).
  // Then sum_u u(row above) w(u -> d, b) = e(b) F with F = sum_u c_u u, and what has to cross rows is F, one value per
  // CLASS (destination, direction of e), not one per source state: 74 values per lane in shared memory instead of 139, two
  // loads less per group, and twice the warps per SM.  The classes depend on the weights' ratios, so they are found
  // numerically when the engine is prepared and checked again when the weights change (big_update_weights asks for the
  // engine to be rebuilt if the partition moved).  The max-plus sweeps do not fold: (u + c) + e and u + (c + e) round differently.
  struct FoldClass { int dst, emitOffLin; std::vector<std::pair<int, int>> members; };      // (group index, fold-factor slot; -1: factor one, the representative)
  std::vector<FoldClass> classes;
  std::vector<int> groupClass;       // per group: its class (insert groups), or -1
  std::vector<int> emitOffLin;       // per group: offset in the linear emission table (match / delete groups), or -1
  int nEmitLin = 0, nFold = 0, threadsLin = 128;
  void* dFold = nullptr;             // __constant__ mb_big_fold in the module
  size_t smemBytesLin = 0;
  int nEmit = 0, nSil = 0, threads = 128;
  std::string source;
  void* mod = nullptr;
  void* kForward = nullptr;
  void* kViterbi = nullptr;
  void* kViterbiScore = nullptr;
  void* dSil = nullptr;              // __constant__ mb_big_sil in the module (linear weights)
  void* dSilLog = nullptr;           // __constant__ mb_big_sil_log
  double* dEmit = nullptr;
  double* dEmitLog = nullptr;
  // Viterbi back-pointers: state d's field is bits[d] wide at (word[d], shift[d]); it holds the index of the winning
  // group among the state's groups [groupStart[d], groupStart[d+1])
  std::vector<int> ptrWord, ptrShift, ptrBits, groupStart;
  int nPtrWords = 1;
  int32_t* dPlan = nullptr;          // traceback tables: see BigTbPlan
  int blocksPerSMV = 1, blocksPerSMVS = 1;
  size_t smemBytes = 0;
  int blocksPerSM = 1, numSMs = 148;
  bool linearOK = false;
};

static BigEngine* be (const mb_machine* m) { return static_cast<BigEngine*> (m->big); }

static int big_type (int a, int b) { return a ? (b ? T_MATCH : T_DELETE) : (b ? T_INSERT : T_SILENT); }

static void big_plan (const mb_machine* m, BigEngine& B) {
  std::map<std::tuple<int, int, int, int>, BigGroup> g;
  std::map<std::tuple<int, int, int, int>, int> seen;
  for (int64_t t = 0; t < m->T; ++t) {
    const int type = big_type (m->in[t], m->out[t]);
    if (type == T_SILENT && m->dst[t] <= m->src[t]) continue;      // only possible on state 0 (machine.cpp:759); contributes nothing
    const int li = type == T_MATCH ? (m->in[t] - 1) * m->nOut + (m->out[t] - 1) : type == T_DELETE ? m->in[t] - 1 : type == T_INSERT ? m->out[t] - 1 : 0;
    const int rank = seen[std::make_tuple ((int) m->dst[t], type, (int) m->src[t], li)]++;
    BigGroup& gr = g[std::make_tuple ((int) m->dst[t], type, (int) m->src[t], rank)];
    gr.self = m->dst[t]; gr.type = type; gr.other = m->src[t]; gr.rank = rank;
    gr.entries.push_back ({ li, t });
  }
  B.groups.clear();
  B.nEmit = B.nSil = 0;
  std::vector<char> isU ((size_t) m->S, 0), isL ((size_t) m->S, 0);
  for (auto& kv: g) {
    BigGroup gr = kv.second;
    gr.tableSize = gr.type == T_MATCH ? m->nIn * m->nOut : gr.type == T_DELETE ? m->nIn : gr.type == T_INSERT ? m->nOut : 1;
    if (gr.type == T_SILENT) gr.silIdx = B.nSil++;
    else { gr.emitOff = B.nEmit; B.nEmit += gr.tableSize; }
    if (gr.type == T_INSERT) isU[gr.other] = 1;
    if (gr.type == T_DELETE || gr.type == T_MATCH) isL[gr.other] = 1;
    B.groups.push_back (gr);
  }
  B.liveU.clear(); B.liveL.clear();
  for (int s = 0; s < m->S; ++s) { if (isU[s]) B.liveU.push_back (s); if (isL[s]) B.liveL.push_back (s); }
  B.unitGroup.assign ((size_t) m->S, -1);
  if (!m->opt.get ("jit_no_norm", 0))
    for (size_t gi = 0; gi < B.groups.size(); ++gi)
      if (B.groups[gi].type == T_SILENT && B.unitGroup[B.groups[gi].self] < 0) B.unitGroup[B.groups[gi].self] = (int) gi;
  // fold classes of the insert groups, by destination: a group joins the first class of its destination whose representative's
  // token vector it is a multiple of (same tokens present, constant log-ratio), else it opens a class
  {
    B.classes.clear();
    B.groupClass.assign (B.groups.size(), -1);
    B.emitOffLin.assign (B.groups.size(), -1);
    B.nEmitLin = 0; B.nFold = 0;
    const bool fold = !m->opt.get ("big_no_fold", 0);
    auto vec = [&] (const BigGroup& gr) { std::vector<double> v ((size_t) gr.tableSize, -INFINITY); for (auto& e: gr.entries) v[e.first] = m->lw[e.second]; return v; };
    for (size_t gi = 0; gi < B.groups.size(); ++gi) {
      const BigGroup& gr = B.groups[gi];
      if (gr.type == T_SILENT) continue;
      if (gr.type != T_INSERT) { B.emitOffLin[gi] = B.nEmitLin; B.nEmitLin += gr.tableSize; continue; }
      const std::vector<double> v = vec (gr);
      int found = -1;
      for (size_t c = 0; c < B.classes.size() && found < 0 && fold; ++c) {
        if (B.classes[c].dst != gr.self) continue;
        const std::vector<double> r = vec (B.groups[B.classes[c].members[0].first]);
        bool same = true, any = false;
        double ratio = 0;
        for (size_t q = 0; q < v.size() && same; ++q) {
          if ((v[q] > -INFINITY) != (r[q] > -INFINITY)) same = false;
          else if (v[q] > -INFINITY) {
            if (!std::isfinite (v[q]) || !std::isfinite (r[q])) same = false;
            else if (!any) { ratio = v[q] - r[q]; any = true; }
            else if (std::fabs ((v[q] - r[q]) - ratio) > 1e-12 * std::max (1.0, std::fabs (ratio))) same = false;
          }
        }
        if (same && any) found = (int) c;
      }
      if (found < 0) {
        BigEngine::FoldClass fc;
        fc.dst = gr.self; fc.emitOffLin = B.nEmitLin; B.nEmitLin += gr.tableSize;
        fc.members.push_back (std::make_pair ((int) gi, -1));
        B.classes.push_back (fc);
        found = (int) B.classes.size() - 1;
      } else B.classes[found].members.push_back (std::make_pair ((int) gi, B.nFold++));
      B.groupClass[gi] = found;
    }
  }
  // pointer fields, packed greedily into 32-bit words (no field straddles a word)
  B.groupStart.assign ((size_t) m->S + 1, 0);
  for (auto& gr: B.groups) B.groupStart[gr.self + 1]++;
  for (int s = 0; s < m->S; ++s) B.groupStart[s + 1] += B.groupStart[s];
  B.ptrWord.assign ((size_t) m->S, 0); B.ptrShift.assign ((size_t) m->S, 0); B.ptrBits.assign ((size_t) m->S, 0);
  int word = 0, used = 0;
  for (int s = 0; s < m->S; ++s) {
    const int n = B.groupStart[s + 1] - B.groupStart[s];
    int bt = 0; while ((1 << bt) < n) ++bt;
    if (bt == 0) continue;
    if (used + bt > 32) { ++word; used = 0; }
    B.ptrWord[s] = word; B.ptrShift[s] = used; B.ptrBits[s] = bt;
    used += bt;
  }
  B.nPtrWords = word + 1;
}

bool big_supported (const mb_machine* m, std::string* why) {
  auto no = [&] (const char* w) { if (why) *why = w; return false; };
  if (m->opt.get ("no_big", 0)) return no ("big engine: disabled (option no_big)");
  if (m->S <= 16) return no ("big engine: small machines belong to the JIT engine");
  if (m->S > 1024 || m->T > 65536) return no ("big engine: more than 1024 states or 65536 transitions");
  if (m->nIn == 0 || m->nOut == 0) return no ("big engine: no two-dimensional matrices without both alphabets");
  BigEngine B;
  big_plan (m, B);
  if (B.groups.size() > 6000) return no ("big engine: more than 6000 transition groups");
  if (B.nSil > 3900) return no ("big engine: silent weights (linear and log copies) exceed the 64 KB of constant memory");
  if (B.liveL.size() > 24) return no ("big engine: more than 24 states cross a column boundary");
  const size_t smem = (size_t) (((B.nEmit + 1) & ~1) + 4 * (B.liveU.size() * 32 + 16 * std::max<size_t> (B.liveL.size(), 1))) * 8;
  if (smem > 220 * 1024) return no ("big engine: emission tables and live states do not fit in shared memory");
  return true;
}

static void big_generate (const mb_machine* m, BigEngine& B) {
  big_plan (m, B);
  const int S = m->S, nLL = std::max<int> ((int) B.liveL.size(), 1);
  // as many warps per CTA (one CTA per SM) as shared memory holds: the emission tables once, the live-up states per warp
  {
    int warps = 8;      // 255 registers per thread: at most 8 warps per SM
    if (m->opt.has ("big_warps")) warps = std::max (1, std::min (8, m->opt.get ("big_warps", 8)));
    // (192 KB, not all 227: what is left is the L1 that holds the spilled registers -- prot2dna => dnapsw ran 3 % faster with 4 warps than with 5)
    int warpsLin = warps;
    const size_t cap = (size_t) std::max (48, std::min (227, m->opt.get ("big_smem_kb", 192))) * 1024;
    while (warps > 1 && (size_t) (((std::max (B.nEmit, 1) + 1) & ~1) + warps * ((int) B.liveU.size() * 32 + 16 * nLL)) * 8 > cap) --warps;
    while (warpsLin > 1 && (size_t) (((std::max (B.nEmitLin, 1) + 1) & ~1) + warpsLin * ((int) B.classes.size() * 32 + 16 * nLL)) * 8 > cap) --warpsLin;
    B.threads = 32 * warps;
    B.threadsLin = 32 * warpsLin;
  }
  std::vector<int> uIdx ((size_t) S, -1), lIdx ((size_t) S, -1);
  for (size_t q = 0; q < B.liveU.size(); ++q) uIdx[B.liveU[q]] = (int) q;
  for (size_t q = 0; q < B.liveL.size(); ++q) lIdx[B.liveL[q]] = (int) q;
  std::ostringstream o;
  o << "// generated by machineboss_b200 (mb_big.cu) for a machine with " << S << " states, " << m->T << " transitions, " << B.groups.size() << " transition groups\n";
  o << "typedef unsigned char uint8_t;\ntypedef int int32_t;\ntypedef long long int64_t;\n";
  o << "#define MB_S " << S << "\n#define MB_NLU " << B.liveU.size() << "\n#define MB_NLL " << nLL << "\n#define MB_NEMIT " << std::max (B.nEmit, 1)
    << "\n#define MB_BIG_THREADS " << B.threads << "\n";
  o << "#define MB_NLU_LIN " << B.classes.size() << "\n#define MB_NEMIT_LIN " << std::max (B.nEmitLin, 1) << "\n#define MB_BIG_THREADS_LIN " << B.threadsLin << "\n";
  {      // which emission-table entries carry a transition (the others stay 0 / -inf): lets a host-side harness fill the tables
    std::string present ((size_t) std::max (B.nEmit, 1), '0');
    for (auto& gr: B.groups) if (gr.type != T_SILENT) for (auto& e: gr.entries) present[(size_t) gr.emitOff + e.first] = '1';
    o << "// MB_EMIT_PRESENT " << present << "\n// MB_NSIL " << B.nSil << "\n";
    std::string presentLin ((size_t) std::max (B.nEmitLin, 1), '0');      // the sums' table: match / delete groups, and one vector per fold class (its representative's)
    for (size_t g = 0; g < B.groups.size(); ++g) if (B.emitOffLin[g] >= 0) for (auto& e: B.groups[g].entries) presentLin[(size_t) B.emitOffLin[g] + e.first] = '1';
    for (auto& fc: B.classes) for (auto& e: B.groups[fc.members[0].first].entries) presentLin[(size_t) fc.emitOffLin + e.first] = '1';
    o << "// MB_EMIT_PRESENT_LIN " << presentLin << "\n// MB_NFOLD " << B.nFold << "\n";
  }
  o << "#define MB_NPW " << B.nPtrWords << "\n";
  o << "__constant__ double mb_big_sil[" << std::max (B.nSil, 1) << "];\n__constant__ double mb_big_sil_log[" << std::max (B.nSil, 1) << "];\n";
  o << "__constant__ double mb_big_fold[" << std::max (B.nFold, 1) << "];      // factors of the folded live-up sums (BigEngine::classes)\n\n";
  // the cell: live-up states read from (and written back to) the lane's column of `up`, left / diagonal cells' states in L / D
  o << "__device__ __forceinline__ void mb_big_cell (double* __restrict__ up, const double (&L)[MB_NLL], const double (&D)[MB_NLL], double (&Lo)[MB_NLL], "
       "const int a, const int b, const bool origin, const double* __restrict__ E, double& res) {\n";
  std::vector<char> loaded ((size_t) S, 0);
  size_t gi = 0;
  // what each state contributes to the folded sums: (class, factor slot)
  std::vector<std::vector<std::pair<int, int>>> foldsOf ((size_t) S);
  for (size_t c = 0; c < B.classes.size(); ++c) for (auto& mem: B.classes[c].members) foldsOf[B.groups[mem.first].other].push_back (std::make_pair ((int) c, mem.second));
  std::vector<char> classUsed (B.classes.size(), 0), classStarted (B.classes.size(), 0);
  // a class's sum is complete after its last member's source state; it is stored then (the OLD sum read into a register first
  // if the class's destination comes later in the state order), so that it does not occupy a register to the end of the cell
  // (measured on B200, config 4: storing early costs the sums 12 % -- 234 registers become 255 -- while it gains the max-plus
  // sweeps 3 - 49 %; option big_early_store turns it on for the sums too)
  const bool earlyStore = m->opt.get ("big_early_store", 0) != 0;
  std::vector<char> classStored (B.classes.size(), 0);
  std::vector<int> classLast (B.classes.size(), -1);
  for (size_t c = 0; c < B.classes.size(); ++c) for (auto& mem: B.classes[c].members) classLast[c] = std::max (classLast[c], B.groups[mem.first].other);
  for (int d = 0; d < S; ++d) {
    bool first = true;
    if (B.unitGroup[d] >= 0) { o << "  double n" << d << " = n" << B.groups[B.unitGroup[d]].other << ";\n"; first = false; }      // the unit group: a copy
    for (; gi < B.groups.size() && B.groups[gi].self == d; ++gi) {
      if ((int) gi == B.unitGroup[d]) continue;
      const BigGroup& gr = B.groups[gi];
      std::ostringstream src, w;
      if (gr.type == T_INSERT) {      // once per class: the folded sum of the row above times the class's token vector
        const int c = B.groupClass[gi];
        if (classUsed[c] == 2) continue;
        if (!classUsed[c]) o << "  const double F" << c << " = up[" << c << " * 32];\n";
        classUsed[c] = 2;
        src << "F" << c; w << "E[" << B.classes[c].emitOffLin << " + b]";
      } else if (gr.type == T_DELETE) { src << "L[" << lIdx[gr.other] << "]"; w << "E[" << B.emitOffLin[gi] << " + a]"; }
      else if (gr.type == T_MATCH) { src << "D[" << lIdx[gr.other] << "]"; w << "E[" << B.emitOffLin[gi] << " + a * " << m->nOut << " + b]"; }
      else { src << "n" << gr.other; w << "mb_big_sil[" << gr.silIdx << "]"; }
      if (first) { o << "  double n" << d << " = " << src.str() << " * " << w.str() << ";\n"; first = false; }
      else o << "  n" << d << " = fma (" << src.str() << ", " << w.str() << ", n" << d << ");\n";
    }
    if (first) o << "  double n" << d << " = 0.0;\n";
    if (d == 0) o << "  if (origin) n0 = 1.0;\n";
    for (auto& fo: foldsOf[d]) {      // n_d is final: add it to the sums it belongs to (its register can be released)
      std::ostringstream term;
      if (fo.second < 0) term << "n" << d; else term << "n" << d << " * mb_big_fold[" << fo.second << "]";
      if (!classStarted[fo.first]) { o << "  double f" << fo.first << " = " << term.str() << ";\n"; classStarted[fo.first] = 1; }
      else if (fo.second < 0) o << "  f" << fo.first << " += n" << d << ";\n";
      else o << "  f" << fo.first << " = fma (n" << d << ", mb_big_fold[" << fo.second << "], f" << fo.first << ");\n";
      const int c = fo.first;
      if (earlyStore && classLast[c] == d) {      // complete: store (a class may list the same source twice only through different groups; the last one closes it)
        bool lastOfState = true;
        for (auto& later: foldsOf[d]) if (&later > &fo && later.first == c) lastOfState = false;
        if (lastOfState) {
          if (!classUsed[c] && B.classes[c].dst > d) { o << "  const double F" << c << " = up[" << c << " * 32];\n"; classUsed[c] = 1; }
          if (classUsed[c] || B.classes[c].dst <= d) { o << "  up[" << c << " * 32] = f" << c << ";\n"; classStored[c] = 1; }
        }
      }
    }
  }
  for (size_t c = 0; c < B.classes.size(); ++c) if (!classStored[c]) o << "  up[" << c << " * 32] = f" << c << ";\n";
  for (size_t q = 0; q < B.liveL.size(); ++q) o << "  Lo[" << q << "] = n" << B.liveL[q] << ";\n";
  if (B.liveL.empty()) o << "  Lo[0] = 0.0;\n";
  o << "  res = n" << S - 1 << ";\n}\n\n";
  // the same cell in the max-plus semiring (viterbi.cpp:30-39): candidates of a state in the reference's order (match,
  // delete, insert, silent sources; each by source state, then transition index), strict '<' keeps the first maximum
  // (dpmatrix.defs.h:171-174); pw receives the packed pointers
  o << "__device__ __forceinline__ void mb_big_cell_vit (double* __restrict__ up, const double (&L)[MB_NLL], const double (&D)[MB_NLL], double (&Lo)[MB_NLL], "
       "const int a, const int b, const bool origin, const double* __restrict__ E, double& res, unsigned (&pw)[MB_NPW]) {\n";
  o << "  const double NI = __longlong_as_double (0xfff0000000000000LL);\n";
  for (int wd = 0; wd < B.nPtrWords; ++wd) o << "  unsigned pw" << wd << " = 0u;\n";
  std::fill (loaded.begin(), loaded.end(), 0);
  // A live-up state's new value goes to shared memory as soon as it is final -- and its pointer into the packed word -- so that
  // neither stays in a register to the end of the cell (139 doubles did: 584 - 856 bytes of spills per thread).  A consumer
  // further down the state order still needs the OLD value: it is read into a register just before the store.
  std::vector<int> lastConsumer ((size_t) S, -1);
  for (auto& gr: B.groups) if (gr.type == T_INSERT) lastConsumer[gr.other] = std::max (lastConsumer[gr.other], gr.self);
  gi = 0;
  for (int d = 0; d < S; ++d) {
    int k = 0;
    for (; gi < B.groups.size() && B.groups[gi].self == d; ++gi, ++k) {
      const BigGroup& gr = B.groups[gi];
      std::ostringstream src, w;
      if (gr.type == T_INSERT) {
        if (!loaded[gr.other]) { o << "  const double u" << gr.other << " = up[" << uIdx[gr.other] << " * 32];\n"; loaded[gr.other] = 1; }
        src << "u" << gr.other; w << "E[" << gr.emitOff << " + b]";
      } else if (gr.type == T_DELETE) { src << "L[" << lIdx[gr.other] << "]"; w << "E[" << gr.emitOff << " + a]"; }
      else if (gr.type == T_MATCH) { src << "D[" << lIdx[gr.other] << "]"; w << "E[" << gr.emitOff << " + a * " << m->nOut << " + b]"; }
      else { src << "n" << gr.other; w << "mb_big_sil_log[" << gr.silIdx << "]"; }
      if (k == 0) { o << "  double n" << d << " = " << src.str() << " + " << w.str() << ";\n"; if (B.ptrBits[d]) o << "  unsigned p" << d << " = 0u;\n"; }
      else o << "  { const double t = " << src.str() << " + " << w.str() << "; if (n" << d << " < t) { n" << d << " = t; p" << d << " = " << k << "u; } }\n";
    }
    if (k == 0) o << "  double n" << d << " = NI;\n";
    if (d == 0) o << "  if (origin) n0 = 0.0;\n";
    if (k > 0 && B.ptrBits[d]) o << "  pw" << B.ptrWord[d] << " |= p" << d << " << " << B.ptrShift[d] << ";\n";
    if (uIdx[d] >= 0) {
      if (lastConsumer[d] > d && !loaded[d]) { o << "  const double u" << d << " = up[" << uIdx[d] << " * 32];\n"; loaded[d] = 1; }
      o << "  up[" << uIdx[d] << " * 32] = n" << d << ";\n";
    }
  }
  for (size_t q = 0; q < B.liveL.size(); ++q) o << "  Lo[" << q << "] = n" << B.liveL[q] << ";\n";
  if (B.liveL.empty()) o << "  Lo[0] = NI;\n";
  for (int wd = 0; wd < B.nPtrWords; ++wd) o << "  pw[" << wd << "] = pw" << wd << ";\n";
  o << "  res = n" << S - 1 << ";\n}\n";
  o << kBigSkeleton;
  B.source = o.str();
}

int big_compile_check (const mb_machine* m, std::string* log) {
  std::string why;
  if (!big_supported (m, &why)) { set_error ("machine not eligible for the big engine: " + why); return 1; }
  BigEngine B;
  big_generate (m, B);
  std::vector<char> cubin;
  return rt_compile (B.source, ".big.cu", cubin, log);
}

void big_destroy (mb_machine* m) {
  BigEngine* B = be (m);
  if (!B) return;
  if (B->mod) rt_unload (B->mod);
  if (B->dEmit) cudaFree (B->dEmit);
  if (B->dEmitLog) cudaFree (B->dEmitLog);
  if (B->dPlan) cudaFree (B->dPlan);
  delete B;
  m->big = nullptr;
}

int big_update_weights (mb_machine* m) {
  BigEngine* B = be (m);
  if (!B) return 0;
  std::vector<double> emit ((size_t) std::max (B->nEmitLin, 1), 0.), sil ((size_t) std::max (B->nSil, 1), 0.), foldF ((size_t) std::max (B->nFold, 1), 0.);
  std::vector<double> emitLog ((size_t) std::max (B->nEmit, 1), -INFINITY), silLog (sil.size(), -INFINITY);
  bool moved = false;      // the fold classes no longer fit the weights: the engine has to be generated again
  bool ok = true;
  const double lim = 24.0 * 0.6931471805599453;
  std::vector<double> ls ((size_t) m->S, 0.);      // log sigma per state; a silent group's source is an earlier state
  for (int d = 0; d < m->S; ++d) {
    if (B->unitGroup[d] < 0) continue;
    const BigGroup& u = B->groups[B->unitGroup[d]];
    const double w = m->lw[u.entries[0].second];
    if (!std::isfinite (w)) { ok = false; continue; }      // a unit weight of 0 cannot be divided out: the wide engine's sweeps take the machine
    ls[d] = w + ls[u.other];
    if (std::fabs (ls[d]) > 100. * 0.6931471805599453) ok = false;
  }
  B->resLog = ls[m->S - 1];
  auto scaledOf = [&] (const BigGroup& gr, double lw) { return lw > -INFINITY ? lw + ls[gr.other] - ls[gr.self] : -INFINITY; };      // the linear sweep's weight, in normalised units
  for (size_t gi = 0; gi < B->groups.size(); ++gi) {
    const BigGroup& gr = B->groups[gi];
    for (auto& e: gr.entries) {
      const double lw = m->lw[e.second];
      if (std::isnan (lw) || lw == INFINITY || (std::isfinite (lw) && std::fabs (lw) > lim)) ok = false;
      const double scaled = scaledOf (gr, lw);
      if (std::isfinite (scaled) && std::fabs (scaled) > 2 * lim) ok = false;
      if (gr.type == T_SILENT) { sil[gr.silIdx] = std::exp (scaled); silLog[gr.silIdx] = lw; }
      else {
        emitLog[(size_t) gr.emitOff + e.first] = lw;
        if (B->emitOffLin[gi] >= 0) emit[(size_t) B->emitOffLin[gi] + e.first] = std::exp (scaled);
      }
    }
  }
  // fold classes: the representative's vector is the class's token table; every other member is a constant multiple of it
  for (auto& fc: B->classes) {
    const BigGroup& rep = B->groups[fc.members[0].first];
    std::vector<double> r ((size_t) rep.tableSize, -INFINITY);
    for (auto& e: rep.entries) { r[e.first] = scaledOf (rep, m->lw[e.second]); emit[(size_t) fc.emitOffLin + e.first] = std::exp (r[e.first]); }
    for (size_t q = 1; q < fc.members.size(); ++q) {
      const BigGroup& gr = B->groups[fc.members[q].first];
      std::vector<double> v ((size_t) gr.tableSize, -INFINITY);
      for (auto& e: gr.entries) v[e.first] = scaledOf (gr, m->lw[e.second]);
      bool any = false;
      double ratio = 0;
      for (size_t t = 0; t < v.size(); ++t) {
        if ((v[t] > -INFINITY) != (r[t] > -INFINITY)) moved = true;
        else if (v[t] > -INFINITY) {
          if (!any) { ratio = v[t] - r[t]; any = true; }
          else if (!(std::fabs ((v[t] - r[t]) - ratio) <= 1e-9 * std::max (1.0, std::fabs (ratio)))) moved = true;
        }
      }
      if (!any) moved = true;
      if (std::fabs (ratio) > 2 * lim) ok = false;
      foldF[fc.members[q].second] = std::exp (ratio);
    }
  }
  B->linearOK = ok;
  if (moved) return 2;
  MB_CUDA (cudaSetDevice (m->device));
  MB_CUDA (cudaMemcpy (B->dEmit, emit.data(), emit.size() * 8, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (B->dSil, sil.data(), sil.size() * 8, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (B->dEmitLog, emitLog.data(), emitLog.size() * 8, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (B->dSilLog, silLog.data(), silLog.size() * 8, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (B->dFold, foldF.data(), foldF.size() * 8, cudaMemcpyHostToDevice));
  return 0;
}

int big_prepare (mb_machine* m) {
  BigEngine* B = new BigEngine;
  m->big = B;
  big_generate (m, *B);
  std::vector<char> cubin;
  if (rt_compile (B->source, ".big.cu", cubin, nullptr)) return 1;
  MB_CUDA (cudaSetDevice (m->device));
  if (rt_load (cubin, &B->mod) || rt_function (B->mod, "mb_k_big_forward", &B->kForward)
      || rt_function (B->mod, "mb_k_big_viterbi", &B->kViterbi) || rt_function (B->mod, "mb_k_big_viterbi_score", &B->kViterbiScore)) return 1;
  size_t bytes = 0;
  if (rt_global (B->mod, "mb_big_sil", &B->dSil, &bytes) || rt_global (B->mod, "mb_big_sil_log", &B->dSilLog, &bytes) || rt_global (B->mod, "mb_big_fold", &B->dFold, &bytes)) return 1;
  MB_CUDA (cudaMalloc (&B->dEmit, (size_t) std::max (B->nEmitLin, 1) * 8));
  MB_CUDA (cudaMalloc (&B->dEmitLog, (size_t) std::max (B->nEmit, 1) * 8));
  {      // traceback tables, one int32 array: [S+1] groupStart | [S] word | [S] shift | [S] bits | [G] type | [G] source | [G] idOff | ids
    std::vector<int32_t> plan;
    for (int v: B->groupStart) plan.push_back (v);
    for (int v: B->ptrWord) plan.push_back (v);
    for (int v: B->ptrShift) plan.push_back (v);
    for (int v: B->ptrBits) plan.push_back (v);
    for (auto& gr: B->groups) plan.push_back (gr.type);
    for (auto& gr: B->groups) plan.push_back (gr.other);
    std::vector<int32_t> ids;
    for (auto& gr: B->groups) { plan.push_back ((int32_t) ids.size()); ids.resize (ids.size() + gr.tableSize, -1); for (auto& e: gr.entries) ids[ids.size() - gr.tableSize + e.first] = (int32_t) e.second; }
    plan.insert (plan.end(), ids.begin(), ids.end());
    MB_CUDA (cudaMalloc (&B->dPlan, plan.size() * 4));
    MB_CUDA (cudaMemcpy (B->dPlan, plan.data(), plan.size() * 4, cudaMemcpyHostToDevice));
  }
  MB_CUDA (cudaDeviceGetAttribute (&B->numSMs, cudaDevAttrMultiProcessorCount, m->device));
  const int warps = B->threads / 32, nLL = std::max<int> ((int) B->liveL.size(), 1);
  B->smemBytes = (size_t) (((std::max (B->nEmit, 1) + 1) & ~1) + warps * ((int) B->liveU.size() * 32 + 16 * nLL)) * 8;
  B->smemBytesLin = (size_t) (((std::max (B->nEmitLin, 1) + 1) & ~1) + (B->threadsLin / 32) * ((int) B->classes.size() * 32 + 16 * nLL)) * 8;
  if (rt_prepare (B->kForward, B->threadsLin, B->smemBytesLin, &B->blocksPerSM) || rt_prepare (B->kViterbi, B->threads, B->smemBytes, &B->blocksPerSMV)
      || rt_prepare (B->kViterbiScore, B->threads, B->smemBytes, &B->blocksPerSMVS)) return 1;
  if (B->blocksPerSM < 1 || B->blocksPerSMV < 1 || B->blocksPerSMVS < 1) { set_error ("big engine: a kernel does not fit on an SM"); return 1; }
  if (m->opt.get ("verbose", 0))
    fprintf (stderr, "big engine: S=%d groups=%zu (silent %d), live-up %zu (sums: %zu folded classes, %d warps per CTA; max-plus: %d), left-going %zu, emission table %d doubles, %zu / %zu B smem, %d CTA(s)/SM\n",
             m->S, B->groups.size(), B->nSil, B->liveU.size(), B->classes.size(), B->threadsLin / 32, B->threads / 32, B->liveL.size(), B->nEmit, B->smemBytesLin, B->smemBytes, B->blocksPerSM);
  const int rc = big_update_weights (m);
  if (rc == 2) { set_error ("big engine: the fold classes do not fit the weights they were built from"); return 1; }
  return rc;
}

bool big_wanted (const mb_machine* m, const mb_batch* b) {
  if (!m->big || !be (m)->linearOK || b->hasEnv) return false;
  return true;
}

struct MBBigArgsHost {      // must match struct MBBigArgs in the skeleton
  const uint8_t* x; const int64_t* xOff;
  const uint8_t* y; const int64_t* yOff;
  const int64_t* order; int64_t nWork; unsigned long long* counter;
  double* bnd; int64_t bndStride;
  double* result; int32_t* flag;
  const double* emit;
  unsigned* bp; const int64_t* bpOff;
  double resLog;
};

int big_forward (mb_machine* m, mb_batch* b, double* loglike) {
  BigEngine& B = *be (m);
  b->lastRedo = 0;
  if (b->nPairs == 0) return 0;
  std::vector<int64_t> order ((size_t) b->nPairs);
  for (int64_t k = 0; k < b->nPairs; ++k) order[k] = k;
  auto cost = [&] (int64_t k) { return (double) (b->xOff[k + 1] - b->xOff[k] + 1) * (double) (b->yOff[k + 1] - b->yOff[k] + 1); };
  std::stable_sort (order.begin(), order.end(), [&] (int64_t p, int64_t q) { return cost (p) > cost (q); });
  int64_t maxLo = 0;
  for (int64_t k = 0; k < b->nPairs; ++k) maxLo = std::max (maxLo, b->yOff[k + 1] - b->yOff[k]);
  const int warps = B.threadsLin / 32, nLL = std::max<int> ((int) B.liveL.size(), 1);
  // one CTA per SM as soon as there are that many pairs (warps pull pairs from a counter; with fewer pairs than warps the pairs
  // spread over all SMs instead of filling half of them: 592 pairs on 8-warp CTAs would otherwise occupy 74 SMs)
  const int64_t grid = std::max<int64_t> (1, std::min<int64_t> ((int64_t) B.numSMs * B.blocksPerSM, b->nPairs));
  const int64_t bndStride = 2 * (maxLo + 1) * (nLL + 1);
  b->wsOrderHoldsFull = false;
  int64_t* dOrder = (int64_t*) ws_reserve (b, WS_ORDER, order.size() * 8);
  unsigned long long* dCounter = (unsigned long long*) ws_reserve (b, WS_COUNTER, 8);
  double* dBnd = (double*) ws_reserve (b, WS_BND, (size_t) (grid * warps * bndStride) * 8);
  double* dRes = (double*) ws_reserve (b, WS_RESULT, (size_t) b->nPairs * 8);
  int32_t* dFlag = (int32_t*) ws_reserve (b, WS_FLAG, (size_t) b->nPairs * 4);
  if (!dOrder || !dCounter || !dBnd || !dRes || !dFlag) return 1;
  MB_CUDA (cudaMemcpyAsync (dOrder, order.data(), order.size() * 8, cudaMemcpyHostToDevice, b->stream));
  MB_CUDA (cudaMemsetAsync (dCounter, 0, 8, b->stream));
  MB_CUDA (cudaMemsetAsync (dFlag, 0, (size_t) b->nPairs * 4, b->stream));
  MBBigArgsHost A;
  A.x = b->dX; A.xOff = b->dXOff; A.y = b->dY; A.yOff = b->dYOff;
  A.order = dOrder; A.nWork = b->nPairs; A.counter = dCounter;
  A.bnd = dBnd; A.bndStride = bndStride;
  A.result = dRes; A.flag = dFlag; A.emit = B.dEmit;
  A.bp = nullptr; A.bpOff = nullptr;
  A.resLog = B.resLog;
  void* params[1] = { &A };
  if (timing_begin (b)) return 1;
  if (rt_launch (B.kForward, (unsigned) grid, (unsigned) B.threadsLin, B.smemBytesLin, b->stream, params)) return 1;
  std::vector<int32_t> flag ((size_t) b->nPairs);
  MB_CUDA (cudaMemcpyAsync (loglike, dRes, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost, b->stream));
  MB_CUDA (cudaMemcpyAsync (flag.data(), dFlag, flag.size() * 4, cudaMemcpyDeviceToHost, b->stream));
  MB_CUDA (cudaStreamSynchronize (b->stream));
  std::vector<int64_t> redo;
  for (int64_t k = 0; k < b->nPairs; ++k) if (flag[k] || !(loglike[k] > -INFINITY)) redo.push_back (k);
  if (m->opt.get ("big_debug", 0)) {
    int64_t nf[8] = { 0, 0, 0, 0, 0, 0, 0, 0 }, ninf = 0;
    for (int64_t k = 0; k < b->nPairs; ++k) { ++nf[flag[k] & 7]; if (!(loglike[k] > -INFINITY)) ++ninf; }
    fprintf (stderr, "big engine: %lld pairs, flags by reason mask 0..7: %lld %lld %lld %lld %lld %lld %lld %lld, -inf or nan results %lld, first results %.10g %.10g\n",
             (long long) b->nPairs, (long long) nf[0], (long long) nf[1], (long long) nf[2], (long long) nf[3], (long long) nf[4], (long long) nf[5], (long long) nf[6], (long long) nf[7],
             (long long) ninf, loglike[0], loglike[b->nPairs > 1 ? 1 : 0]);
  }
  int64_t launches = 1;
  if (!redo.empty()) {      // dangerous dynamic range, or no path at all: the wide engine's log-domain sweep decides
    if (wide_forward_log_subset (m, b, redo, dRes)) return 1;
    ++launches;
  }
  b->lastRedo = (int64_t) redo.size();
  if (timing_end (b, launches)) return 1;
  if (!redo.empty()) MB_CUDA (cudaMemcpy (loglike, dRes, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  return 0;
}

bool big_wanted_viterbi (const mb_machine* m, const mb_batch* b) { return m->big && !b->hasEnv; }

struct BigTbPlan {
  const int32_t* groupStart; const int32_t* word; const int32_t* shift; const int32_t* bits;
  const int32_t* type; const int32_t* source; const int32_t* idOff; const int32_t* ids;
  int32_t S, nOut, nWords;
};

// DPMatrix::traceBack (dpmatrix.defs.h:82-110) over the packed pointers of mb_k_big_viterbi, one thread per pair.
// out == nullptr: lengths only; otherwise the path is written start -> end at out[outOff[n] ..).
__global__ void big_traceback_kernel (BigTbPlan p, DevBatch b, const int64_t* __restrict__ order, int64_t nWork,
                                      const unsigned* __restrict__ bp, const int64_t* __restrict__ bpOff,
                                      const double* __restrict__ score, int64_t* __restrict__ lenOut, int32_t* __restrict__ out,
                                      const int64_t* __restrict__ outOff) {
  const int64_t n = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= nWork) return;
  const int64_t k = order[n];
  const uint8_t* x = b.x + b.xOff[k];
  const uint8_t* y = b.y + b.yOff[k];
  const int64_t Li = b.xOff[k + 1] - b.xOff[k], Lo = b.yOff[k + 1] - b.yOff[k];
  const int64_t nStrips = (Li + 32) / 32;
  const unsigned* base = bp + bpOff[n];
  int64_t len = 0;
  if (score[k] > -INFINITY) {      // boss.cpp:831
    const int64_t total = out ? lenOut[n] : 0;
    int64_t i = Li, o = Lo;
    int s = p.S - 1;
    while (i > 0 || o > 0 || s != 0) {
      const int g0 = p.groupStart[s], ng = p.groupStart[s + 1] - g0;
      if (ng == 0) break;      // cannot happen on a finite path
      int ptr = 0;
      if (p.bits[s]) {
        const unsigned w = base[(((o + (i & 31)) * nStrips + (i >> 5)) * p.nWords + p.word[s]) * 32 + (i & 31)];      // sweep order: the cell was stored at step o + lane
        ptr = (int) ((w >> p.shift[s]) & ((1u << p.bits[s]) - 1u));
      }
      if (ptr >= ng) break;
      const int g = g0 + ptr, type = p.type[g];
      const int a = i ? x[i - 1] - 1 : 0, c = o ? y[o - 1] - 1 : 0;
      const int li = type == T_MATCH ? a * p.nOut + c : type == T_DELETE ? a : type == T_INSERT ? c : 0;
      if (out) out[outOff[n] + total - 1 - len] = p.ids[p.idOff[g] + li];
      ++len;
      if (type == T_MATCH || type == T_DELETE) --i;
      if (type == T_MATCH || type == T_INSERT) --o;
      s = p.source[g];
      if (i < 0 || o < 0) break;
    }
  }
  if (!out) lenOut[n] = len;
}

int big_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen) {
  BigEngine& B = *be (m);
  if (b->nPairs == 0) return 0;
  const bool trace = pathLen != nullptr;
  std::vector<int64_t> order ((size_t) b->nPairs);
  for (int64_t k = 0; k < b->nPairs; ++k) order[k] = k;
  auto cost = [&] (int64_t k) { return (double) (b->xOff[k + 1] - b->xOff[k] + 1) * (double) (b->yOff[k + 1] - b->yOff[k] + 1); };
  std::stable_sort (order.begin(), order.end(), [&] (int64_t p, int64_t q) { return cost (p) > cost (q); });
  int64_t maxLo = 0;
  for (int64_t k = 0; k < b->nPairs; ++k) maxLo = std::max (maxLo, b->yOff[k + 1] - b->yOff[k]);
  const int warps = B.threads / 32, nLL = std::max<int> ((int) B.liveL.size(), 1);
  const int perSM = trace ? B.blocksPerSMV : B.blocksPerSMVS;
  const int64_t maxGrid = (int64_t) B.numSMs * perSM;
  const int64_t bndStride = 2 * (maxLo + 1) * (nLL + 1);
  b->wsOrderHoldsFull = false;
  unsigned long long* dCounter = (unsigned long long*) ws_reserve (b, WS_COUNTER, 8);
  double* dBnd = (double*) ws_reserve (b, WS_BND, (size_t) (maxGrid * warps * bndStride) * 8);
  double* dRes = (double*) ws_reserve (b, WS_RESULT2, (size_t) b->nPairs * 8);
  if (!dCounter || !dBnd || !dRes) return 1;
  MBBigArgsHost A;
  A.x = b->dX; A.xOff = b->dXOff; A.y = b->dY; A.yOff = b->dYOff;
  A.counter = dCounter; A.bnd = dBnd; A.bndStride = bndStride;
  A.result = dRes; A.flag = nullptr; A.emit = B.dEmitLog;
  A.bp = nullptr; A.bpOff = nullptr;
  A.resLog = 0;
  void* params[1] = { &A };
  auto launch = [&] (const std::vector<int64_t>& work, const int64_t* dOrder) {
    const int64_t grid = std::max<int64_t> (1, std::min<int64_t> (maxGrid, (int64_t) work.size()));
    A.order = dOrder; A.nWork = (int64_t) work.size();
    MB_CUDA (cudaMemsetAsync (dCounter, 0, 8, b->stream));
    return rt_launch (trace ? B.kViterbi : B.kViterbiScore, (unsigned) grid, (unsigned) B.threads, B.smemBytes, b->stream, params);
  };
  if (!trace) {
    int64_t* dOrder = (int64_t*) ws_reserve (b, WS_ORDER, order.size() * 8);
    if (!dOrder) return 1;
    MB_CUDA (cudaMemcpyAsync (dOrder, order.data(), order.size() * 8, cudaMemcpyHostToDevice, b->stream));
    if (timing_begin (b)) return 1;
    if (launch (order, dOrder)) return 1;
    if (timing_end (b, 1)) return 1;
    MB_CUDA (cudaMemcpy (score, dRes, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
    return 0;
  }
  // chunks of pairs whose pointers ((Lo+1) rows x strips x MB_NPW words x 32 lanes) fit in free memory
  size_t freeB = 0, totalB = 0;
  MB_CUDA (cudaMemGetInfo (&freeB, &totalB));
  const double budget = 0.75 * (double) freeB;
  BigTbPlan tp;
  {
    const int S = m->S, G = (int) B.groups.size();
    const int32_t* q = B.dPlan;
    tp.groupStart = q; q += S + 1; tp.word = q; q += S; tp.shift = q; q += S; tp.bits = q; q += S;
    tp.type = q; q += G; tp.source = q; q += G; tp.idOff = q; q += G; tp.ids = q;
    tp.S = S; tp.nOut = m->nOut; tp.nWords = B.nPtrWords;
  }
  int64_t launches = 0;
  double ms = 0;
  for (size_t c0 = 0; c0 < order.size();) {
    std::vector<int64_t> chunk, bpOff;
    double words = 0;
    size_t c1 = c0;
    for (; c1 < order.size(); ++c1) {
      const int64_t k = order[c1];
      const double need = (double) (b->yOff[k + 1] - b->yOff[k] + 32) * (double) ((b->xOff[k + 1] - b->xOff[k] + 32) / 32) * B.nPtrWords * 32;      // (Lo + 32) steps per strip
      if (need * 4 > budget) { set_error ("pair " + std::to_string (k) + " needs more device memory for its back-pointers than is free (" + std::to_string (need * 4) + " bytes)"); return 1; }
      if (!chunk.empty() && (words + need) * 4 > budget) break;
      chunk.push_back (k);
      bpOff.push_back ((int64_t) words);
      words += need;
    }
    // A pair is one warp's work from start to end, so a chunk costs as many "waves" as its pairs fill the resident warps:
    // when pairs remain for another chunk, cut this one back to whole waves (1000 pairs of which 840 fit: 592 + 408 are two
    // waves, 840 + 160 would be three)
    {
      const size_t resident = (size_t) maxGrid * warps;
      if (c1 < order.size() && chunk.size() > resident) {
        const size_t keep = chunk.size() / resident * resident;
        c1 = c0 + keep;
        words = (double) bpOff[keep];
        chunk.resize (keep); bpOff.resize (keep);
      }
    }
    c0 = c1;
    DevBuf dBp, dBpOff, dOrder, dLen, dOutOff;
    if (dBp.alloc ((size_t) words * 4) || dBpOff.alloc (bpOff.size() * 8) || dOrder.alloc (chunk.size() * 8) || dLen.alloc (chunk.size() * 8) || dOutOff.alloc (chunk.size() * 8)) return 1;
    MB_CUDA (cudaMemcpyAsync (dBpOff.p, bpOff.data(), bpOff.size() * 8, cudaMemcpyHostToDevice, b->stream));
    MB_CUDA (cudaMemcpyAsync (dOrder.p, chunk.data(), chunk.size() * 8, cudaMemcpyHostToDevice, b->stream));
    A.bp = dBp.as<unsigned>(); A.bpOff = dBpOff.as<int64_t>();
    if (timing_begin (b)) return 1;
    if (launch (chunk, dOrder.as<int64_t>())) return 1;
    const int64_t nWork = (int64_t) chunk.size();
    const unsigned tg = (unsigned) ((nWork + 63) / 64);
    big_traceback_kernel<<<tg, 64, 0, b->stream>>> (tp, b->dev, dOrder.as<int64_t>(), nWork, dBp.as<unsigned>(), dBpOff.as<int64_t>(), dRes, dLen.as<int64_t>(), nullptr, nullptr);
    MB_CUDA (cudaGetLastError());
    if (paths_place (b, chunk.data(), nWork, dLen.as<int64_t>(), dOutOff.as<int64_t>())) return 1;
    big_traceback_kernel<<<tg, 64, 0, b->stream>>> (tp, b->dev, dOrder.as<int64_t>(), nWork, dBp.as<unsigned>(), dBpOff.as<int64_t>(), dRes, dLen.as<int64_t>(), b->dPaths, dOutOff.as<int64_t>());
    MB_CUDA (cudaGetLastError());
    launches += 3;
    if (timing_end (b, launches)) return 1;
    ms += b->lastMs;
  }
  b->lastMs = ms;
  b->lastLaunches = launches;
  MB_CUDA (cudaMemcpy (score, dRes, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  return 0;
}

}  // namespace mb
