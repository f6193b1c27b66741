// mb_jit.cu -- the specialised engine for small machines (dnapsw, protpsw and the like).
//
// The reference interprets the machine through nested std::map lookups per cell-state
// (src/dpmatrix.h:101-115); its own code generator (src/compiler.cpp) shows what flattening that
// buys on a CPU.  Here the host turns the machine into straight-line CUDA -- one expression per
// (destination state, transition group) in the reference's candidate order -- puts it in front of
// the strip-kernel skeleton (mb_jit_skeleton.h) and compiles it with NVRTC for sm_100a the first
// time a machine structure is seen.  Weights are kernel arguments / shared-memory tables, so
// mb_machine_update_weights (one per EM iteration) never recompiles.
//
// A "slot" is one candidate of a state: all transitions between the same (source, destination)
// with the same kind (match / delete / insert / silent), i.e. one add + one log-sum-exp (or max)
// per cell, with the log-weight looked up by the cell's tokens.  Slots of a state are ordered like
// the reference's candidate list (kind, then other state, then transition index), which is what
// makes the Viterbi back-pointer tie-break identical (src/dpmatrix.defs.h:93-99,171-174).
#include <cuda.h>
#include <dlfcn.h>
#include <nvrtc.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <sstream>

#include "mb_internal.h"
#include "mb_jit_skeleton.h"

namespace mb {

// ---------------------------------------------------------------------------------------------
// driver API + NVRTC, resolved at run time so that the library loads on a machine without a GPU
// ---------------------------------------------------------------------------------------------
struct Driver {
  CUresult (*ModuleLoadData) (CUmodule*, const void*) = nullptr;
  CUresult (*ModuleUnload) (CUmodule) = nullptr;
  CUresult (*ModuleGetFunction) (CUfunction*, CUmodule, const char*) = nullptr;
  CUresult (*ModuleGetGlobal) (CUdeviceptr*, size_t*, CUmodule, const char*) = nullptr;
  CUresult (*LaunchKernel) (CUfunction, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, unsigned, CUstream, void**, void**) = nullptr;
  CUresult (*FuncSetAttribute) (CUfunction, CUfunction_attribute, int) = nullptr;
  CUresult (*FuncGetAttribute) (int*, CUfunction_attribute, CUfunction) = nullptr;
  CUresult (*OccupancyMaxActiveBlocksPerMultiprocessor) (int*, CUfunction, int, size_t) = nullptr;
  CUresult (*GetErrorString) (CUresult, const char**) = nullptr;
  bool ok = false;
};

struct Nvrtc {
  void* handle = nullptr;
  nvrtcResult (*CreateProgram) (nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
  nvrtcResult (*CompileProgram) (nvrtcProgram, int, const char* const*) = nullptr;
  nvrtcResult (*GetCUBINSize) (nvrtcProgram, size_t*) = nullptr;
  nvrtcResult (*GetCUBIN) (nvrtcProgram, char*) = nullptr;
  nvrtcResult (*GetProgramLogSize) (nvrtcProgram, size_t*) = nullptr;
  nvrtcResult (*GetProgramLog) (nvrtcProgram, char*) = nullptr;
  nvrtcResult (*DestroyProgram) (nvrtcProgram*) = nullptr;
  const char* (*GetErrorString) (nvrtcResult) = nullptr;
  bool ok = false;
};

static Driver g_drv;
static Nvrtc g_nvrtc;
static std::mutex g_loadMutex;      // several host threads (one per GPU) may create machines at once

static bool load_driver() {
  std::lock_guard<std::mutex> lock (g_loadMutex);
  if (g_drv.ok) return true;
  auto get = [] (const char* name, void** fn) {
    cudaDriverEntryPointQueryResult st;
    return cudaGetDriverEntryPoint (name, fn, cudaEnableDefault, &st) == cudaSuccess && st == cudaDriverEntryPointSuccess && *fn;
  };
  bool ok = get ("cuModuleLoadData", (void**) &g_drv.ModuleLoadData) && get ("cuModuleUnload", (void**) &g_drv.ModuleUnload)
    && get ("cuModuleGetFunction", (void**) &g_drv.ModuleGetFunction) && get ("cuLaunchKernel", (void**) &g_drv.LaunchKernel)
    && get ("cuModuleGetGlobal", (void**) &g_drv.ModuleGetGlobal)
    && get ("cuFuncSetAttribute", (void**) &g_drv.FuncSetAttribute) && get ("cuFuncGetAttribute", (void**) &g_drv.FuncGetAttribute)
    && get ("cuOccupancyMaxActiveBlocksPerMultiprocessor", (void**) &g_drv.OccupancyMaxActiveBlocksPerMultiprocessor)
    && get ("cuGetErrorString", (void**) &g_drv.GetErrorString);
  if (!ok) { set_error ("could not resolve the CUDA driver entry points (no driver?)"); return false; }
  g_drv.ok = true;
  return true;
}

static bool load_nvrtc() {
  std::lock_guard<std::mutex> lock (g_loadMutex);
  if (g_nvrtc.ok) return true;
  std::vector<std::string> cands;
  if (const char* e = getenv ("MB_NVRTC_LIB")) cands.push_back (e);
  cands.push_back ("libnvrtc.so.12");
  cands.push_back ("/usr/local/cuda/lib64/libnvrtc.so.12");
  cands.push_back ("/usr/local/cuda/lib64/libnvrtc.so");
  cands.push_back ("libnvrtc.so");
  for (auto& c: cands) { g_nvrtc.handle = dlopen (c.c_str(), RTLD_NOW | RTLD_GLOBAL); if (g_nvrtc.handle) break; }
  if (!g_nvrtc.handle) { set_error ("libnvrtc.so.12 not found (set MB_NVRTC_LIB)"); return false; }
  auto sym = [&] (const char* n) { return dlsym (g_nvrtc.handle, n); };
  g_nvrtc.CreateProgram = (decltype (g_nvrtc.CreateProgram)) sym ("nvrtcCreateProgram");
  g_nvrtc.CompileProgram = (decltype (g_nvrtc.CompileProgram)) sym ("nvrtcCompileProgram");
  g_nvrtc.GetCUBINSize = (decltype (g_nvrtc.GetCUBINSize)) sym ("nvrtcGetCUBINSize");
  g_nvrtc.GetCUBIN = (decltype (g_nvrtc.GetCUBIN)) sym ("nvrtcGetCUBIN");
  g_nvrtc.GetProgramLogSize = (decltype (g_nvrtc.GetProgramLogSize)) sym ("nvrtcGetProgramLogSize");
  g_nvrtc.GetProgramLog = (decltype (g_nvrtc.GetProgramLog)) sym ("nvrtcGetProgramLog");
  g_nvrtc.DestroyProgram = (decltype (g_nvrtc.DestroyProgram)) sym ("nvrtcDestroyProgram");
  g_nvrtc.GetErrorString = (decltype (g_nvrtc.GetErrorString)) sym ("nvrtcGetErrorString");
  if (!g_nvrtc.CreateProgram || !g_nvrtc.CompileProgram || !g_nvrtc.GetCUBINSize || !g_nvrtc.GetCUBIN || !g_nvrtc.GetProgramLogSize
      || !g_nvrtc.GetProgramLog || !g_nvrtc.DestroyProgram) { set_error ("libnvrtc is missing symbols"); return false; }
  g_nvrtc.ok = true;
  return true;
}

static bool cu_ok (CUresult r, const char* what) {
  if (r == CUDA_SUCCESS) return true;
  const char* s = nullptr;
  if (g_drv.GetErrorString) g_drv.GetErrorString (r, &s);
  set_error (std::string ("CUDA driver error: ") + (s ? s : "?") + " in " + what);
  return false;
}

// ---------------------------------------------------------------------------------------------
// the plan: slots, tables, generated source
// ---------------------------------------------------------------------------------------------
struct Slot {
  int type, self, other, rank;
  int emitOff = -1;   // offset into the emission table (non-silent slots)
  int silIdx = -1;    // index into the silent-weight array (silent slots)
  int idOff = 0;      // offset into the transition-id table
  int tableSize = 1;
};

struct Program {
  std::vector<Slot> slots;                    // ordered by (self, type, other, rank)
  std::vector<int> stateSlot0;                // [S+1] first slot of each state
  std::vector<int32_t> idTab;                 // transition id per table entry, -1 = no such transition
  std::vector<int32_t> emitId;                // transition id per emission-table entry
  std::vector<int32_t> silId;                 // transition id per silent slot
  int nEmit = 0, nSil = 0;
  // The same emission weights in ROW layout (score module): one row per input token holding, for every match
  // group, its nOut weights and, for every delete group, its weight; then one row per output token holding every
  // insert group's weight.  A cell's column keeps the shared-memory address of its input token's row in a
  // register, so a match weight is at (row + 8 * outTok) + constant, a delete weight at row + constant and an
  // insert weight at (the step's output-token row) + constant: one add per cell instead of an index computation
  // per weight.  rowOff[slot] = offset of the group inside its row; rowId[entry] = transition id (-1: none).
  int WA = 0, WB = 0;
  std::vector<int> rowOff;
  std::vector<int32_t> rowId;
  std::vector<int> rowSlot;                   // the group every row-layout entry belongs to
  // Linear-domain normalisation (score module).  State values are only defined up to a constant factor per
  // state: with value'(d) = value(d) / sigma_d every group's weight becomes w * sigma_src / sigma_d, and
  // choosing sigma_d = w_u * sigma_src(u) for ONE silent group u of d makes that group's weight exactly 1 --
  // its multiply disappears from the cell (dnapsw: 11 multiply-adds per cell become 7).  unitSlot[d] = u, or -1.
  std::vector<int> unitSlot;
};

static int table_size (int type, int nIn, int nOut) {
  return type == T_MATCH ? nIn * nOut : type == T_DELETE ? nIn : type == T_INSERT ? nOut : 1;
}

static int label_index (int type, int a, int b, int nOut) {   // a, b are 1-based tokens
  return type == T_MATCH ? (a - 1) * nOut + (b - 1) : type == T_DELETE ? a - 1 : type == T_INSERT ? b - 1 : 0;
}

static int trans_type (int a, int b) { return a ? (b ? T_MATCH : T_DELETE) : (b ? T_INSERT : T_SILENT); }

static void build_program (const mb_machine* m, bool forward, Program& p) {
  struct Key { int self, type, other, rank; bool operator< (const Key& k) const { return std::tie (self, type, other, rank) < std::tie (k.self, k.type, k.other, k.rank); } };
  std::map<Key, std::vector<std::pair<int, int>>> groups;       // -> (label index, transition id)
  std::map<std::tuple<int, int, int, int>, int> seen;           // (self, type, other, label) -> how many so far
  for (int64_t t = 0; t < m->T; ++t) {
    const int type = trans_type (m->in[t], m->out[t]);
    if (type == T_SILENT && m->dst[t] <= m->src[t]) continue;   // only possible on state 0 (machine.cpp:759); reads -inf in the reference
    const int self = forward ? m->dst[t] : m->src[t], other = forward ? m->src[t] : m->dst[t];
    const int li = label_index (type, m->in[t], m->out[t], m->nOut);
    const int rank = seen[std::make_tuple (self, type, other, li)]++;
    groups[Key { self, type, other, rank }].push_back ({ li, (int) t });
  }
  p.stateSlot0.assign ((size_t) m->S + 1, 0);
  for (auto& g: groups) {
    Slot s;
    s.type = g.first.type; s.self = g.first.self; s.other = g.first.other; s.rank = g.first.rank;
    s.tableSize = table_size (s.type, m->nIn, m->nOut);
    s.idOff = (int) p.idTab.size();
    p.idTab.resize (p.idTab.size() + s.tableSize, -1);
    for (auto& e: g.second) p.idTab[s.idOff + e.first] = e.second;
    if (s.type == T_SILENT) { s.silIdx = p.nSil++; p.silId.push_back (g.second[0].second); }
    else {
      s.emitOff = p.nEmit;
      p.nEmit += s.tableSize;
      p.emitId.resize ((size_t) p.nEmit, -1);
      for (auto& e: g.second) p.emitId[s.emitOff + e.first] = e.second;
    }
    p.stateSlot0[s.self + 1]++;
    p.slots.push_back (s);
  }
  for (int s = 0; s < m->S; ++s) p.stateSlot0[s + 1] += p.stateSlot0[s];
  // row layout
  p.rowOff.assign (p.slots.size(), -1);
  for (size_t k = 0; k < p.slots.size(); ++k) {
    const Slot& sl = p.slots[k];
    if (sl.type == T_MATCH) { p.rowOff[k] = p.WA; p.WA += m->nOut; }
    else if (sl.type == T_DELETE) { p.rowOff[k] = p.WA; p.WA += 1; }
    else if (sl.type == T_INSERT) { p.rowOff[k] = p.WB; p.WB += 1; }
  }
  p.rowId.assign ((size_t) std::max (m->nIn * p.WA + m->nOut * p.WB, 1), -1);
  p.rowSlot.assign (p.rowId.size(), -1);
  for (size_t k = 0; k < p.slots.size(); ++k) {
    const Slot& sl = p.slots[k];
    auto put = [&] (int entry, int label) { p.rowId[entry] = p.idTab[sl.idOff + label]; p.rowSlot[entry] = (int) k; };
    if (sl.type == T_MATCH) { for (int a = 0; a < m->nIn; ++a) for (int b = 0; b < m->nOut; ++b) put (a * p.WA + p.rowOff[k] + b, a * m->nOut + b); }
    else if (sl.type == T_DELETE) { for (int a = 0; a < m->nIn; ++a) put (a * p.WA + p.rowOff[k], a); }
    else if (sl.type == T_INSERT) { for (int b = 0; b < m->nOut; ++b) put (m->nIn * p.WA + b * p.WB + p.rowOff[k], b); }
  }
  // the unit group of a state: its first silent group
  p.unitSlot.assign ((size_t) m->S, -1);
  for (int d = 0; d < m->S; ++d)
    for (int k = p.stateSlot0[d]; k < p.stateSlot0[d + 1]; ++k)
      if (p.slots[k].type == T_SILENT) { p.unitSlot[d] = k; break; }
}

struct JitEngine {
  Program fwd, bwd;
  int C = 4, tbBytes = 1, threads = 128, minBlocks = 4, minBlocksLin = 5, minBlocksCnt = 4;
  // The score-only kernels (Viterbi, linear Forward / Backward) are compiled as a second module with
  // MB_C = CV columns per lane: fewer shuffles, boundary reads and loop overhead per cell (Viterbi fill
  // 26.5 -> 15.8 ms for 10 000 1 kb pairs).  256 columns under ONE power-of-two frame would exceed the
  // FP64 range on ordinary pairs, so in that module the linear sweeps keep a frame per lane
  // (MB_LANE_FRAMES); the E-step kernels, whose stored Forward blocks share a frame per warp, stay at C.
  int CV = 4, minBlocksV = 4;
  int minBlocksLinV = 4;      // the score module's normalised sums: 4 CTAs per SM at 128 registers beat 3 at 168 (8.33 against 8.80 ms)
  // the same three kernels at C columns per lane (first module): chosen per call for batches whose pairs
  // would leave most of a 32 * CV column strip empty (300 aa proteins: 2 strips of 256 against 3 of 128)
  CUfunction kViterbiN = nullptr, kForwardLinN = nullptr, kBackwardLinN = nullptr, kViterbiScoreN = nullptr;
  int blocksPerSMN[4] = { 1, 1, 1, 1 };
  CUfunction kViterbiScore = nullptr;      // Viterbi without back-pointers (mb_viterbi with pathLen == NULL, boss -V)
  // score module: row-layout tables (Program::WA) -- log weights for Viterbi, normalised linear weights for the sums
  double* dRowVit = nullptr;
  double* dRowFLinN = nullptr;
  double* dRowBLinN = nullptr;
  std::vector<char> silParamLinN;         // MBSilN { f[], b[], originF, originB, resLogF, resLogB }
  bool normOK = false;                    // every unit group's weight is usable: the normalised linear kernels may run
  std::string sourceV;
  // FITTED strip widths: when every pair of a batch fits one strip of 32 * Cf columns for a Cf between the two built-in widths
  // (or just above the wider one), a score module with MB_C = Cf sweeps a third fewer cells than the built-in ones
  // (300 aa proteins: 1 strip of 320 columns against 3 of 128 or 2 of 256).  Compiled the first time a batch asks for it,
  // at most kMaxFitModules per machine.
  struct FitModule { int C = 0; CUmodule mod = nullptr; CUfunction k[4] = { nullptr, nullptr, nullptr, nullptr }; int blocksPerSM[4] = { 1, 1, 1, 1 }; };      // viterbi, forward_lin, backward_lin, viterbi_score
  std::vector<FitModule> fit;
  std::vector<int> fitFailed;
  // split mode (strips as work items): the score module once more with MB_SPLIT 1, compiled when a call first needs it
  std::string sourceS;
  CUmodule modS = nullptr;
  bool splitTried = false;
  CUfunction kSplit[4] = { nullptr, nullptr, nullptr, nullptr };      // viterbi, forward_lin, backward_lin, viterbi_score
  int blocksPerSMS[4] = { 1, 1, 1, 1 };
  // E-step: Forward states kept per cell (those with an emitting transition group coming in, plus the
  // start state); the others follow from them inside the cell through the silent groups
  std::vector<int> stored;
  int storeQ = 1;      // 16-byte chunks per cell
  CUmodule modV = nullptr;
  std::vector<int> shift, bits;          // Viterbi back-pointer packing per state
  std::string source;
  CUmodule mod = nullptr;
  CUfunction kForward = nullptr, kBackward = nullptr, kViterbi = nullptr, kFStore = nullptr, kBCounts = nullptr;
  int blocksPerSM[10] = { 1, 1, 1, 1, 1, 1, 1, 1, 1, 1 };      // index 9: mb_k_viterbi_score
  size_t smemBytes[10] = { 0, 0, 0, 0, 0, 0, 0, 0, 0, 0 };
  int nCtx = 0;                          // thread-private count accumulators per lane (backward program's emitting slots)
  std::vector<int> ctxBase;              // per backward slot, -1 for silent
  int32_t* dIdTabB = nullptr;
  // scaled linear-domain sweeps
  CUfunction kForwardLin = nullptr, kBackwardLin = nullptr, kFStoreLin = nullptr, kBCountsLin = nullptr;
  bool linearOK = false;
  double* dEmitFLin = nullptr;
  double* dEmitBLin = nullptr;
  std::vector<char> silParamLin;
  int numSMs = 148;
  // device tables
  double* dEmitF = nullptr;
  double* dEmitB = nullptr;
  int32_t* dTbPlan = nullptr;             // packed arrays for the traceback kernel
  std::vector<char> silParam;             // MBSil { double f[max(nSilF,1)]; double b[max(nSilB,1)]; }
  unsigned long long* dCounter = nullptr;
};

static std::string term_expr (const Slot& s, int nOut, bool forward) {
  std::ostringstream e;
  const char* arr = s.type == T_MATCH ? "D" : s.type == T_DELETE ? "L" : s.type == T_INSERT ? "U" : nullptr;
  if (arr) e << arr << "[" << s.other << "]";
  else e << "n" << s.other;
  e << " + ";
  if (s.type == T_MATCH) e << "E[" << s.emitOff << " + a * " << nOut << " + b]";
  else if (s.type == T_DELETE) e << "E[" << s.emitOff << " + a]";
  else if (s.type == T_INSERT) e << "E[" << s.emitOff << " + b]";
  else e << "P." << (forward ? "f" : "b") << "[" << s.silIdx << "]";
  return e.str();
}

static void gen_cell (std::ostringstream& o, const mb_machine* m, const Program& p, bool forward, bool viterbi, const JitEngine& J) {
  const char* name = viterbi ? "mb_cell_vit" : forward ? "mb_cell_fwd" : "mb_cell_bwd";
  o << "__device__ __forceinline__ " << (viterbi ? "mb_tbword " : "void ") << name
    << " (const double (&D)[MB_S], const double (&L)[MB_S], const double (&U)[MB_S], double (&N)[MB_S], const int a, const int b, const bool origin, "
    << (viterbi ? "const bool sink, " : "") << "const double* __restrict__ E, const MBSil& P) {\n";
  if (viterbi) o << "  mb_tbword word = 0;\n";
  const int originState = forward ? 0 : m->S - 1;
  // Viterbi: a state nothing leaves (the end state, normally) is only ever read -- as the score, and by
  // the traceback's first step -- in the pair's last cell; everywhere else its value and pointer are
  // dead, so they are computed under `sink` (false at compile time in the steady-state step)
  std::vector<char> isSource ((size_t) m->S, 0);
  for (auto& sl: p.slots) isSource[sl.other] = 1;
  for (int q = 0; q < m->S; ++q) {
    const int d = forward ? q : m->S - 1 - q;
    const int s0 = p.stateSlot0[d], s1 = p.stateSlot0[d + 1];
    const bool sinkOnly = viterbi && !isSource[d] && d != originState && s0 != s1;
    if (s0 == s1 || sinkOnly) o << "  double n" << d << " = mb_neg_inf();\n";
    if (sinkOnly) o << "  if (sink) {\n";
    for (int k = s0; k < s1; ++k) {
      const std::string t = term_expr (p.slots[k], m->nOut, forward);
      if (k == s0) o << (sinkOnly ? "  n" : "  double n") << d << " = " << t << ";\n";
      else if (viterbi) {
        // strict '<': the first maximum keeps the pointer (dpmatrix.defs.h:171-174); the pointer field
        // of this state is overwritten in place, one logic op under the compare's predicate
        const unsigned long long field = ((1ull << J.bits[d]) - 1ull) << J.shift[d], val = (unsigned long long) (k - s0) << J.shift[d];
        o << "  { const double t = " << t << "; if (n" << d << " < t) { n" << d << " = t; word = (word & (mb_tbword) " << (~field) << "ull) | (mb_tbword) " << val << "ull; } }\n";
      }
      else o << "  n" << d << " = mb_lse (n" << d << ", " << t << ");\n";
    }
    if (sinkOnly) o << "  }\n";
    if (d == originState) o << "  if (origin) n" << d << " = 0.0;\n";
  }
  for (int d = 0; d < m->S; ++d) o << "  N[" << d << "] = n" << d << ";\n";
  if (viterbi) o << "  return word;\n";
  o << "}\n\n";
}

// ---- score module: cell functions over the row-layout tables (see Program::WA) ----
// ea = shared-memory byte address of the input token's row, em = ea + 8 * output token, ebr = address of the
// output token's row.  MB_LDS (address, byte offset) reads one weight.
static std::string row_weight (const Slot& s, int rowOff) {
  std::ostringstream e;
  e << "MB_LDS (" << (s.type == T_MATCH ? "em" : s.type == T_DELETE ? "ea" : "ebr") << ", " << rowOff * 8 << ")";
  return e.str();
}

static std::string source_expr (const Slot& s) {
  std::ostringstream e;
  const char* arr = s.type == T_MATCH ? "D" : s.type == T_DELETE ? "L" : s.type == T_INSERT ? "U" : nullptr;
  if (arr) e << arr << "[" << s.other << "]"; else e << "n" << s.other;
  return e.str();
}

// Viterbi: FP64 add + compare in the reference's candidate order.  PTR = also record which candidate won: the
// pointer field of the state goes straight into the step's packed words (pk, the cell's word starting at bit sh:
// a constant once the column loop is unrolled) under the compare's own predicate -- mb_vmax is one compare, the
// select of the value and ONE predicated logic instruction, with no per-cell word to build, shift and merge.
// (Comparing the bit patterns on the integer pipe instead -- valid when no log-weight is positive -- was measured
// slower: 17.2 against 15.9 ms for 10 000 dnapsw pairs of 1 kb; an integer compare of two doubles is two
// instructions and the sweep is short of issue slots, not of FP64 cycles.)
static void gen_cell_row_vit (std::ostringstream& o, const mb_machine* m, const Program& p, const JitEngine& J) {
  o << "template<bool PTR> __device__ __forceinline__ void mb_cell_vitr (const double (&D)[MB_S], const double (&L)[MB_S], const double (&U)[MB_S], double (&N)[MB_S], "
       "const unsigned ea, const unsigned em, const unsigned ebr, const bool origin, const bool sink, const MBSil& P, unsigned (&pk)[MB_PKW], const int sh) {\n";
  std::vector<char> isSource ((size_t) m->S, 0);
  for (auto& sl: p.slots) isSource[sl.other] = 1;
  for (int d = 0; d < m->S; ++d) {
    const int s0 = p.stateSlot0[d], s1 = p.stateSlot0[d + 1];
    const bool sinkOnly = !isSource[d] && d != 0 && s0 != s1;
    if (s0 == s1 || sinkOnly) o << "  double n" << d << " = mb_neg_inf();\n";
    if (sinkOnly) o << "  if (sink) {\n";
    for (int k = s0; k < s1; ++k) {
      const Slot& sl = p.slots[k];
      std::ostringstream t;
      t << source_expr (sl) << " + ";
      if (sl.type == T_SILENT) t << "P.f[" << sl.silIdx << "]"; else t << row_weight (sl, p.rowOff[k]);
      if (k == s0) o << (sinkOnly ? "  n" : "  double n") << d << " = " << t.str() << ";\n";
      else {
        // the field never straddles a 32-bit word (see generate()): word index and shift inside it
        const unsigned field = (unsigned) ((1ull << J.bits[d]) - 1ull), val = (unsigned) (k - s0);
        o << "  mb_vmax<PTR> (n" << d << ", " << t.str() << ", pk[(sh + " << J.shift[d] << ") >> 5], " << field << "u << ((sh + " << J.shift[d] << ") & 31), "
          << val << "u << ((sh + " << J.shift[d] << ") & 31));\n";
      }
    }
    if (sinkOnly) o << "  }\n";
    if (d == 0) o << "  if (origin) n" << d << " = 0.0;\n";
  }
  for (int d = 0; d < m->S; ++d) o << "  N[" << d << "] = n" << d << ";\n";
  o << "}\n\n";
}

// Linear domain, normalised: the unit group of a state is a plain copy, every other group one multiply-add
// with its scaled weight
static void gen_cell_row_lin (std::ostringstream& o, const mb_machine* m, const Program& p, bool forward) {
  o << "__device__ __forceinline__ void " << (forward ? "mb_cell_fwd_linr" : "mb_cell_bwd_linr")
    << " (const double (&D)[MB_S], const double (&L)[MB_S], const double (&U)[MB_S], double (&N)[MB_S], "
       "const unsigned ea, const unsigned em, const unsigned ebr, const bool origin, const MBSilN& P) {\n";
  const int originState = forward ? 0 : m->S - 1;
  for (int q = 0; q < m->S; ++q) {
    const int d = forward ? q : m->S - 1 - q;
    const int s0 = p.stateSlot0[d], s1 = p.stateSlot0[d + 1], unit = p.unitSlot[d];
    if (s0 == s1) o << "  double n" << d << " = 0.0;\n";
    if (unit >= 0) o << "  double n" << d << " = " << source_expr (p.slots[unit]) << ";\n";
    bool first = unit < 0;
    for (int k = s0; k < s1; ++k) {
      if (k == unit) continue;
      const Slot& sl = p.slots[k];
      std::ostringstream w;
      if (sl.type == T_SILENT) w << "P." << (forward ? "f" : "b") << "[" << sl.silIdx << "]"; else w << row_weight (sl, p.rowOff[k]);
      if (first) o << "  double n" << d << " = " << source_expr (sl) << " * " << w.str() << ";\n";
      else o << "  n" << d << " = fma (" << source_expr (sl) << ", " << w.str() << ", n" << d << ");\n";
      first = false;
    }
    if (d == originState) o << "  if (origin) n" << d << " = P." << (forward ? "originF" : "originB") << ";\n";
  }
  for (int d = 0; d < m->S; ++d) o << "  N[" << d << "] = n" << d << ";\n";
  o << "}\n\n";
}

static int ctx_count (int type, int C, int nOut) { return type == T_MATCH ? C * nOut : type == T_DELETE ? C : type == T_INSERT ? nOut : 0; }

// Backward cell fused with posterior counts (backward.cpp:62-87): for state s and each of its
// outgoing transition groups, term = w + B(dest cell, dest) feeds both B(s) and
// exp((F(s) - ll) + term), which is added to the group's accumulator.
static void gen_cell_counts (std::ostringstream& o, const mb_machine* m, const JitEngine& J) {
  const Program& p = J.bwd;
  o << "__device__ __forceinline__ void mb_cell_cnt (const double (&D)[MB_S], const double (&L)[MB_S], const double (&U)[MB_S], double (&N)[MB_S], const int a, const int b, const bool origin, const double* __restrict__ E, const MBSil& P, const double (&F)[MB_S], float (&cs)[MB_NSIL_B > 0 ? MB_NSIL_B : 1], float* __restrict__ acc, const int c) {\n";
  for (int q = 0; q < m->S; ++q) {
    const int d = m->S - 1 - q;
    const int s0 = p.stateSlot0[d], s1 = p.stateSlot0[d + 1];
    if (s0 == s1) o << "  double n" << d << " = mb_neg_inf();\n";
    for (int k = s0; k < s1; ++k) {
      const Slot& sl = p.slots[k];
      o << "  const double t" << k << " = " << term_expr (sl, m->nOut, false) << ";\n";
      if (k == s0) o << "  double n" << d << " = t" << k << ";\n";
      else o << "  n" << d << " = mb_lse (n" << d << ", t" << k << ");\n";
      o << "  { const float p = mb_post (F[" << d << "] + t" << k << "); ";
      if (sl.type == T_SILENT) o << "cs[" << sl.silIdx << "] += p; }\n";
      else {
        o << "acc[(" << J.ctxBase[k] << " + ";
        if (sl.type == T_MATCH) o << "c * " << m->nOut << " + b";
        else if (sl.type == T_DELETE) o << "c";
        else o << "b";
        o << ") * 32] += p; }\n";
      }
    }
    if (d == m->S - 1) o << "  if (origin) n" << d << " = 0.0;\n";
  }
  for (int d = 0; d < m->S; ++d) o << "  N[" << d << "] = n" << d << ";\n";
  o << "}\n\n";
  // flush: per strip, accumulators -> global double counts
  o << "__device__ __forceinline__ void mb_flush_counts (float (&cs)[MB_NSIL_B > 0 ? MB_NSIL_B : 1], float* __restrict__ acc, const int (&ta)[MB_C], double* __restrict__ counts, const int32_t* __restrict__ idTab, const int lane) {\n";
  for (size_t k = 0; k < p.slots.size(); ++k) {
    const Slot& sl = p.slots[k];
    if (sl.type == T_SILENT) {
      o << "  { const float v = mb_warp_sum (cs[" << sl.silIdx << "]); if (lane == 0 && v != 0.f) atomicAdd (counts + " << p.silId[sl.silIdx] << ", (double) v); }\n";
    } else if (sl.type == T_MATCH) {
      o << "  _Pragma(\"unroll\") for (int c = 0; c < MB_C; ++c) for (int b = 0; b < " << m->nOut << "; ++b) { const float v = acc[(" << J.ctxBase[k] << " + c * " << m->nOut << " + b) * 32]; if (v != 0.f) { const int id = idTab[" << sl.idOff << " + ta[c] * " << m->nOut << " + b]; if (id >= 0) atomicAdd (counts + id, (double) v); } }\n";
    } else if (sl.type == T_DELETE) {
      o << "  _Pragma(\"unroll\") for (int c = 0; c < MB_C; ++c) { const float v = acc[(" << J.ctxBase[k] << " + c) * 32]; if (v != 0.f) { const int id = idTab[" << sl.idOff << " + ta[c]]; if (id >= 0) atomicAdd (counts + id, (double) v); } }\n";
    } else {
      o << "  for (int b = 0; b < " << m->nOut << "; ++b) { const float v = acc[(" << J.ctxBase[k] << " + b) * 32]; if (v != 0.f) { const int id = idTab[" << sl.idOff << " + b]; if (id >= 0) atomicAdd (counts + id, (double) v); } }\n";
    }
  }
  o << "}\n\n";
}

// Linear-domain cell: value(state) = sum over its transition groups of value(source) * weight.
static void gen_cell_lin (std::ostringstream& o, const mb_machine* m, const Program& p, bool forward) {
  o << "__device__ __forceinline__ void " << (forward ? "mb_cell_fwd_lin" : "mb_cell_bwd_lin")
    << " (const double (&D)[MB_S], const double (&L)[MB_S], const double (&U)[MB_S], double (&N)[MB_S], const int a, const int b, const bool origin, const double* __restrict__ E, const MBSil& P) {\n";
  const int originState = forward ? 0 : m->S - 1;
  for (int q = 0; q < m->S; ++q) {
    const int d = forward ? q : m->S - 1 - q;
    const int s0 = p.stateSlot0[d], s1 = p.stateSlot0[d + 1];
    if (s0 == s1) o << "  double n" << d << " = 0.0;\n";
    for (int k = s0; k < s1; ++k) {
      const Slot& sl = p.slots[k];
      std::ostringstream src, w;
      const char* arr = sl.type == T_MATCH ? "D" : sl.type == T_DELETE ? "L" : sl.type == T_INSERT ? "U" : nullptr;
      if (arr) src << arr << "[" << sl.other << "]"; else src << "n" << sl.other;
      if (sl.type == T_MATCH) w << "E[" << sl.emitOff << " + a * " << m->nOut << " + b]";
      else if (sl.type == T_DELETE) w << "E[" << sl.emitOff << " + a]";
      else if (sl.type == T_INSERT) w << "E[" << sl.emitOff << " + b]";
      else w << "P." << (forward ? "f" : "b") << "[" << sl.silIdx << "]";
      if (k == s0) o << "  double n" << d << " = " << src.str() << " * " << w.str() << ";\n";
      else o << "  n" << d << " = fma (" << src.str() << ", " << w.str() << ", n" << d << ");\n";
    }
    if (d == originState) o << "  if (origin) n" << d << " = 1.0;\n";
  }
  for (int d = 0; d < m->S; ++d) o << "  N[" << d << "] = n" << d << ";\n";
  o << "}\n\n";
}

// The E-step's stored Forward cell (linear domain).  A state all of whose incoming transition groups
// are silent is a linear function of lower-numbered states of the SAME cell, so only the states that
// something emitting enters (and the start state, which carries the origin) need to be kept: 3 of
// dnapsw's 8.  mb_fpack_lin rounds those to their high words; mb_fexpand_lin rebuilds the whole cell,
// scaled by kap, for the posterior products.
static void gen_fstore_lin (std::ostringstream& o, const mb_machine* m, JitEngine& J) {
  const Program& p = J.fwd;
  std::vector<char> keep ((size_t) m->S, 0);
  keep[0] = 1;
  for (auto& sl: p.slots) if (sl.type != T_SILENT) keep[sl.self] = 1;
  J.stored.clear();
  for (int d = 0; d < m->S; ++d) if (keep[d]) J.stored.push_back (d);
  J.storeQ = ((int) J.stored.size() + 3) / 4;
  o << "#define MB_SQ " << J.storeQ << "      // 16-byte chunks per cell in the stored Forward blocks (" << J.stored.size() << " of " << m->S << " states kept)\n";
  o << "__device__ __forceinline__ void mb_fpack_lin (const double (&N)[MB_S], unsigned (&hw)[4 * MB_SQ]) {\n";
  for (int j = 0; j < 4 * J.storeQ; ++j) {
    if (j < (int) J.stored.size()) o << "  hw[" << j << "] = (unsigned) __double2hiint (N[" << J.stored[j] << "]) + ((unsigned) __double2loint (N[" << J.stored[j] << "]) >> 31);\n";
    else o << "  hw[" << j << "] = 0u;\n";
  }
  o << "}\n\n";
  o << "__device__ __forceinline__ void mb_fexpand_lin (const unsigned (&hw)[4 * MB_SQ], const double kap, double (&F)[MB_S], const MBSil& P) {\n";
  for (int d = 0; d < m->S; ++d) {
    if (keep[d]) {
      const int j = (int) (std::find (J.stored.begin(), J.stored.end(), d) - J.stored.begin());
      o << "  const double f" << d << " = __hiloint2double ((int) hw[" << j << "], 0) * kap;\n";
      continue;
    }
    const int s0 = p.stateSlot0[d], s1 = p.stateSlot0[d + 1];
    if (s0 == s1) { o << "  const double f" << d << " = 0.0;\n"; continue; }
    for (int k = s0; k < s1; ++k) {
      const Slot& sl = p.slots[k];
      if (k == s0) o << "  double f" << d << " = f" << sl.other << " * P.f[" << sl.silIdx << "];\n";
      else o << "  f" << d << " = fma (f" << sl.other << ", P.f[" << sl.silIdx << "], f" << d << ");\n";
    }
  }
  for (int d = 0; d < m->S; ++d) o << "  F[" << d << "] = f" << d << ";\n";
  o << "}\n\n";
}

// Linear-domain Backward cell fused with the posterior counts: per transition group
//   t = B(dest) * w;  B(s) += t;  count(group) += F'(s) * t     with F' = F * 2^(eF+eB) / Z
static void gen_cell_counts_lin (std::ostringstream& o, const mb_machine* m, const JitEngine& J) {
  const Program& p = J.bwd;
  o << "__device__ __forceinline__ void mb_cell_cnt_lin (const double (&D)[MB_S], const double (&L)[MB_S], const double (&U)[MB_S], double (&N)[MB_S], const int a, const int b, const bool origin, const double* __restrict__ E, const MBSil& P, const double (&F)[MB_S], double (&cs)[MB_NSIL_B > 0 ? MB_NSIL_B : 1], double* __restrict__ acc, const int c) {\n";
  for (int q = 0; q < m->S; ++q) {
    const int d = m->S - 1 - q;
    const int s0 = p.stateSlot0[d], s1 = p.stateSlot0[d + 1];
    if (s0 == s1) o << "  double n" << d << " = 0.0;\n";
    for (int k = s0; k < s1; ++k) {
      const Slot& sl = p.slots[k];
      std::ostringstream src, w;
      const char* arr = sl.type == T_MATCH ? "D" : sl.type == T_DELETE ? "L" : sl.type == T_INSERT ? "U" : nullptr;
      if (arr) src << arr << "[" << sl.other << "]"; else src << "n" << sl.other;
      if (sl.type == T_MATCH) w << "E[" << sl.emitOff << " + a * " << m->nOut << " + b]";
      else if (sl.type == T_DELETE) w << "E[" << sl.emitOff << " + a]";
      else if (sl.type == T_INSERT) w << "E[" << sl.emitOff << " + b]";
      else w << "P.b[" << sl.silIdx << "]";
      o << "  const double t" << k << " = " << src.str() << " * " << w.str() << ";\n";
      if (k == s0) o << "  double n" << d << " = t" << k << ";\n";
      else o << "  n" << d << " += t" << k << ";\n";
      if (sl.type == T_SILENT) o << "  cs[" << sl.silIdx << "] = fma (F[" << d << "], t" << k << ", cs[" << sl.silIdx << "]);\n";
      else {
        std::ostringstream ix;
        ix << "(" << J.ctxBase[k] << " + ";
        if (sl.type == T_MATCH) ix << "c * " << m->nOut << " + b";
        else if (sl.type == T_DELETE) ix << "c";
        else ix << "b";
        ix << ") * 32";
        o << "  acc[" << ix.str() << "] = fma (F[" << d << "], t" << k << ", acc[" << ix.str() << "]);\n";
      }
    }
    if (d == m->S - 1) o << "  if (origin) n" << d << " = 1.0;\n";
  }
  for (int d = 0; d < m->S; ++d) o << "  N[" << d << "] = n" << d << ";\n";
  o << "}\n\n";
  o << "__device__ __forceinline__ void mb_flush_counts_lin (double (&cs)[MB_NSIL_B > 0 ? MB_NSIL_B : 1], double* __restrict__ acc, const int (&ta)[MB_C], double* __restrict__ counts, const int32_t* __restrict__ idTab, const int lane) {\n";
  for (size_t k = 0; k < p.slots.size(); ++k) {
    const Slot& sl = p.slots[k];
    if (sl.type == T_SILENT) {
      o << "  { const double v = mb_warp_sum_d (cs[" << sl.silIdx << "]); if (lane == 0 && v != 0.0) atomicAdd (counts + " << p.silId[sl.silIdx] << ", v); }\n";
    } else if (sl.type == T_MATCH) {
      o << "  _Pragma(\"unroll\") for (int c = 0; c < MB_C; ++c) for (int b = 0; b < " << m->nOut << "; ++b) { const double v = acc[(" << J.ctxBase[k] << " + c * " << m->nOut << " + b) * 32]; if (v != 0.0) { const int id = idTab[" << sl.idOff << " + ta[c] * " << m->nOut << " + b]; if (id >= 0) atomicAdd (counts + id, v); } }\n";
    } else if (sl.type == T_DELETE) {
      o << "  _Pragma(\"unroll\") for (int c = 0; c < MB_C; ++c) { const double v = acc[(" << J.ctxBase[k] << " + c) * 32]; if (v != 0.0) { const int id = idTab[" << sl.idOff << " + ta[c]]; if (id >= 0) atomicAdd (counts + id, v); } }\n";
    } else {
      o << "  for (int b = 0; b < " << m->nOut << "; ++b) { const double v = acc[(" << J.ctxBase[k] << " + b) * 32]; if (v != 0.0) { const int id = idTab[" << sl.idOff << " + b]; if (id >= 0) atomicAdd (counts + id, v); } }\n";
    }
  }
  o << "}\n\n";
}

bool jit_supported (const mb_machine* m, std::string* why) {
  auto no = [&] (const char* w) { if (why) *why = w; return false; };
  if (m->S > 16) return no ("more than 16 states");
  if (m->T > 4096) return no ("more than 4096 transitions");
  Program f, b;
  build_program (m, true, f);
  build_program (m, false, b);
  if (f.slots.size() > 160 || b.slots.size() > 160) return no ("more than 160 transition groups");
  if (f.nEmit > 3072 || b.nEmit > 3072) return no ("emission tables exceed 24 KB of shared memory");
  if (f.nSil + b.nSil > 400) return no ("too many silent transitions for the kernel-parameter block");
  int totalBits = 0;
  for (int s = 0; s < m->S; ++s) {
    const int n = f.stateSlot0[s + 1] - f.stateSlot0[s];
    int bt = 0; while ((1 << bt) < n) ++bt;
    if (bt && (totalBits >> 5) != ((totalBits + bt - 1) >> 5)) totalBits = (totalBits + 31) & ~31;      // as in generate()
    totalBits += bt;
  }
  if (totalBits > 64) return no ("Viterbi back-pointers need more than 64 bits per cell");
  { const int C = m->S <= 8 ? 4 : 2; int n = 0; for (auto& sl: b.slots) n += ctx_count (sl.type, C, m->nOut); if (n > 160) return no ("too many emitting transition groups for the per-lane count accumulators"); }
  return true;
}

// A directory of compiled modules (mb_set_kernel_cache_dir): <FNV-1a 64 of the compiler options, the CUDA version this library was
// built with and the generated source>.cubin.  A process that meets a machine structure it -- or an earlier process -- has
// compiled before loads the module instead of running NVRTC (dnapsw: 4 s of compilation per process otherwise, which is most of
// what a command-line call of one batch takes).  Off unless a directory is set.
static std::mutex g_cacheMutex;
static std::string g_cacheDir;
void rt_set_cache_dir (const char* dir) { std::lock_guard<std::mutex> lock (g_cacheMutex); g_cacheDir = dir ? dir : ""; }
static std::string cache_path (const std::string& source, const char* const* opts, int nOpts) {
  std::string dir;
  { std::lock_guard<std::mutex> lock (g_cacheMutex); dir = g_cacheDir; }
  if (dir.empty()) return dir;
  unsigned long long h = 1469598103934665603ull;
  auto mix = [&] (const char* p, size_t n) { for (size_t q = 0; q < n; ++q) { h ^= (unsigned char) p[q]; h *= 1099511628211ull; } };
  for (int q = 0; q < nOpts; ++q) mix (opts[q], strlen (opts[q]) + 1);
  const int version = CUDART_VERSION;
  mix ((const char*) &version, sizeof version);
  mix (source.data(), source.size());
  char name[40];
  snprintf (name, sizeof name, "/%016llx.cubin", h);
  return dir + name;
}

static int nvrtc_compile (const std::string& source, const char* dumpSuffix, std::vector<char>& cubin, std::string* logOut) {
  const char* cacheOpts[] = { "--gpu-architecture=sm_100a", "-lineinfo", "--std=c++17", "--ptxas-options=-v", "-default-device" };
  const std::string cached = cache_path (source, cacheOpts, 5);
  if (!cached.empty()) {
    if (FILE* f = fopen (cached.c_str(), "rb")) {
      fseek (f, 0, SEEK_END);
      const long n = ftell (f);
      fseek (f, 0, SEEK_SET);
      cubin.resize (n > 0 ? (size_t) n : 0);
      const bool ok = n > 0 && fread (cubin.data(), 1, (size_t) n, f) == (size_t) n;
      fclose (f);
      if (ok) { if (logOut) *logOut = "(module taken from the kernel cache: " + cached + ")"; return 0; }
    }
  }
  if (!load_nvrtc()) return 1;
  nvrtcProgram prog;
  if (g_nvrtc.CreateProgram (&prog, source.c_str(), "mb_jit_kernels.cu", 0, nullptr, nullptr) != NVRTC_SUCCESS) { set_error ("nvrtcCreateProgram failed"); return 1; }
  const char* opts[] = { "--gpu-architecture=sm_100a", "-lineinfo", "--std=c++17", "--ptxas-options=-v", "-default-device" };
  const nvrtcResult r = g_nvrtc.CompileProgram (prog, 5, opts);
  size_t ln = 0;
  g_nvrtc.GetProgramLogSize (prog, &ln);
  std::string log (ln, 0);
  if (ln) g_nvrtc.GetProgramLog (prog, &log[0]);
  while (!log.empty() && log.back() == 0) log.pop_back();
  if (logOut) *logOut = log;
  if (const char* d = getenv ("MB_JIT_DUMP")) { FILE* f = fopen ((std::string (d) + dumpSuffix).c_str(), "w"); if (f) { fputs (source.c_str(), f); fclose (f); } }
  if (r != NVRTC_SUCCESS) {
    set_error ("NVRTC compilation failed:\n" + log);
    g_nvrtc.DestroyProgram (&prog);
    return 1;
  }
  size_t n = 0;
  g_nvrtc.GetCUBINSize (prog, &n);
  cubin.resize (n);
  g_nvrtc.GetCUBIN (prog, cubin.data());
  g_nvrtc.DestroyProgram (&prog);
  if (!cached.empty()) {      // written under another name first: a reader never sees half a file
    const std::string tmp = cached + ".tmp" + std::to_string ((long long) getpid());
    if (FILE* f = fopen (tmp.c_str(), "wb")) {
      const bool ok = fwrite (cubin.data(), 1, n, f) == n;
      fclose (f);
      if (!ok || rename (tmp.c_str(), cached.c_str())) remove (tmp.c_str());
    }
  }
  if (const char* d = getenv ("MB_JIT_DUMP")) { FILE* f = fopen ((std::string (d) + dumpSuffix + ".cubin").c_str(), "wb"); if (f) { fwrite (cubin.data(), 1, n, f); fclose (f); } }
  return 0;
}

static int compile (mb_machine* m, JitEngine& J) {
  std::vector<char> cubin, cubinV;
  if (nvrtc_compile (J.source, "", cubin, nullptr) || !load_driver()) return 1;
  if (!J.sourceV.empty() && nvrtc_compile (J.sourceV, ".viterbi.cu", cubinV, nullptr)) return 1;
  MB_CUDA (cudaFree (0));   // make sure the primary context exists and is current
  if (!cu_ok (g_drv.ModuleLoadData (&J.mod, cubin.data()), "cuModuleLoadData")) return 1;
  if (!J.sourceV.empty() && !cu_ok (g_drv.ModuleLoadData (&J.modV, cubinV.data()), "cuModuleLoadData")) return 1;
  if (!cu_ok (g_drv.ModuleGetFunction (&J.kForward, J.mod, "mb_k_forward"), "cuModuleGetFunction")
      || !cu_ok (g_drv.ModuleGetFunction (&J.kBackward, J.mod, "mb_k_backward"), "cuModuleGetFunction")
      || !cu_ok (g_drv.ModuleGetFunction (&J.kViterbi, J.modV ? J.modV : J.mod, "mb_k_viterbi"), "cuModuleGetFunction")
      || !cu_ok (g_drv.ModuleGetFunction (&J.kViterbiScore, J.modV ? J.modV : J.mod, "mb_k_viterbi_score"), "cuModuleGetFunction")
      || !cu_ok (g_drv.ModuleGetFunction (&J.kFStore, J.mod, "mb_k_fstore"), "cuModuleGetFunction")
      || !cu_ok (g_drv.ModuleGetFunction (&J.kBCounts, J.mod, "mb_k_bcounts"), "cuModuleGetFunction")
      || !cu_ok (g_drv.ModuleGetFunction (&J.kForwardLin, J.modV ? J.modV : J.mod, "mb_k_forward_lin"), "cuModuleGetFunction")
      || !cu_ok (g_drv.ModuleGetFunction (&J.kBackwardLin, J.modV ? J.modV : J.mod, "mb_k_backward_lin"), "cuModuleGetFunction")
      || !cu_ok (g_drv.ModuleGetFunction (&J.kFStoreLin, J.mod, "mb_k_fstore_lin"), "cuModuleGetFunction")
      || !cu_ok (g_drv.ModuleGetFunction (&J.kBCountsLin, J.mod, "mb_k_bcounts_lin"), "cuModuleGetFunction")) return 1;
  if (J.modV && (!cu_ok (g_drv.ModuleGetFunction (&J.kViterbiN, J.mod, "mb_k_viterbi"), "cuModuleGetFunction")
                 || !cu_ok (g_drv.ModuleGetFunction (&J.kViterbiScoreN, J.mod, "mb_k_viterbi_score"), "cuModuleGetFunction")
                 || !cu_ok (g_drv.ModuleGetFunction (&J.kForwardLinN, J.mod, "mb_k_forward_lin"), "cuModuleGetFunction")
                 || !cu_ok (g_drv.ModuleGetFunction (&J.kBackwardLinN, J.mod, "mb_k_backward_lin"), "cuModuleGetFunction"))) return 1;
  int dev = 0;
  MB_CUDA (cudaGetDevice (&dev));
  MB_CUDA (cudaDeviceGetAttribute (&J.numSMs, cudaDevAttrMultiProcessorCount, dev));
  CUfunction fn[10] = { J.kForward, J.kBackward, J.kViterbi, J.kFStore, J.kBCounts, J.kForwardLin, J.kBackwardLin, J.kFStoreLin, J.kBCountsLin, J.kViterbiScore };
  const int ne[10] = { J.fwd.nEmit, J.bwd.nEmit, J.fwd.nEmit, J.fwd.nEmit, J.bwd.nEmit, J.fwd.nEmit, J.bwd.nEmit, J.fwd.nEmit, J.bwd.nEmit, J.fwd.nEmit };
  for (int q = 0; q < 10; ++q) {
    const bool needAcc = q == 4 || q == 8;      // only the count kernels use the per-lane accumulators (FP32 / FP64)
    J.smemBytes[q] = (size_t) (((ne[q] + 1) & ~1) + (J.threads / 32) * (16 + 32 * (m->S + 1))) * 8
      + (needAcc ? (size_t) (J.threads / 32) * 32 * std::max (J.nCtx, 1) * (q == 8 ? 8 : 4) : 0)
      + (q == 8 ? (size_t) (J.threads / 32) * 2 * (32 * J.C * J.storeQ * 4) * 4 : 0);     // two staged Forward blocks per warp
    if (!cu_ok (g_drv.FuncSetAttribute (fn[q], CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int) J.smemBytes[q]), "cuFuncSetAttribute")) return 1;
    int nb = 0;
    if (!cu_ok (g_drv.OccupancyMaxActiveBlocksPerMultiprocessor (&nb, fn[q], J.threads, J.smemBytes[q]), "occupancy")) return 1;
    J.blocksPerSM[q] = std::max (1, nb);
  }
  if (J.modV) {
    CUfunction fnN[4] = { J.kViterbiN, J.kForwardLinN, J.kBackwardLinN, J.kViterbiScoreN };
    const int qOf[4] = { 2, 5, 6, 9 };
    for (int q = 0; q < 4; ++q) {
      if (!cu_ok (g_drv.FuncSetAttribute (fnN[q], CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int) J.smemBytes[qOf[q]]), "cuFuncSetAttribute")) return 1;
      int nb = 0;
      if (!cu_ok (g_drv.OccupancyMaxActiveBlocksPerMultiprocessor (&nb, fnN[q], J.threads, J.smemBytes[qOf[q]]), "occupancy")) return 1;
      J.blocksPerSMN[q] = std::max (1, nb);
    }
  }
  return 0;
}

// The split-mode module, on first use.
static int ensure_split_module (mb_machine* m, JitEngine& J) {
  if (J.modS) return 0;
  if (J.splitTried) { set_error ("jit engine: the split-mode module could not be built"); return 1; }
  J.splitTried = true;
  std::vector<char> cubin;
  if (nvrtc_compile (J.sourceS, ".split.cu", cubin, nullptr)) return 1;
  if (!cu_ok (g_drv.ModuleLoadData (&J.modS, cubin.data()), "cuModuleLoadData")) return 1;
  const char* names[4] = { "mb_k_viterbi", "mb_k_forward_lin", "mb_k_backward_lin", "mb_k_viterbi_score" };
  const int qOf[4] = { 2, 5, 6, 9 };
  for (int q = 0; q < 4; ++q) {
    if (!cu_ok (g_drv.ModuleGetFunction (&J.kSplit[q], J.modS, names[q]), "cuModuleGetFunction")) return 1;
    if (!cu_ok (g_drv.FuncSetAttribute (J.kSplit[q], CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int) J.smemBytes[qOf[q]]), "cuFuncSetAttribute")) return 1;
    int nb = 0;
    if (!cu_ok (g_drv.OccupancyMaxActiveBlocksPerMultiprocessor (&nb, J.kSplit[q], J.threads, J.smemBytes[qOf[q]]), "occupancy")) return 1;
    J.blocksPerSMS[q] = std::max (1, nb);
  }
  if (m->opt.get ("verbose", 0)) fprintf (stderr, "[mb_jit] split-mode module compiled\n");
  return 0;
}

static std::string module_source (const mb_machine* m, JitEngine& J, int passC, int pass, int passMinBlocks, int passMinBlocksLin);

// A fitted score module (MB_C = C), on first use.  Returns its index in J.fit, or -1 when it cannot be built (the caller
// falls back to a built-in width).
static const int kMaxFitModules = 3;
static int ensure_fit_module (mb_machine* m, JitEngine& J, int C) {
  for (size_t q = 0; q < J.fit.size(); ++q) if (J.fit[q].C == C) return (int) q;
  for (int c: J.fitFailed) if (c == C) return -1;
  if ((int) J.fit.size() >= kMaxFitModules) return -1;
  JitEngine::FitModule F;
  F.C = C;
  std::vector<char> cubin;
  // wider lanes need more registers: the sums at 3 CTAs per SM (168 registers) as the Viterbi kernels
  const std::string src = module_source (m, J, C, 1, J.minBlocksV, C > 8 ? std::min (J.minBlocksLinV, 3) : J.minBlocksLinV);
  bool ok = !nvrtc_compile (src, ".fit.cu", cubin, nullptr) && cu_ok (g_drv.ModuleLoadData (&F.mod, cubin.data()), "cuModuleLoadData");
  const char* names[4] = { "mb_k_viterbi", "mb_k_forward_lin", "mb_k_backward_lin", "mb_k_viterbi_score" };
  const int qOf[4] = { 2, 5, 6, 9 };
  for (int q = 0; q < 4 && ok; ++q) {
    ok = cu_ok (g_drv.ModuleGetFunction (&F.k[q], F.mod, names[q]), "cuModuleGetFunction")
      && cu_ok (g_drv.FuncSetAttribute (F.k[q], CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int) J.smemBytes[qOf[q]]), "cuFuncSetAttribute");
    int nb = 0;
    ok = ok && cu_ok (g_drv.OccupancyMaxActiveBlocksPerMultiprocessor (&nb, F.k[q], J.threads, J.smemBytes[qOf[q]]), "occupancy");
    F.blocksPerSM[q] = std::max (1, nb);
  }
  if (!ok) { if (F.mod && g_drv.ModuleUnload) g_drv.ModuleUnload (F.mod); J.fitFailed.push_back (C); return -1; }
  J.fit.push_back (F);
  if (m->opt.get ("verbose", 0)) fprintf (stderr, "[mb_jit] score module fitted to the batch compiled: %d columns per lane (strips of %d)\n", C, 32 * C);
  return (int) J.fit.size() - 1;
}

// Columns per lane for a score-only call over `pairs`: the built-in C (narrow) or CV (wide), or a width FITTED to the batch.
// Modelled cost = lane-cells swept (strips * 32 C * (Lo + 32) per pair) * cost per lane-cell, the latter measured on B200
// (100 000 protpsw pairs of 300 aa; ps per lane-cell at C = 4 / 8 / 10): sums 1.16 / 0.92 / 0.97, Viterbi scores 1.33 / 1.17 /
// 1.19, Viterbi with pointers 2.19 / 1.41 / 1.5.  A fitted module costs a compilation (about a second), so it must promise
// 12 % on a batch of at least 256 pairs.  kind: 0 sums, 1 Viterbi + pointers, 2 Viterbi scores.
static int choose_width (mb_machine* m, JitEngine& J, const mb_batch* b, const std::vector<int64_t>& pairs, int kind) {
  if (!J.modV) return J.C;
  if (m->opt.has ("jit_narrow")) return m->opt.get ("jit_narrow", 0) ? J.C : J.CV;
  static const double c4[3] = { 1.16, 2.19, 1.33 }, c8[3] = { 0.92, 1.41, 1.17 };
  auto perCell = [&] (int C) {      // interpolated in 1 / C between the built-in widths, 5 % above the wide one beyond it
    if (C >= J.CV) return C == J.CV ? c8[kind] : 1.05 * c8[kind];
    if (C <= J.C) return c4[kind];
    const double t = (1. / C - 1. / J.CV) / (1. / J.C - 1. / J.CV);
    return c8[kind] + t * (c4[kind] - c8[kind]);
  };
  int64_t maxLi = 0;
  for (int64_t k: pairs) maxLi = std::max (maxLi, b->xOff[k + 1] - b->xOff[k]);
  auto cost = [&] (int C) {
    double cells = 0;
    for (int64_t k: pairs) {
      const double Li = (double) (b->xOff[k + 1] - b->xOff[k]), rows = (double) (b->yOff[k + 1] - b->yOff[k]) + 32;
      cells += std::ceil ((Li + 1) / (32.0 * C)) * 32.0 * C * rows;
    }
    return cells * perCell (C);
  };
  const double costN = cost (J.C), costW = cost (J.CV);
  int best = costN < costW ? J.C : J.CV;
  const double bestBuiltin = std::min (costN, costW);
  const int forced = m->opt.get ("jit_fit_c", -1);      // > 0: this fitted width whenever it holds the batch in one strip; 0: never fit
  const int Cf = forced > 0 ? forced : (int) ((maxLi + 1 + 31) / 32);
  if (forced != 0 && Cf >= 2 && Cf <= 12 && Cf != J.C && Cf != J.CV && Cf * J.tbBytes <= 16 && (int64_t) 32 * Cf >= maxLi + 1
      && (forced > 0 || (pairs.size() >= 256 && cost (Cf) < 0.88 * bestBuiltin)) && ensure_fit_module (m, J, Cf) >= 0) best = Cf;
  return best;
}

// ---- the same run-time compilation plumbing for the other generated engine (mb_big.cu) ----
int rt_compile (const std::string& source, const char* dumpSuffix, std::vector<char>& cubin, std::string* log) { return nvrtc_compile (source, dumpSuffix, cubin, log); }
int rt_load (const std::vector<char>& cubin, void** module) {
  if (!load_driver()) return 1;
  MB_CUDA (cudaFree (0));
  CUmodule mod = nullptr;
  if (!cu_ok (g_drv.ModuleLoadData (&mod, cubin.data()), "cuModuleLoadData")) return 1;
  *module = mod;
  return 0;
}
void rt_unload (void* module) { if (module && g_drv.ModuleUnload) g_drv.ModuleUnload ((CUmodule) module); }
int rt_function (void* module, const char* name, void** fn) {
  CUfunction f = nullptr;
  if (!cu_ok (g_drv.ModuleGetFunction (&f, (CUmodule) module, name), "cuModuleGetFunction")) return 1;
  *fn = f;
  return 0;
}
int rt_global (void* module, const char* name, void** devPtr, size_t* bytes) {
  CUdeviceptr p = 0;
  if (!cu_ok (g_drv.ModuleGetGlobal (&p, bytes, (CUmodule) module, name), "cuModuleGetGlobal")) return 1;
  *devPtr = (void*) p;
  return 0;
}
int rt_prepare (void* fn, int threads, size_t smemBytes, int* blocksPerSM) {
  if (!cu_ok (g_drv.FuncSetAttribute ((CUfunction) fn, CU_FUNC_ATTRIBUTE_MAX_DYNAMIC_SHARED_SIZE_BYTES, (int) smemBytes), "cuFuncSetAttribute")) return 1;
  int nb = 0;
  if (!cu_ok (g_drv.OccupancyMaxActiveBlocksPerMultiprocessor (&nb, (CUfunction) fn, threads, smemBytes), "occupancy")) return 1;
  *blocksPerSM = nb;
  return 0;
}
int rt_launch (void* fn, unsigned grid, unsigned threads, size_t smemBytes, cudaStream_t stream, void** params) {
  return cu_ok (g_drv.LaunchKernel ((CUfunction) fn, grid, 1, 1, threads, 1, 1, (unsigned) smemBytes, (CUstream) stream, params, nullptr), "cuLaunchKernel") ? 0 : 1;
}

// Row-layout tables of one program (Program::WA): the log weights as they are (Viterbi), and the normalised
// linear weights w * sigma_src / sigma_self with sigma from the unit groups (Program::unitSlot).  ok = false when
// a unit group's weight is zero or not finite, or a scale leaves 2^+-100: the normalised kernels must not run then.
struct RowTables { std::vector<double> rowLog, rowLinN, silN; double originInv = 1, resLog = 0; bool ok = true; };

static void row_tables (const mb_machine* m, const Program& p, bool forward, RowTables& r) {
  const int S = m->S;
  const double kLn2 = 0.6931471805599453;
  std::vector<double> ls ((size_t) S, 0.);      // log sigma
  r.ok = true;
  for (int q = 0; q < S; ++q) {
    const int d = forward ? q : S - 1 - q;      // a silent group's source comes earlier in this order
    const int u = p.unitSlot[d];
    if (u < 0) continue;
    const double w = m->lw[p.silId[p.slots[u].silIdx]];
    if (!std::isfinite (w)) { r.ok = false; continue; }
    ls[d] = w + ls[p.slots[u].other];
    if (std::fabs (ls[d]) > 100. * kLn2) r.ok = false;
  }
  auto scaled = [&] (int slot, double w) {      // linear weight of a group's transition in normalised units
    if (!(w > -INFINITY)) return 0.;
    const double lw = w + ls[p.slots[slot].other] - ls[p.slots[slot].self];
    if (!std::isfinite (lw) || std::fabs (lw) > 48. * kLn2) r.ok = false;
    return std::exp (lw);
  };
  r.rowLog.assign (p.rowId.size(), -INFINITY);
  r.rowLinN.assign (p.rowId.size(), 0.);
  for (size_t e = 0; e < p.rowId.size(); ++e) {
    if (p.rowId[e] < 0) continue;
    const double w = m->lw[p.rowId[e]];
    r.rowLog[e] = w + 0.0;      // (-0.0 becomes +0.0: the integer compare of bit patterns needs one zero)
    r.rowLinN[e] = scaled (p.rowSlot[e], w);
  }
  r.silN.assign ((size_t) std::max (p.nSil, 1), 1.);
  for (size_t k = 0; k < p.slots.size(); ++k)
    if (p.slots[k].type == T_SILENT && (int) k != p.unitSlot[p.slots[k].self]) r.silN[p.slots[k].silIdx] = scaled ((int) k, m->lw[p.silId[p.slots[k].silIdx]]);
  const int originState = forward ? 0 : S - 1, resState = forward ? S - 1 : 0;
  r.originInv = std::exp (-ls[originState]);
  r.resLog = ls[resState];
}

static void fill_weights (const mb_machine* m, JitEngine& J, std::vector<double>& ef, std::vector<double>& eb) {
  const double ninf = -INFINITY;
  ef.assign ((size_t) std::max (J.fwd.nEmit, 1), ninf);
  eb.assign ((size_t) std::max (J.bwd.nEmit, 1), ninf);
  for (int q = 0; q < J.fwd.nEmit; ++q) if (J.fwd.emitId[q] >= 0) ef[q] = m->lw[J.fwd.emitId[q]];
  for (int q = 0; q < J.bwd.nEmit; ++q) if (J.bwd.emitId[q] >= 0) eb[q] = m->lw[J.bwd.emitId[q]];
  const int nf = std::max (J.fwd.nSil, 1), nb = std::max (J.bwd.nSil, 1);
  J.silParam.assign ((size_t) (nf + nb) * 8, 0);
  double* sp = (double*) J.silParam.data();
  for (int q = 0; q < J.fwd.nSil; ++q) sp[q] = m->lw[J.fwd.silId[q]] + 0.0;      // (+ 0.0: no negative zero, see row_tables)
  for (int q = 0; q < J.bwd.nSil; ++q) sp[nf + q] = m->lw[J.bwd.silId[q]] + 0.0;
  J.silParamLin.assign (J.silParam.size(), 0);
  double* sl = (double*) J.silParamLin.data();
  for (int q = 0; q < nf + nb; ++q) sl[q] = std::exp (sp[q]);
  // the scaled linear sweep is used only when no finite weight is extreme (see MB_RESCALE in the skeleton)
  J.linearOK = true;
  for (double w: m->lw) if (std::isfinite (w) && std::fabs (w) > 24.0 * 0.6931471805599453) J.linearOK = false;
  for (double w: m->lw) if (std::isnan (w) || w == INFINITY) J.linearOK = false;
  if (m->opt.get ("jit_no_linear", 0)) J.linearOK = false;
}

// score module: row-layout tables and the parameter block of the normalised linear kernels
static int upload_row_tables (const mb_machine* m, JitEngine& J) {
  RowTables f, b;
  row_tables (m, J.fwd, true, f);
  row_tables (m, J.bwd, false, b);
  J.normOK = f.ok && b.ok && J.linearOK && !m->opt.get ("jit_no_norm", 0);
  const int nf = std::max (J.fwd.nSil, 1), nb = std::max (J.bwd.nSil, 1);
  J.silParamLinN.assign ((size_t) (nf + nb + 4) * 8, 0);
  double* sn = (double*) J.silParamLinN.data();
  for (int q = 0; q < nf; ++q) sn[q] = f.silN[q];
  for (int q = 0; q < nb; ++q) sn[nf + q] = b.silN[q];
  sn[nf + nb] = f.originInv; sn[nf + nb + 1] = b.originInv; sn[nf + nb + 2] = f.resLog; sn[nf + nb + 3] = b.resLog;
  if (!J.dRowVit) {
    MB_CUDA (cudaMalloc (&J.dRowVit, f.rowLog.size() * 8));
    MB_CUDA (cudaMalloc (&J.dRowFLinN, f.rowLinN.size() * 8));
    MB_CUDA (cudaMalloc (&J.dRowBLinN, b.rowLinN.size() * 8));
  }
  MB_CUDA (cudaMemcpy (J.dRowVit, f.rowLog.data(), f.rowLog.size() * 8, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (J.dRowFLinN, f.rowLinN.data(), f.rowLinN.size() * 8, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (J.dRowBLinN, b.rowLinN.data(), b.rowLinN.size() * 8, cudaMemcpyHostToDevice));
  return 0;
}

int jit_update_weights (mb_machine* m) {
  if (!m->jit) return 0;
  JitEngine& J = *(JitEngine*) m->jit;
  std::vector<double> ef, eb;
  fill_weights (m, J, ef, eb);
  MB_CUDA (cudaMemcpy (J.dEmitF, ef.data(), ef.size() * 8, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (J.dEmitB, eb.data(), eb.size() * 8, cudaMemcpyHostToDevice));
  for (auto& v: ef) v = std::exp (v);
  for (auto& v: eb) v = std::exp (v);
  MB_CUDA (cudaMemcpy (J.dEmitFLin, ef.data(), ef.size() * 8, cudaMemcpyHostToDevice));
  MB_CUDA (cudaMemcpy (J.dEmitBLin, eb.data(), eb.size() * 8, cudaMemcpyHostToDevice));
  return upload_row_tables (m, J);
}

// layout of the traceback plan on the device (int32): [0..S] stateSlot0, then per slot type, other,
// idOff, then per state shift, bits, then the id table
struct TbPlan {
  const int32_t* stateSlot0;
  const int32_t* slotType;
  const int32_t* slotOther;
  const int32_t* slotIdOff;
  const int32_t* shift;
  const int32_t* bits;
  const int32_t* idTab;
  int32_t S, nOut, tbBytes, W;
  int32_t C, laneBytes;        // sweep order: cell (i, o) at ((strip * (Lo + 32) + o + lane) * 32 + lane) * laneBytes + (i % C) * tbBytes, strip = i / W, lane = (i % W) / C
};

static std::string module_source (const mb_machine* m, JitEngine& J, int passC, int pass, int passMinBlocks, int passMinBlocksLin);

static void generate (const mb_machine* m, JitEngine& J) {
  build_program (m, true, J.fwd);
  build_program (m, false, J.bwd);
  J.shift.assign ((size_t) m->S, 0);
  J.bits.assign ((size_t) m->S, 0);
  int totalBits = 0;
  for (int s = 0; s < m->S; ++s) {
    const int n = J.fwd.stateSlot0[s + 1] - J.fwd.stateSlot0[s];
    int bt = 0; while ((1 << bt) < n) ++bt;
    if (bt && (totalBits >> 5) != ((totalBits + bt - 1) >> 5)) totalBits = (totalBits + 31) & ~31;      // a field stays inside one 32-bit word
    J.shift[s] = totalBits; J.bits[s] = bt; totalBits += bt;
  }
  J.tbBytes = totalBits <= 8 ? 1 : totalBits <= 16 ? 2 : totalBits <= 32 ? 4 : 8;
  J.C = m->S <= 8 ? 4 : 2;
  if (m->opt.has ("jit_c")) J.C = std::max (1, std::min (8, m->opt.get ("jit_c", 4)));
  while (J.C * J.tbBytes > 16) J.C /= 2;
  J.CV = J.C; J.minBlocksV = J.minBlocks;
  if (m->S <= 8 && J.C == 4 && 8 * J.tbBytes <= 16) { J.CV = 8; J.minBlocksV = 3; }
  if (m->opt.has ("jit_cv")) J.CV = std::max (1, std::min (16, m->opt.get ("jit_cv", 8)));
  while (J.CV * J.tbBytes > 16) J.CV /= 2;
  if (m->opt.has ("jit_minblocks_v")) J.minBlocksV = std::max (1, std::min (16, m->opt.get ("jit_minblocks_v", 3)));
  J.minBlocksLinV = std::max (J.minBlocksV, 4);
  if (m->opt.has ("jit_minblocks_linv")) J.minBlocksLinV = std::max (1, std::min (16, m->opt.get ("jit_minblocks_linv", 4)));
  if (m->opt.has ("jit_minblocks")) J.minBlocks = std::max (1, std::min (16, m->opt.get ("jit_minblocks", 4)));
  if (m->opt.has ("jit_minblocks_cnt")) J.minBlocksCnt = std::max (1, std::min (16, m->opt.get ("jit_minblocks_cnt", 4)));
  if (m->opt.has ("jit_minblocks_lin")) J.minBlocksLin = std::max (1, std::min (16, m->opt.get ("jit_minblocks_lin", 5)));
  if (m->opt.has ("jit_threads")) J.threads = std::max (32, std::min (1024, m->opt.get ("jit_threads", 128) / 32 * 32));

  J.ctxBase.assign (J.bwd.slots.size(), -1);
  J.nCtx = 0;
  for (size_t k = 0; k < J.bwd.slots.size(); ++k) {
    const int n = ctx_count (J.bwd.slots[k].type, J.C, m->nOut);
    if (n) { J.ctxBase[k] = J.nCtx; J.nCtx += n; }
  }

  J.source = module_source (m, J, J.C, 0, J.minBlocks, J.minBlocksLin);
  J.sourceV = J.CV != J.C ? module_source (m, J, J.CV, 1, J.minBlocksV, J.minBlocksLinV) : std::string();
  J.sourceS = "#define MB_SPLIT 1\n" + (J.sourceV.empty() ? J.source : J.sourceV);
}

// One module's source: every kernel at passC columns per lane.  pass 0: the first module (E-step and log-domain kernels, and
// the narrow score kernels); pass 1: the score module (frame per lane, steady loop unrolled).
static std::string module_source (const mb_machine* m, JitEngine& J, int passC, int pass, int passMinBlocks, int passMinBlocksLin) {
  std::ostringstream o;
  o << "// generated by machineboss_b200 (mb_jit.cu) for a machine with " << m->S << " states, " << m->T << " transitions\n";
  if (pass) o << "#define MB_SCORE_MODULE 1\n#define MB_LANE_FRAMES 1\n";
  o << "#define MB_ROWTAB 1\n";      // the score kernels of both modules read row-layout tables; the E-step and log-domain kernels keep the indexed ones
  o << "#define MB_STEADY_UNROLL " << std::max (1, std::min (4, m->opt.get ("jit_unroll", pass ? 2 : 1))) << "\n";
  o << "typedef unsigned char uint8_t;\ntypedef int int32_t;\ntypedef long long int64_t;\ntypedef unsigned long long uint64_t;\n";
  o << "#define MB_S " << m->S << "\n#define MB_C " << passC << "\n#define MB_NIN " << m->nIn << "\n#define MB_NOUT " << m->nOut << "\n";
  o << "#define MB_NEMIT_F " << J.fwd.nEmit << "\n#define MB_NEMIT_B " << J.bwd.nEmit << "\n#define MB_TBBYTES " << J.tbBytes << "\n#define MB_THREADS " << J.threads << "\n";
  unsigned long long liveF = 0, liveB = 0;
  for (auto& sl: J.fwd.slots) if (sl.type != T_SILENT) liveF |= 1ull << sl.other;
  for (auto& sl: J.bwd.slots) if (sl.type != T_SILENT) liveB |= 1ull << sl.other;
  o << "#define MB_LIVE_F " << liveF << "ull\n#define MB_LIVE_B " << liveB << "ull\n";
  { const int cb = passC * J.tbBytes; if (cb != 1 && cb != 2 && cb != 4 && cb != 8 && cb != 16) o << "#define MB_TBPAD " << 16 / J.tbBytes << "\n"; }
  o << "#define MB_MINBLOCKS " << passMinBlocks << "\n#ifdef MB_SPLIT\n#define MB_MINBLOCKS_LIN " << std::min (2, passMinBlocksLin) << "      // (the split-mode sums spill below 170 registers)\n#else\n#define MB_MINBLOCKS_LIN "
    << passMinBlocksLin << "\n#endif\n#define MB_MINBLOCKS_CNT " << J.minBlocksCnt << "\n";
  o << "#define MB_NSIL_B " << J.bwd.nSil << "\n#define MB_NCTX " << std::max (J.nCtx, 1) << "\n";
  o << "typedef " << (J.tbBytes <= 4 ? "unsigned" : "unsigned long long") << " mb_tbword;\n";
  o << "struct MBSil { double f[" << std::max (J.fwd.nSil, 1) << "]; double b[" << std::max (J.bwd.nSil, 1) << "]; };\n";
  o << "__device__ __forceinline__ double mb_neg_inf();\n__device__ __forceinline__ double mb_lse (double, double);\n";
  o << "__device__ __forceinline__ float mb_post (double);\n__device__ __forceinline__ float mb_warp_sum (float);\n__device__ __forceinline__ double mb_warp_sum_d (double);\n\n";
  {
    // row-layout emission tables and the normalised linear parameter block (see Program::WA, Program::unitSlot)
    o << "// MB_ROWCELLS_BEGIN (the host harness of tests/test_jit_rowcells_host.py compiles from here to MB_ROWCELLS_END)\n";
    o << "#define MB_WA_F " << J.fwd.WA << "\n#define MB_WB_F " << J.fwd.WB << "\n#define MB_WA_B " << J.bwd.WA << "\n#define MB_WB_B " << J.bwd.WB << "\n";
    o << "struct MBSilN { double f[" << std::max (J.fwd.nSil, 1) << "]; double b[" << std::max (J.bwd.nSil, 1) << "]; double originF, originB, resLogF, resLogB; };\n";
    o << "#ifndef MB_LDS\n"
         "template<int OFF> __device__ __forceinline__ double mb_lds (const unsigned addr) { double v; asm (\"ld.shared.f64 %0, [%1+%2];\" : \"=d\"(v) : \"r\"(addr), \"n\"(OFF)); return v; }\n"
         "#define MB_LDS(addr, off) mb_lds<off> (addr)\n#endif\n";
    o << "#define MB_PKW " << (passC * J.tbBytes + 3) / 4 << "      // 32-bit words of packed back-pointers per lane and step\n";
    o << "#ifndef MB_HOST_HARNESS\n"
         "// n = max (n, t) with the reference's tie-break (a later candidate wins only if strictly greater); with PTR the\n"
         "// winner's field value replaces the field in `word`: (word & ~field) | val, or a plain OR for a one-bit field\n"
         "template<bool PTR> __device__ __forceinline__ void mb_vmax (double& n, const double t, unsigned& word, const unsigned field, const unsigned val) {\n"
         "  if (!PTR) { if (n < t) n = t; return; }\n"
         "  if (field == val) asm (\"{ .reg .pred p; setp.lt.f64 p, %0, %2; selp.f64 %0, %2, %0, p; @p or.b32 %1, %1, %3; }\" : \"+d\"(n), \"+r\"(word) : \"d\"(t), \"r\"(val));\n"
         "  else asm (\"{ .reg .pred p; setp.lt.f64 p, %0, %2; selp.f64 %0, %2, %0, p; @p lop3.b32 %1, %1, %3, %4, 0xEA; }\" : \"+d\"(n), \"+r\"(word) : \"d\"(t), \"r\"(~field), \"r\"(val));\n"
         "}\n#endif\n\n";
    gen_cell_row_vit (o, m, J.fwd, J);
    gen_cell_row_lin (o, m, J.fwd, true);
    gen_cell_row_lin (o, m, J.bwd, false);
    o << "// MB_ROWCELLS_END\n";
  }
  gen_cell (o, m, J.fwd, true, false, J);
  gen_cell (o, m, J.bwd, false, false, J);
  gen_cell (o, m, J.fwd, true, true, J);
  gen_cell_counts (o, m, J);
  gen_cell_lin (o, m, J.fwd, true);
  gen_cell_lin (o, m, J.bwd, false);
  gen_cell_counts_lin (o, m, J);
  gen_fstore_lin (o, m, J);
  o << kJitSkeleton;
  return o.str();
}

// Diagnostic used by the CPU tests: the tables the score module's kernels read, as the host prepares them for
// these weights (no device).  which: 0 forward row-layout log weights (Viterbi), 1 forward / 2 backward row-layout
// normalised linear weights, 3 the log parameter block (f | b), 4 the normalised block (f | b | originF, originB,
// resLogF, resLogB), 5 { normalisation usable, no positive log-weight }.
int jit_host_tables (const mb_machine* m, int which, std::vector<double>& out) {
  std::string why;
  if (!jit_supported (m, &why)) { set_error ("machine not eligible for the JIT engine: " + why); return 1; }
  JitEngine J;
  generate (m, J);
  std::vector<double> ef, eb;
  fill_weights (m, J, ef, eb);
  RowTables f, b;
  row_tables (m, J.fwd, true, f);
  row_tables (m, J.bwd, false, b);
  const int nf = std::max (J.fwd.nSil, 1), nb = std::max (J.bwd.nSil, 1);
  out.clear();
  if (which == 0) out = f.rowLog;
  else if (which == 1) out = f.rowLinN;
  else if (which == 2) out = b.rowLinN;
  else if (which == 3) { const double* sp = (const double*) J.silParam.data(); out.assign (sp, sp + nf + nb); }
  else if (which == 4) {
    out.insert (out.end(), f.silN.begin(), f.silN.begin() + nf);
    out.insert (out.end(), b.silN.begin(), b.silN.begin() + nb);
    out.push_back (f.originInv); out.push_back (b.originInv); out.push_back (f.resLog); out.push_back (b.resLog);
  } else if (which == 5) out.push_back (f.ok && b.ok && J.linearOK ? 1. : 0.);
  else { set_error ("mb_jit_host_tables: which must be 0..5"); return 1; }
  return 0;
}

// Diagnostic used by build() and the CPU tests: generate and NVRTC-compile the kernels of a machine
// structure without touching a device.
int jit_compile_check (const mb_machine* m, std::string* log) {
  std::string why;
  if (!jit_supported (m, &why)) { set_error ("machine not eligible for the JIT engine: " + why); return 1; }
  JitEngine J;
  generate (m, J);
  std::vector<char> cubin;
  if (nvrtc_compile (J.source, "", cubin, log)) return 1;
  if (!J.sourceV.empty()) {
    std::string logV;
    if (nvrtc_compile (J.sourceV, ".viterbi.cu", cubin, &logV)) return 1;
    if (log) *log += "\n---- Viterbi module (MB_C = " + std::to_string (J.CV) + ") ----\n" + logV;
  }
  if (m->opt.get ("jit_split", -1) > 0) {
    std::string logS;
    if (nvrtc_compile (J.sourceS, ".split.cu", cubin, &logS)) return 1;
    if (log) *log += "\n---- split-mode module ----\n" + logS;
  }
  return 0;
}

int jit_prepare (mb_machine* m) {
  JitEngine* Jp = new JitEngine;
  m->jit = Jp;
  JitEngine& J = *Jp;
  generate (m, J);
  if (compile (m, J)) return 1;

  std::vector<double> ef, eb;
  fill_weights (m, J, ef, eb);
  MB_CUDA (cudaMalloc (&J.dEmitF, ef.size() * 8));
  MB_CUDA (cudaMalloc (&J.dEmitB, eb.size() * 8));
  MB_CUDA (cudaMalloc (&J.dEmitFLin, ef.size() * 8));
  MB_CUDA (cudaMalloc (&J.dEmitBLin, eb.size() * 8));
  MB_CUDA (cudaMalloc (&J.dCounter, 8));
  if (jit_update_weights (m)) return 1;
  MB_CUDA (cudaMalloc (&J.dIdTabB, std::max<size_t> (J.bwd.idTab.size(), 1) * 4));
  MB_CUDA (cudaMemcpy (J.dIdTabB, J.bwd.idTab.data(), J.bwd.idTab.size() * 4, cudaMemcpyHostToDevice));
  // traceback plan
  std::vector<int32_t> plan;
  for (int v: J.fwd.stateSlot0) plan.push_back (v);
  for (auto& s: J.fwd.slots) plan.push_back (s.type);
  for (auto& s: J.fwd.slots) plan.push_back (s.other);
  for (auto& s: J.fwd.slots) plan.push_back (s.idOff);
  for (int v: J.shift) plan.push_back (v);
  for (int v: J.bits) plan.push_back (v);
  for (int v: J.fwd.idTab) plan.push_back (v);
  MB_CUDA (cudaMalloc (&J.dTbPlan, std::max<size_t> (plan.size(), 1) * 4));
  MB_CUDA (cudaMemcpy (J.dTbPlan, plan.data(), plan.size() * 4, cudaMemcpyHostToDevice));
  return 0;
}

void jit_destroy (mb_machine* m) {
  if (!m->jit) return;
  JitEngine* J = (JitEngine*) m->jit;
  if (J->mod && g_drv.ModuleUnload) g_drv.ModuleUnload (J->mod);
  if (J->modV && g_drv.ModuleUnload) g_drv.ModuleUnload (J->modV);
  if (J->modS && g_drv.ModuleUnload) g_drv.ModuleUnload (J->modS);
  for (auto& f: J->fit) if (f.mod && g_drv.ModuleUnload) g_drv.ModuleUnload (f.mod);
  if (J->dEmitF) cudaFree (J->dEmitF);
  if (J->dEmitB) cudaFree (J->dEmitB);
  if (J->dEmitFLin) cudaFree (J->dEmitFLin);
  if (J->dEmitBLin) cudaFree (J->dEmitBLin);
  if (J->dTbPlan) cudaFree (J->dTbPlan);
  if (J->dIdTabB) cudaFree (J->dIdTabB);
  if (J->dCounter) cudaFree (J->dCounter);
  if (J->dRowVit) cudaFree (J->dRowVit);
  if (J->dRowFLinN) cudaFree (J->dRowFLinN);
  if (J->dRowBLinN) cudaFree (J->dRowBLinN);
  delete J;
  m->jit = nullptr;
}

// ---------------------------------------------------------------------------------------------
// launches
// ---------------------------------------------------------------------------------------------
struct MBArgsHost {   // must match struct MBArgs in the skeleton
  const uint8_t* x; const int64_t* xOff;
  const uint8_t* y; const int64_t* yOff;
  const int64_t* order; int64_t nWork; unsigned long long* counter;
  double* bnd; int64_t bndStride;
  double* result;
  const double* emit;
  uint8_t* tb; const int64_t* tbOff;
  double* F; const int64_t* fOff;
  const double* ll;
  double* counts;
  const int32_t* idTabB;
  int32_t* flag;
  unsigned* F32; const int64_t* f32Off;
  int32_t* ef; const int64_t* efOff;
  const int64_t* items; const int64_t* itemBnd; int* prog;
};

static std::vector<int64_t> cost_order (const mb_batch* b, const std::vector<int64_t>& pairs) {
  std::vector<int64_t> o = pairs;
  std::stable_sort (o.begin(), o.end(), [&] (int64_t p, int64_t q) {
    const double cp = (double) (b->xOff[p + 1] - b->xOff[p] + 1) * (double) (b->yOff[p + 1] - b->yOff[p] + 1);
    const double cq = (double) (b->xOff[q + 1] - b->xOff[q] + 1) * (double) (b->yOff[q + 1] - b->yOff[q] + 1);
    return cp > cq;
  });
  return o;
}

static const std::vector<int64_t>& full_order (mb_batch* b) {
  if ((int64_t) b->fullOrder.size() != b->nPairs) {
    std::vector<int64_t> all ((size_t) b->nPairs);
    for (int64_t k = 0; k < b->nPairs; ++k) all[k] = k;
    b->fullOrder = cost_order (b, all);
    b->wsOrderHoldsFull = false;
  }
  return b->fullOrder;
}

struct CountArgs { double* F = nullptr; const int64_t* fOff = nullptr; const double* ll = nullptr; double* counts = nullptr; int32_t* flag = nullptr;
                   unsigned* F32 = nullptr; const int64_t* f32Off = nullptr; int32_t* ef = nullptr; const int64_t* efOff = nullptr; };

static int launch (mb_machine* m, mb_batch* b, int which, const std::vector<int64_t>& order, double* dResult, uint8_t* dTb, const int64_t* dTbOff,
                   const CountArgs& ca = CountArgs(), int useC = 0) {      // useC: columns per lane of a score kernel (0: the default module's)
  JitEngine& J = *(JitEngine*) m->jit;
  const bool scoreKernel = which == 2 || which == 5 || which == 6 || which == 9;
  bool narrow = useC == J.C && useC != J.CV;
  const int scoreIdx = which == 2 ? 0 : which == 5 ? 1 : which == 6 ? 2 : 3;
  const JitEngine::FitModule* fitM = nullptr;
  if (scoreKernel && useC && useC != J.C && useC != J.CV) {
    for (auto& f: J.fit) if (f.C == useC) fitM = &f;
    if (!fitM) { set_error ("jit engine: no module fitted to " + std::to_string (useC) + " columns per lane"); return 1; }
  }
  if ((which == 5 || which == 6) && !J.normOK) { set_error ("jit engine: the normalised linear sweep was asked for a machine whose unit weights cannot be divided out"); return 1; }
  narrow = narrow && J.modV && scoreKernel;
  const bool rowTab = scoreKernel;      // the score kernels of both modules read the row-layout tables
  const int slot = which;
  CUfunction fn = narrow ? (which == 2 ? J.kViterbiN : which == 5 ? J.kForwardLinN : which == 6 ? J.kBackwardLinN : J.kViterbiScoreN)
    : which == 9 ? J.kViterbiScore : which == 0 ? J.kForward : which == 1 ? J.kBackward : which == 2 ? J.kViterbi : which == 3 ? J.kFStore : which == 4 ? J.kBCounts : which == 5 ? J.kForwardLin : which == 6 ? J.kBackwardLin : which == 7 ? J.kFStoreLin : J.kBCountsLin;
  const bool lin = which >= 5 && which <= 8;      // 9: the score-only Viterbi, log domain
  int64_t maxLo = 0;
  for (int64_t k: order) maxLo = std::max (maxLo, b->yOff[k + 1] - b->yOff[k]);
  const int warpsPerBlock = J.threads / 32;
  int64_t grid = (int64_t) J.numSMs * (fitM ? fitM->blocksPerSM[scoreIdx] : narrow ? J.blocksPerSMN[scoreIdx] : J.blocksPerSM[slot]);
  if (fitM) fn = fitM->k[scoreIdx];
  // SPLIT mode: with fewer pairs than resident warps the strips of a pair become work items of their own, and the warps
  // that claim them run as a pipeline down the strips (see MBArgs::items in the skeleton)
  const int W = 32 * (scoreKernel && J.modV ? J.CV : J.C);      // (the split module has the score module's columns per lane)
  bool split = false;
  std::vector<int64_t> items, itemBnd;
  if (scoreKernel && !narrow && !fitM && m->opt.get ("jit_split", -1) != 0) {      // (the caller laid out its back-pointers for the strips it chose: narrow strips are never split)
    int64_t nItems = 0;
    for (int64_t k: order) nItems += (b->xOff[k + 1] - b->xOff[k] + W) / W;
    split = nItems > (int64_t) order.size() && (m->opt.get ("jit_split", -1) > 0 || (double) order.size() < 0.75 * (double) (grid * warpsPerBlock));
    if (split) {
      int64_t at = 0;
      for (int64_t k: order) {
        const int64_t nStrips = (b->xOff[k + 1] - b->xOff[k] + W) / W, Lo = b->yOff[k + 1] - b->yOff[k];
        if (nStrips > 0xffff) { split = false; break; }
        for (int64_t st = 0; st < nStrips; ++st) { items.push_back ((k << 16) | st); itemBnd.push_back (at); at += (Lo + 1) * (m->S + 1); }
      }
      itemBnd.push_back (at);
    }
  }
  if (split) {
    if (ensure_split_module (m, J)) return 1;
    const int q = which == 2 ? 0 : which == 5 ? 1 : which == 6 ? 2 : 3;
    fn = J.kSplit[q];
    grid = (int64_t) J.numSMs * J.blocksPerSMS[q];
  }
  const int64_t nWorkItems = split ? (int64_t) items.size() : (int64_t) order.size();
  grid = std::min<int64_t> (grid, (nWorkItems + warpsPerBlock - 1) / warpsPerBlock);
  grid = std::max<int64_t> (grid, 1);
  const int64_t bndStride = 2 * (maxLo + 1) * (m->S + 1);   // the linear sweeps append the frame exponent to each row
  if (ws_bytes (b, WS_ORDER) < order.size() * 8) b->wsOrderHoldsFull = false;   // the slot is about to be re-allocated
  int64_t* dOrder = (int64_t*) ws_reserve (b, WS_ORDER, order.size() * 8);
  double* dBnd = (double*) ws_reserve (b, WS_BND, (size_t) (split ? itemBnd.back() + bndStride : grid * warpsPerBlock * bndStride) * 8);
  unsigned long long* dCounter = (unsigned long long*) ws_reserve (b, WS_COUNTER, 8);
  if (!dOrder || !dBnd || !dCounter) return 1;
  const bool isFull = &order == &b->fullOrder;
  if (!(isFull && b->wsOrderHoldsFull))
    MB_CUDA (cudaMemcpyAsync (dOrder, order.data(), order.size() * 8, cudaMemcpyHostToDevice, b->stream));
  b->wsOrderHoldsFull = isFull;
  MB_CUDA (cudaMemsetAsync (dCounter, 0, 8, b->stream));
  MBArgsHost A;
  A.x = b->dX; A.xOff = b->dXOff; A.y = b->dY; A.yOff = b->dYOff;
  A.order = dOrder; A.nWork = nWorkItems; A.counter = dCounter;
  A.items = nullptr; A.itemBnd = nullptr; A.prog = nullptr;
  if (split) {
    int64_t* dItems = (int64_t*) ws_reserve (b, WS_ITEMS, items.size() * 8);
    int64_t* dItemBnd = (int64_t*) ws_reserve (b, WS_ITEMBND, itemBnd.size() * 8);
    int* dProg = (int*) ws_reserve (b, WS_PROG, items.size() * 4);
    if (!dItems || !dItemBnd || !dProg) return 1;
    MB_CUDA (cudaMemcpyAsync (dItems, items.data(), items.size() * 8, cudaMemcpyHostToDevice, b->stream));
    MB_CUDA (cudaMemcpyAsync (dItemBnd, itemBnd.data(), itemBnd.size() * 8, cudaMemcpyHostToDevice, b->stream));
    MB_CUDA (cudaMemsetAsync (dProg, 0, items.size() * 4, b->stream));
    if (ca.flag) MB_CUDA (cudaMemsetAsync (ca.flag, 0, (size_t) b->nPairs * 4, b->stream));      // strips OR their reasons into the pair's flag
    A.items = dItems; A.itemBnd = dItemBnd; A.prog = dProg;
  }
  A.bnd = dBnd; A.bndStride = bndStride;
  A.result = dResult;
  A.emit = (which == 5 || which == 7) ? J.dEmitFLin : (which == 6 || which == 8) ? J.dEmitBLin : (which == 1 || which == 4) ? J.dEmitB : J.dEmitF;
  if (rowTab) A.emit = which == 5 ? J.dRowFLinN : which == 6 ? J.dRowBLinN : J.dRowVit;
  A.flag = ca.flag;
  A.F32 = ca.F32; A.f32Off = ca.f32Off; A.ef = ca.ef; A.efOff = ca.efOff;
  A.tb = dTb; A.tbOff = dTbOff;
  A.F = ca.F; A.fOff = ca.fOff; A.ll = ca.ll; A.counts = ca.counts; A.idTabB = J.dIdTabB;
  if (m->opt.get ("verbose", 0))
    fprintf (stderr, "[mb_jit] kernel %d%s grid %lld x %d threads, %zu B smem, %d CTAs/SM, C=%d, %zu pairs, bnd %.1f MB\n", which, split ? " (split: strips as work items)" : rowTab && lin ? " (normalised)" : "", (long long) grid, J.threads,
             J.smemBytes[which], J.blocksPerSM[slot], fitM ? fitM->C : ((which == 2 || which == 5 || which == 6 || which == 9) && !narrow) ? J.CV : J.C, order.size(), (double) (grid * warpsPerBlock * bndStride) * 8 / 1e6);
  void* params[2] = { (rowTab && lin) ? (void*) J.silParamLinN.data() : lin ? (void*) J.silParamLin.data() : (void*) J.silParam.data(), (void*) &A };
  if (!cu_ok (g_drv.LaunchKernel (fn, (unsigned) grid, 1, 1, (unsigned) J.threads, 1, 1, (unsigned) J.smemBytes[which], (CUstream) b->stream, params, nullptr), "cuLaunchKernel")) return 1;
  return 0;
}

int jit_forward (mb_machine* m, mb_batch* b, double* loglike, bool backward) {
  JitEngine& J = *(JitEngine*) m->jit;
  if (b->nPairs == 0) return 0;
  const std::vector<int64_t>& order = full_order (b);
  double* dRes = (double*) ws_reserve (b, WS_RESULT, (size_t) b->nPairs * 8);
  if (!dRes) return 1;
  if (timing_begin (b)) return 1;
  int64_t launches = 1;
  if (J.linearOK && J.normOK) {
    // scaled linear-domain sweep (normalised: see Program::unitSlot; a machine whose unit weights cannot be divided
    // out -- a silent transition of weight 0 -- takes the log-domain kernel); pairs it flags (dangerous dynamic
    // range) or scores -inf are re-run with the log-domain kernel, which has no range limit
    int32_t* dFlag = (int32_t*) ws_reserve (b, WS_FLAG, (size_t) b->nPairs * 4);
    if (!dFlag) return 1;
    CountArgs ca;
    ca.flag = dFlag;
    if (launch (m, b, backward ? 6 : 5, order, dRes, nullptr, nullptr, ca, choose_width (m, J, b, order, 0))) return 1;
    std::vector<int32_t> flag ((size_t) b->nPairs);
    MB_CUDA (cudaMemcpyAsync (loglike, dRes, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost, b->stream));
    MB_CUDA (cudaMemcpyAsync (flag.data(), dFlag, (size_t) b->nPairs * 4, cudaMemcpyDeviceToHost, b->stream));
    MB_CUDA (cudaStreamSynchronize (b->stream));
    std::vector<int64_t> redo;
    for (int64_t k = 0; k < b->nPairs; ++k) if (flag[k] || !(loglike[k] > -INFINITY)) redo.push_back (k);
    b->lastRedo = (int64_t) redo.size();
    if (m->opt.get ("verbose", 0) && !redo.empty()) {
      int64_t nf[8] = { 0, 0, 0, 0, 0, 0, 0, 0 };
      for (int64_t k = 0; k < b->nPairs; ++k) ++nf[flag[k] & 7];
      fprintf (stderr, "[mb_jit] linear sweep flagged %lld of %lld pairs; by reason mask (1 spread, 2 neighbour frame, 4 boundary frame) 0..7: %lld %lld %lld %lld %lld %lld %lld %lld\n",
               (long long) redo.size(), (long long) b->nPairs, (long long) nf[0], (long long) nf[1], (long long) nf[2], (long long) nf[3], (long long) nf[4], (long long) nf[5], (long long) nf[6], (long long) nf[7]);
    }
    if (!redo.empty()) {
      if (launch (m, b, backward ? 1 : 0, cost_order (b, redo), dRes, nullptr, nullptr)) return 1;
      ++launches;
    }
  } else { b->lastRedo = 0; if (launch (m, b, backward ? 1 : 0, order, dRes, nullptr, nullptr)) return 1; }
  if (timing_end (b, launches)) return 1;
  MB_CUDA (cudaMemcpy (loglike, dRes, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  return 0;
}

// DPMatrix::traceBack (dpmatrix.defs.h:82-110) over the packed back-pointers written by
// mb_k_viterbi, in two passes.
//   1. jit_traceback_kernel: one thread per pair walks from (Li, Lo, end state) to (0, 0, start
//      state).  The walk is a chain of dependent loads, so it does as little as possible per step:
//      the pointer word of the cell is fetched only when the path moves to another cell (the silent
//      steps of a cell reuse it), the tables it decodes with sit in shared memory, and all it
//      records is the transition GROUP it took, one byte, end-aligned in the pair's scratch slot so
//      that the record reads start -> end.  The pointers a few rows up the diagonal are prefetched
//      into L2 because that is where the path most likely goes.
//   2. jit_path_ids_kernel: one warp per pair turns the groups into transition ids, all steps in
//      parallel: a warp scan of the groups' (input, output) moves gives the cell of every step, the
//      cell gives the tokens, group + tokens give the id (the group's token-indexed id table).
#define TB_MAXS 64
#define TB_MAXSLOTS 256
__global__ void __launch_bounds__(64) jit_traceback_kernel (TbPlan p, int nSlots, DevBatch b, const int64_t* __restrict__ pairs, int64_t nPairsHere,
                                      const uint8_t* __restrict__ tb, const int64_t* __restrict__ tbOff,
                                      const double* __restrict__ score, int64_t* __restrict__ len,
                                      uint8_t* __restrict__ tmp, const int64_t* __restrict__ tmpOff) {
  __shared__ unsigned perState[TB_MAXS + 1];      // shift | bits << 8 | first slot << 16
  __shared__ unsigned char slotMove[TB_MAXSLOTS], slotOther[TB_MAXSLOTS];      // moves: bit 0 input, bit 1 output
  for (int q = threadIdx.x; q <= p.S; q += blockDim.x)
    perState[q] = (q < p.S ? (unsigned) p.shift[q] | ((unsigned) p.bits[q] << 8) : 0u) | ((unsigned) p.stateSlot0[q] << 16);
  for (int q = threadIdx.x; q < nSlots; q += blockDim.x) {
    const int type = p.slotType[q];
    slotMove[q] = (unsigned char) (((type == T_MATCH || type == T_DELETE) ? 1 : 0) | ((type == T_MATCH || type == T_INSERT) ? 2 : 0));
    slotOther[q] = (unsigned char) p.slotOther[q];
  }
  __syncthreads();
  const int64_t slot = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (slot >= nPairsHere) return;
  const int64_t k = pairs[slot];
  const int64_t Li = b.xOff[k + 1] - b.xOff[k], Lo = b.yOff[k + 1] - b.yOff[k];
  const uint8_t* base = tb + tbOff[k];
  uint8_t* out = tmp + tmpOff[slot + 1];     // one past the end of this pair's slot
  int64_t n = 0;
  if (score[k] > -INFINITY) {
    int64_t i = Li, o = Lo;
    int s = p.S - 1;
    auto fetch = [&] (int64_t ii, int64_t oo) {
      const unsigned ui = (unsigned) ii, strip = ui / (unsigned) p.W, within = ui - strip * (unsigned) p.W, lane = within / (unsigned) p.C;      // (32-bit: the walk is a chain of dependent steps, 64-bit divisions would dominate it)
      const uint8_t* wp = base + ((((int64_t) strip * (Lo + 32) + oo + lane) * 32 + lane) * p.laneBytes + (within - lane * (unsigned) p.C) * p.tbBytes);
      // where the path most likely goes: eight cells up the diagonal (the same strip's block sixteen steps back, one lane to the left for 8 columns per lane)
      // (three L1 prefetches there -- the block and the steps before and after it -- were measured: no gain, 14.18 against 14.25 ms)
      if (within >= 8 && oo >= 8) asm volatile ("prefetch.global.L2 [%0];" :: "l"(wp - ((int64_t) (8 + 8 / p.C) * 32 + 8 / p.C) * p.laneBytes));
      unsigned long long w = 0;
      for (int q = 0; q < p.tbBytes; ++q) w |= (unsigned long long) wp[q] << (8 * q);
      return w;
    };
    unsigned long long word = fetch (i, o);
    while (i > 0 || o > 0 || s != 0) {
      const unsigned ps = perState[s];
      const int ptr = (int) ((word >> (ps & 0xffu)) & ((1ull << ((ps >> 8) & 0xffu)) - 1ull));
      const unsigned sl = (ps >> 16) + (unsigned) ptr;
      if (sl >= (perState[s + 1] >> 16)) break;    // corrupt pointer: cannot happen on a finite path
      ++n;
      out[-n] = (uint8_t) sl;
      const unsigned mv = slotMove[sl];
      s = slotOther[sl];
      if (mv) {
        i -= mv & 1u; o -= mv >> 1;
        if (i < 0 || o < 0) break;
        word = fetch (i, o);
      }
    }
  }
  len[slot] = n;
}

// pass 2: one warp per pair; step q of the path (start -> end) took group g[q]; the cell it arrives in is
// the inclusive prefix sum of the groups' moves; its id is idTab[idOff[g] + label (tokens of that cell)]
__global__ void __launch_bounds__(256) jit_path_ids_kernel (TbPlan p, int nSlots, DevBatch b, const int64_t* __restrict__ pairs, int64_t nPairsHere,
                                     const int64_t* __restrict__ len, const uint8_t* __restrict__ tmp, const int64_t* __restrict__ tmpOff,
                                     int32_t* __restrict__ out, const int64_t* __restrict__ outOff) {
  __shared__ int slotIdOff[TB_MAXSLOTS];
  __shared__ unsigned char slotType[TB_MAXSLOTS];
  for (int q = threadIdx.x; q < nSlots; q += blockDim.x) { slotIdOff[q] = p.slotIdOff[q]; slotType[q] = (unsigned char) p.slotType[q]; }
  __syncthreads();
  const int64_t slot = ((int64_t) blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (slot >= nPairsHere) return;
  const int64_t k = pairs[slot];
  const uint8_t* x = b.x + b.xOff[k];
  const uint8_t* y = b.y + b.yOff[k];
  const int64_t n = len[slot];
  const uint8_t* src = tmp + tmpOff[slot + 1] - n;
  int32_t* dst = out + outOff[slot];
  int ci = 0, co = 0;      // cell reached before this chunk of 32 steps
  for (int64_t q0 = 0; q0 < n; q0 += 32) {
    const int64_t q = q0 + lane;
    const int g = q < n ? src[q] : 0;
    const int type = q < n ? slotType[g] : T_SILENT;
    int mv = ((type == T_MATCH || type == T_DELETE) ? 1 : 0) | ((type == T_MATCH || type == T_INSERT) ? 0x10000 : 0);
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int up = __shfl_up_sync (0xffffffffu, mv, d); if (lane >= d) mv += up; }
    const int i = ci + (mv & 0xffff), o = co + (mv >> 16);
    if (q < n) {
      const int a = i ? x[i - 1] - 1 : 0, c = o ? y[o - 1] - 1 : 0;
      const int li = type == T_MATCH ? a * p.nOut + c : type == T_DELETE ? a : type == T_INSERT ? c : 0;
      dst[q] = p.idTab[slotIdOff[g] + li];
    }
    const int tot = __shfl_sync (0xffffffffu, mv, 31);
    ci += tot & 0xffff; co += tot >> 16;
  }
}


static size_t device_total_bytes (int device) {
  static size_t cache[64] = { 0 };
  if (device >= 0 && device < 64 && cache[device]) return cache[device];
  size_t freeB = 0, totalB = 0;
  if (cudaMemGetInfo (&freeB, &totalB) != cudaSuccess) return (size_t) 64 << 30;
  if (device >= 0 && device < 64) cache[device] = totalB;
  return totalB;
}

// How much one chunk of scratch may take.  If what the slot already holds is enough for `wanted`
// no driver query is made (cudaMemGetInfo costs milliseconds with large allocations live).
static double memory_budget (const mb_machine* m, const mb_batch* b, int slot, double wanted, const char* capOption) {
  // a cap set by option (MiB): tests use it to force several chunks
  const double cap = m->opt.has (capOption) ? (double) m->opt.get (capOption, 0) * 1048576.0 : 1e300;
  if (wanted <= (double) ws_bytes (b, slot)) return std::min (cap, (double) ws_bytes (b, slot));
  // a fresh batch of a repeated call (the end-to-end path creates one per call) finds the previous batch's
  // scratch in the pool: no driver query then either (cudaMemGetInfo took 2 - 16 ms with 10 GB live)
  if (wanted <= cap && ws_pool_fits (b->device, (size_t) wanted)) return wanted;
  size_t freeB = 0, totalB = 0;
  if (cudaMemGetInfo (&freeB, &totalB) != cudaSuccess) return 0;
  // the slot's current buffer is released before it grows; at most half the device per chunk, so the
  // scratch can stay attached to the batch between calls (keep_scratch_bytes) without starving others
  return std::min (cap, std::min (0.85 * (double) (freeB + ws_bytes (b, slot) + ws_pool_bytes (b->device)), 0.5 * (double) totalB));
}

// Large scratch (back-pointers, stored Forward values) stays attached to the batch between calls, so
// that repeated calls (EM iterations) do no cudaMalloc, unless it is more than 60 % of the device;
// mb_batch_trim or destroying the batch gives it back.
#define kKeepScratchBytes ((size_t) (0.6 * (double) device_total_bytes (b->device)))

int jit_viterbi (mb_machine* m, mb_batch* b, double* score, int64_t* pathLen) {
  JitEngine& J = *(JitEngine*) m->jit;
  if (b->nPairs == 0) return 0;
  const bool trace = pathLen != nullptr;
  const int useC = choose_width (m, J, b, full_order (b), trace ? 1 : 2);
  if (!trace) {      // scores only (boss -V): no back-pointers, no scratch beyond the strip boundaries
    double* dRes = (double*) ws_reserve (b, WS_RESULT2, (size_t) b->nPairs * 8);
    if (!dRes) return 1;
    if (timing_begin (b)) return 1;
    if (launch (m, b, 9, full_order (b), dRes, nullptr, nullptr, CountArgs(), useC)) return 1;
    if (timing_end (b, 1)) return 1;
    MB_CUDA (cudaMemcpy (score, dRes, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
    return 0;
  }
  const int W = 32 * useC;
  // back-pointer storage in sweep order: per strip (Lo + 32) steps of 32 lanes' groups (a fitted width whose lane bytes are not
  // a power of two: 16 bytes per lane, MB_TBPAD); chunk the batch if it does not fit
  const int laneBytes = useC * J.tbBytes;
  const bool padded = laneBytes != 1 && laneBytes != 2 && laneBytes != 4 && laneBytes != 8 && laneBytes != 16;
  const int64_t stepBytes = 32 * (padded ? 16 : laneBytes);      // one (strip, step) block of pointers
  double wanted = 0;
  for (int64_t k = 0; k < b->nPairs; ++k)
    wanted += (double) (((((b->xOff[k + 1] - b->xOff[k]) + W) / W) * ((b->yOff[k + 1] - b->yOff[k]) + 32) * stepBytes + 255) & ~(int64_t) 255);
  const double budget = memory_budget (m, b, WS_TB, wanted, "jit_tb_budget_mb");
  std::vector<std::vector<int64_t>> chunks (1);
  std::vector<int64_t> tbOffHost ((size_t) b->nPairs, 0);
  std::vector<int64_t> chunkBytes (1, 0);
  for (int64_t k = 0; k < b->nPairs; ++k) {
    const int64_t Li = b->xOff[k + 1] - b->xOff[k], Lo = b->yOff[k + 1] - b->yOff[k];
    int64_t need = ((Li + W) / W) * (Lo + 32) * stepBytes;
    need = (need + 255) & ~(int64_t) 255;
    if ((double) need > budget) { set_error ("pair " + std::to_string (k) + ": Viterbi back-pointers do not fit in device memory"); return 1; }
    if (!chunks.back().empty() && (double) (chunkBytes.back() + need) > budget) { chunks.emplace_back(); chunkBytes.push_back (0); }
    tbOffHost[k] = chunkBytes.back();
    chunkBytes.back() += need;
    chunks.back().push_back (k);
  }
  int64_t maxChunk = 0;
  for (int64_t v: chunkBytes) maxChunk = std::max (maxChunk, v);
  uint8_t* dTb = (uint8_t*) ws_reserve (b, WS_TB, (size_t) maxChunk);
  double* dRes = (double*) ws_reserve (b, WS_RESULT2, (size_t) b->nPairs * 8);
  int64_t* dTbOff = (int64_t*) ws_reserve (b, WS_TBOFF, (size_t) b->nPairs * 8);
  int64_t* dPairs = (int64_t*) ws_reserve (b, WS_PAIRS, (size_t) b->nPairs * 8);
  int64_t* dLen = (int64_t*) ws_reserve (b, WS_LEN, (size_t) b->nPairs * 8);
  int64_t* dOutOff = (int64_t*) ws_reserve (b, WS_OUTOFF, (size_t) b->nPairs * 8);
  if (!dTb || !dRes || !dTbOff || !dPairs || !dLen || !dOutOff) return 1;
  MB_CUDA (cudaMemcpyAsync (dTbOff, tbOffHost.data(), (size_t) b->nPairs * 8, cudaMemcpyHostToDevice, b->stream));
  char* plan = (char*) J.dTbPlan;
  const size_t nSlots = J.fwd.slots.size();
  TbPlan tp;
  tp.stateSlot0 = (const int32_t*) plan;
  tp.slotType = tp.stateSlot0 + (m->S + 1);
  tp.slotOther = tp.slotType + nSlots;
  tp.slotIdOff = tp.slotOther + nSlots;
  tp.shift = tp.slotIdOff + nSlots;
  tp.bits = tp.shift + m->S;
  tp.idTab = tp.bits + m->S;
  tp.S = m->S; tp.nOut = m->nOut; tp.tbBytes = J.tbBytes; tp.W = W;
  tp.C = useC; tp.laneBytes = padded ? 16 : laneBytes;
  int64_t launches = 0;
  double ms = 0;
  for (size_t c = 0; c < chunks.size(); ++c) {
    std::vector<int64_t> chunkOrder;
    if (chunks.size() > 1) chunkOrder = cost_order (b, chunks[c]);
    const std::vector<int64_t>& order = chunks.size() > 1 ? chunkOrder : full_order (b);
    if (timing_begin (b)) return 1;
    if (launch (m, b, 2, order, dRes, dTb, dTbOff, CountArgs(), useC)) return 1;
    ++launches;
    if (trace) {
      const size_t n = chunks[c].size();
      // scratch slots sized for the longest possible path: every loud transition consumes a symbol, and
      // between two of them at most (silent depth) silent transitions fit
      const int64_t depth = (int64_t) m->fwdLevelOff.size() - 1;
      std::vector<int64_t> tmpOff (n + 1, 0);
      for (size_t q = 0; q < n; ++q) {
        const int64_t k = chunks[c][q];
        tmpOff[q + 1] = tmpOff[q] + ((b->xOff[k + 1] - b->xOff[k]) + (b->yOff[k + 1] - b->yOff[k]) + 1) * depth;
      }
      uint8_t* dTmp = (uint8_t*) ws_reserve (b, WS_PATHTMP, (size_t) tmpOff[n]);
      int64_t* dTmpOff = (int64_t*) ws_reserve (b, WS_PATHTMPOFF, (n + 1) * 8);
      if (!dTmp || !dTmpOff) return 1;
      MB_CUDA (cudaMemcpyAsync (dPairs, chunks[c].data(), n * 8, cudaMemcpyHostToDevice, b->stream));
      MB_CUDA (cudaMemcpyAsync (dTmpOff, tmpOff.data(), (n + 1) * 8, cudaMemcpyHostToDevice, b->stream));
      const unsigned tg = (unsigned) ((n + 63) / 64);
      jit_traceback_kernel<<<tg, 64, 0, b->stream>>> (tp, (int) nSlots, b->dev, dPairs, (int64_t) n, dTb, dTbOff, dRes, dLen, dTmp, dTmpOff);
      MB_CUDA (cudaGetLastError());
      if (paths_place (b, chunks[c].data(), (int64_t) n, dLen, dOutOff)) return 1;
      jit_path_ids_kernel<<<(unsigned) ((n * 32 + 255) / 256), 256, 0, b->stream>>> (tp, (int) nSlots, b->dev, dPairs, (int64_t) n, dLen, dTmp, dTmpOff, b->dPaths, dOutOff);
      MB_CUDA (cudaGetLastError());
      launches += 2;
    }
    if (timing_end (b, launches)) return 1;   // synchronises the stream
    ms += b->lastMs;
  }
  b->lastMs = ms;
  b->lastLaunches = launches;
  MB_CUDA (cudaMemcpy (score, dRes, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  if (ws_bytes (b, WS_TB) > kKeepScratchBytes) ws_release (b, WS_TB);
  return 0;
}

// MachineCounts over `pairs` (counts.cpp:37-64) with the log-domain kernels: per pair a Forward sweep
// that stores its FP64 matrix, then the fused Backward + posterior-count sweep.  Counts are ADDED to
// hostCounts, log-likelihoods written to loglike[k].  Chunked by free device memory.
static int counts_log (mb_machine* m, mb_batch* b, const std::vector<int64_t>& pairs, bool wantCounts,
                       std::vector<double>& hostCounts, double* loglike, int64_t& launches, double& ms) {
  if (pairs.empty()) return 0;
  double wanted = 0;
  for (int64_t k: pairs) wanted += 8.0 * (double) (((((b->xOff[k + 1] - b->xOff[k]) + 1) * ((b->yOff[k + 1] - b->yOff[k]) + 1) * m->S) + 31) & ~(int64_t) 31);
  const double budget = memory_budget (m, b, WS_F, wanted, "jit_f_budget_mb") / 8.0;
  std::vector<std::vector<int64_t>> chunks (1);
  std::vector<int64_t> fOffHost ((size_t) b->nPairs, 0), chunkDoubles (1, 0);
  for (int64_t k: pairs) {
    const int64_t Li = b->xOff[k + 1] - b->xOff[k], Lo = b->yOff[k + 1] - b->yOff[k];
    const int64_t need = (((Li + 1) * (Lo + 1) * m->S) + 31) & ~(int64_t) 31;
    if ((double) need > budget) { set_error ("pair " + std::to_string (k) + ": the Forward matrix does not fit in device memory"); return 1; }
    if (!chunks.back().empty() && (double) (chunkDoubles.back() + need) > budget) { chunks.emplace_back(); chunkDoubles.push_back (0); }
    fOffHost[k] = chunkDoubles.back();
    chunkDoubles.back() += need;
    chunks.back().push_back (k);
  }
  int64_t maxChunk = 0;
  for (int64_t v: chunkDoubles) maxChunk = std::max (maxChunk, v);
  const size_t T = (size_t) std::max<int64_t> (m->T, 1);
  double* dF = (double*) ws_reserve (b, WS_F, (size_t) maxChunk * 8);
  double* dLL = (double*) ws_reserve (b, WS_RESULT, (size_t) b->nPairs * 8);
  double* dBack = (double*) ws_reserve (b, WS_RESULT2, (size_t) b->nPairs * 8);
  int64_t* dFOff = (int64_t*) ws_reserve (b, WS_FOFF, (size_t) b->nPairs * 8);
  double* dCounts = (double*) ws_reserve (b, WS_COUNTS, T * 8);
  if (!dF || !dLL || !dBack || !dFOff || !dCounts) return 1;
  MB_CUDA (cudaMemcpyAsync (dFOff, fOffHost.data(), (size_t) b->nPairs * 8, cudaMemcpyHostToDevice, b->stream));
  MB_CUDA (cudaMemsetAsync (dCounts, 0, T * 8, b->stream));
  for (size_t c = 0; c < chunks.size(); ++c) {
    const std::vector<int64_t> order = cost_order (b, chunks[c]);
    CountArgs ca;
    ca.F = dF; ca.fOff = dFOff; ca.ll = dLL; ca.counts = dCounts;
    if (timing_begin (b)) return 1;
    if (launch (m, b, 3, order, dLL, nullptr, nullptr, ca)) return 1;
    ++launches;
    if (wantCounts) { if (launch (m, b, 4, order, dBack, nullptr, nullptr, ca)) return 1; ++launches; }
    if (timing_end (b, launches)) return 1;
    ms += b->lastMs;
  }
  std::vector<double> ll ((size_t) b->nPairs), cnt (T);
  MB_CUDA (cudaMemcpy (ll.data(), dLL, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost));
  for (int64_t k: pairs) loglike[k] = ll[k];
  if (wantCounts) {
    MB_CUDA (cudaMemcpy (cnt.data(), dCounts, T * 8, cudaMemcpyDeviceToHost));
    for (int64_t t = 0; t < m->T; ++t) hostCounts[t] += cnt[t];
  }
  if (ws_bytes (b, WS_F) > kKeepScratchBytes) ws_release (b, WS_F);
  return 0;
}

// The same E-step with the scaled linear-domain kernels: Forward stores the high words of its values
// (4 bytes per cell-state) and the frame of every rescale block; Backward multiplies them back in.
// Pairs the Forward sweep flags, and whole chunks in which the Backward sweep flags a pair, are
// handed to counts_log.
static int counts_lin (mb_machine* m, mb_batch* b, const std::vector<int64_t>& pairs, bool wantCounts,
                       std::vector<double>& hostCounts, double* loglike, int64_t& launches, double& ms) {
  JitEngine& J = *(JitEngine*) m->jit;
  const int W = 32 * J.C;
  double wanted = 0;
  for (int64_t k: pairs)
    wanted += 4.0 * (double) ((((b->xOff[k + 1] - b->xOff[k]) + W) / W) * ((b->yOff[k + 1] - b->yOff[k]) + 32) * (int64_t) (32 * J.C * J.storeQ * 4));
  const double budget = memory_budget (m, b, WS_F, wanted, "jit_f_budget_mb") / 4.0;     // in 32-bit words
  std::vector<std::vector<int64_t>> chunks (1);
  std::vector<int64_t> fOffHost ((size_t) b->nPairs, 0), efOffHost ((size_t) b->nPairs, 0), chunkWords (1, 0), chunkEf (1, 0);
  for (int64_t k: pairs) {
    const int64_t Li = b->xOff[k + 1] - b->xOff[k], Lo = b->yOff[k + 1] - b->yOff[k];
    // one block of 32 lanes x C cells x ceil(S/4) 16-byte chunks per (strip, step), in the order the sweep produces them
    const int64_t need = ((Li + W) / W) * (Lo + 32) * (int64_t) (32 * J.C * J.storeQ * 4);
    const int64_t needEf = ((Li + W) / W) * ((Lo + 32 + 15) / 16);
    if ((double) need > budget) { set_error ("pair " + std::to_string (k) + ": the Forward matrix does not fit in device memory"); return 1; }
    if (!chunks.back().empty() && (double) (chunkWords.back() + need) > budget) { chunks.emplace_back(); chunkWords.push_back (0); chunkEf.push_back (0); }
    fOffHost[k] = chunkWords.back();
    efOffHost[k] = chunkEf.back();
    chunkWords.back() += need;
    chunkEf.back() += needEf;
    chunks.back().push_back (k);
  }
  int64_t maxChunk = 0, maxEf = 0;
  for (int64_t v: chunkWords) maxChunk = std::max (maxChunk, v);
  for (int64_t v: chunkEf) maxEf = std::max (maxEf, v);
  const size_t T = (size_t) std::max<int64_t> (m->T, 1);
  unsigned* dF32 = (unsigned*) ws_reserve (b, WS_F, (size_t) maxChunk * 4);
  int32_t* dEf = (int32_t*) ws_reserve (b, WS_EF, (size_t) std::max<int64_t> (maxEf, 1) * 4);
  double* dLL = (double*) ws_reserve (b, WS_RESULT, (size_t) b->nPairs * 8);
  double* dBack = (double*) ws_reserve (b, WS_RESULT2, (size_t) b->nPairs * 8);
  int64_t* dFOff = (int64_t*) ws_reserve (b, WS_FOFF, (size_t) b->nPairs * 8);
  int64_t* dEfOff = (int64_t*) ws_reserve (b, WS_EFOFF, (size_t) b->nPairs * 8);
  double* dCounts = (double*) ws_reserve (b, WS_COUNTS, T * 8);
  int32_t* dFlag = (int32_t*) ws_reserve (b, WS_FLAG, (size_t) b->nPairs * 4);
  if (!dF32 || !dEf || !dLL || !dBack || !dFOff || !dEfOff || !dCounts || !dFlag) return 1;
  MB_CUDA (cudaMemcpyAsync (dFOff, fOffHost.data(), (size_t) b->nPairs * 8, cudaMemcpyHostToDevice, b->stream));
  MB_CUDA (cudaMemcpyAsync (dEfOff, efOffHost.data(), (size_t) b->nPairs * 8, cudaMemcpyHostToDevice, b->stream));
  std::vector<int64_t> redo;
  std::vector<double> ll ((size_t) b->nPairs), cnt (T);
  std::vector<int32_t> flag ((size_t) b->nPairs);
  for (size_t c = 0; c < chunks.size(); ++c) {
    CountArgs ca;
    ca.F32 = dF32; ca.f32Off = dFOff; ca.ef = dEf; ca.efOff = dEfOff; ca.ll = dLL; ca.counts = dCounts; ca.flag = dFlag;
    if (timing_begin (b)) return 1;
    MB_CUDA (cudaMemsetAsync (dFlag, 0, (size_t) b->nPairs * 4, b->stream));
    if (launch (m, b, 7, cost_order (b, chunks[c]), dLL, nullptr, nullptr, ca)) return 1;
    ++launches;
    MB_CUDA (cudaMemcpyAsync (ll.data(), dLL, (size_t) b->nPairs * 8, cudaMemcpyDeviceToHost, b->stream));
    MB_CUDA (cudaMemcpyAsync (flag.data(), dFlag, (size_t) b->nPairs * 4, cudaMemcpyDeviceToHost, b->stream));
    MB_CUDA (cudaStreamSynchronize (b->stream));
    std::vector<int64_t> good;
    for (int64_t k: chunks[c]) {
      if (flag[k] || !(ll[k] > -INFINITY)) redo.push_back (k);
      else { good.push_back (k); loglike[k] = ll[k]; }
    }
    if (wantCounts && !good.empty()) {
      MB_CUDA (cudaMemsetAsync (dCounts, 0, T * 8, b->stream));
      MB_CUDA (cudaMemsetAsync (dFlag, 0, (size_t) b->nPairs * 4, b->stream));
      if (launch (m, b, 8, cost_order (b, good), dBack, nullptr, nullptr, ca)) return 1;
      ++launches;
      MB_CUDA (cudaMemcpyAsync (flag.data(), dFlag, (size_t) b->nPairs * 4, cudaMemcpyDeviceToHost, b->stream));
      MB_CUDA (cudaMemcpyAsync (cnt.data(), dCounts, T * 8, cudaMemcpyDeviceToHost, b->stream));
      MB_CUDA (cudaStreamSynchronize (b->stream));
      bool anyFlag = false;
      for (int64_t k: good) anyFlag |= flag[k] != 0;
      if (anyFlag) redo.insert (redo.end(), good.begin(), good.end());     // discard this chunk's linear counts
      else for (int64_t t = 0; t < m->T; ++t) hostCounts[t] += cnt[t];
    }
    if (timing_end (b, launches)) return 1;
    ms += b->lastMs;
  }
  if (ws_bytes (b, WS_F) > kKeepScratchBytes) ws_release (b, WS_F);
  b->lastRedo = (int64_t) redo.size();
  std::sort (redo.begin(), redo.end());
  return counts_log (m, b, redo, wantCounts, hostCounts, loglike, launches, ms);
}

int jit_counts (mb_machine* m, mb_batch* b, double* counts, double* loglike) {
  JitEngine& J = *(JitEngine*) m->jit;
  if (counts) for (int64_t t = 0; t < m->T; ++t) counts[t] = 0;
  if (b->nPairs == 0) return 0;
  std::vector<int64_t> all ((size_t) b->nPairs);
  for (int64_t k = 0; k < b->nPairs; ++k) all[k] = k;
  std::vector<double> hostCounts ((size_t) std::max<int64_t> (m->T, 1), 0.), ll ((size_t) b->nPairs, 0.);
  int64_t launches = 0;
  double ms = 0;
  const int rc = J.linearOK ? counts_lin (m, b, all, counts != nullptr, hostCounts, ll.data(), launches, ms)
                            : counts_log (m, b, all, counts != nullptr, hostCounts, ll.data(), launches, ms);
  if (rc) return rc;
  b->lastMs = ms;
  b->lastLaunches = launches;
  if (loglike) for (int64_t k = 0; k < b->nPairs; ++k) loglike[k] = ll[k];
  if (counts) for (int64_t t = 0; t < m->T; ++t) counts[t] = hostCounts[t];
  return 0;
}

}  // namespace mb
