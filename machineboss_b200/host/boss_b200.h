// boss_b200.h -- host-side mirror of the reference's C++ surface for the batched
// Forward / Backward / Viterbi path, on top of the C ABI (include/machineboss_b200.h).
//
// Same names, argument meaning and error behaviour as the reference classes, so code written
// against   EvaluatedMachine / SeqPair / SeqPairList / ForwardMatrix / RollingOutputForwardMatrix /
// BackwardMatrix / ViterbiMatrix / MachineCounts   (src/eval.h:59-98, src/seqpair.h:18-121,
// src/forward.h:8-28, src/backward.h:10-56, src/viterbi.h:8-17, src/counts.h:11-25) keeps working,
// with every DP running on the GPU.  What is NOT mirrored is the symbolic layer (Machine,
// WeightExpr, Params: SURVEY.md section 2 rows 13-15): an EvaluatedMachine is built here from
// numbers -- its flat JSON form, or (states, alphabets, transitions) -- not from Machine + Params.
// INTEGRATION.md shows the ten-line adapter that flattens the reference's own EvaluatedMachine.
//
// Differences a caller can observe, all deliberate:
//   * the fills keep O(strip) state on the device: the first cell(i,o,s) of a matrix fetches it (mb_matrix);
//   * Envelope ARGUMENTS are accepted and, as in the reference (dpmatrix.defs.h:1-27 builds the index
//     mapper from the SeqPair alone), ignored; what restricts a matrix is the SeqPair itself: one
//     that carries an alignment gets the path envelope (Envelope::initPath), as in the reference;
//   * the batched entry points (MachineCounts over a list, forwardLogLikes, viterbiPaths) send
//     the whole SeqPairList to the device in one call instead of looping.
#ifndef MB_HOST_BOSS_B200_H
#define MB_HOST_BOSS_B200_H

#include <cstdint>
#include <fstream>
#include <iostream>
#include <limits>
#include <algorithm>
#include <functional>
#include <list>
#include <map>
#include <queue>
#include <memory>
#include <random>
#include <cmath>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

#include <zlib.h>

#include "../../include/machineboss_b200.h"
#include "mbjson.h"

namespace MachineBoss {

using std::list;
using std::map;
using std::ostream;
using std::runtime_error;
using std::string;
using std::vector;

typedef unsigned long long StateIndex;
typedef string InputSymbol;
typedef string OutputSymbol;
typedef int InputToken;
typedef int OutputToken;
typedef double LogWeight;

// whole file as text; a name ending in .gz is inflated on the way (the larger preset machines ship compressed)
inline string readTextFile (const string& filename) {
  if (filename.size() > 3 && filename.compare (filename.size() - 3, 3, ".gz") == 0) {
    gzFile f = gzopen (filename.c_str(), "rb");
    if (!f) throw std::runtime_error ("File not found: " + filename);
    string text;
    char buf[1 << 16];
    for (int n; (n = gzread (f, buf, sizeof buf)) > 0;) text.append (buf, (size_t) n);
    gzclose (f);
    return text;
  }
  std::ifstream in (filename);
  if (!in) throw std::runtime_error ("File not found: " + filename);
  std::stringstream ss;
  ss << in.rdbuf();
  return ss.str();
}

inline void mbCheck (int rc) { if (rc != 0) throw runtime_error (mb_last_error()); }   // Assert -> Abort -> throw (util.cpp:39-48)

// infinity-safe number printing, default stream precision (src/jsonio.h:14-22)
inline string toInfinitySafeString (double x) {
  if (x == std::numeric_limits<double>::infinity()) return "\"Infinity\"";
  if (x == -std::numeric_limits<double>::infinity()) return "\"-Infinity\"";
  std::ostringstream out;
  out << x;
  return out.str();
}

// ---- Tokenizer (src/eval.h:11-49): token 0 is the empty string, 1..N follow the alphabet order ----
template<typename Symbol, typename Token>
struct Tokenizer {
  vector<Symbol> tok2sym;
  map<Symbol, Token> sym2tok;
  Tokenizer() { tok2sym.push_back (Symbol()); sym2tok[Symbol()] = 0; }
  Tokenizer (const vector<Symbol>& symbols) {
    tok2sym.push_back (Symbol());
    tok2sym.insert (tok2sym.end(), symbols.begin(), symbols.end());
    for (Token tok = 0; tok < (Token) tok2sym.size(); ++tok) sym2tok[tok2sym[tok]] = tok;
  }
  static inline Token emptyToken() { return 0; }
  bool canTokenize (const vector<Symbol>& symSeq) const {
    for (const auto& sym: symSeq) if (!sym2tok.count (sym)) return false;
    return true;
  }
  vector<Token> tokenize (const vector<Symbol>& symSeq) const {
    vector<Token> tokSeq;
    tokSeq.reserve (symSeq.size());
    for (const auto& sym: symSeq) {
      if (!sym2tok.count (sym)) {
        std::ostringstream err;
        err << "Can't tokenize symbol " << sym << " using this alphabet:";
        for (const auto& s: tok2sym) err << ' ' << s;
        throw runtime_error (err.str());
      }
      tokSeq.push_back (sym2tok.at (sym));
    }
    return tokSeq;
  }
  vector<Symbol> detokenize (const vector<Token>& tokSeq) const {
    vector<Symbol> symSeq;
    for (auto tok: tokSeq) symSeq.push_back (tok2sym[tok]);
    return symSeq;
  }
};
typedef Tokenizer<InputSymbol, InputToken> InputTokenizer;
typedef Tokenizer<OutputSymbol, OutputToken> OutputTokenizer;

// ---- sequences (src/seqpair.h:18-73) ----
template<typename Symbol>
struct NamedSeq {
  string name;
  vector<Symbol> seq;
  void readJson (const Json& j) {
    if (j.has ("name")) name = j.at ("name").asString();
    seq.clear();
    for (const auto& s: j.at ("sequence").arr) seq.push_back (s.asString());
  }
  void writeJson (ostream& out) const {
    out << "{\"name\":\"" << name << "\",\"sequence\":[";
    for (size_t n = 0; n < seq.size(); ++n) out << (n > 0 ? "," : "") << "\"" << seq[n] << "\"";
    out << "]}";
  }
};
typedef NamedSeq<InputSymbol> NamedInputSeq;
typedef NamedSeq<OutputSymbol> NamedOutputSeq;

// A transition on a path: what the reference's MachinePath stores per step (machine.h:207-218),
// plus its source state and index so callers can map it back to MachineCounts::count[src][index].
struct MachineTransition {
  InputSymbol in;
  OutputSymbol out;
  StateIndex src = 0, dest = 0;
  size_t transIndex = 0;
  int32_t id = 0;   // global transition id = transOffset[src] + transIndex
  LogWeight logWeight = 0;
  bool inputEmpty() const { return in.empty(); }
  bool outputEmpty() const { return out.empty(); }
  bool isSilent() const { return in.empty() && out.empty(); }
};
typedef list<MachineTransition> TransList;

struct EvaluatedMachine;

struct MachinePath {
  typedef std::pair<InputSymbol, OutputSymbol> AlignCol;
  typedef list<AlignCol> AlignPath;
  TransList trans;
  AlignPath alignment() const {   // seqpair.cpp:59-65
    AlignPath ap;
    for (const auto& t: trans) if (!t.isSilent()) ap.push_back (AlignCol (t.in, t.out));
    return ap;
  }
  void writeJson (ostream& out, const EvaluatedMachine& m) const;   // machine.cpp:1980-1998
};

struct SeqPair {
  typedef MachinePath::AlignCol AlignCol;
  typedef MachinePath::AlignPath AlignPath;
  NamedInputSeq input;
  NamedOutputSeq output;
  AlignPath alignment;
  Json metadata;
  void readJson (const Json& pj) {   // seqpair.cpp:8-38
    input.name = "input";
    output.name = "output";
    if (pj.has ("alignment")) {
      vector<InputSymbol> in;
      vector<OutputSymbol> out;
      for (const auto& col: pj.at ("alignment").arr) {
        const string inSym = col.at (0).asString(), outSym = col.at (1).asString();
        if (inSym.size()) in.push_back (inSym);
        if (outSym.size()) out.push_back (outSym);
        alignment.push_back (AlignCol (inSym, outSym));
      }
      input.seq = in;
      output.seq = out;
      if (pj.has ("input") && pj.at ("input").has ("name")) input.name = pj.at ("input").at ("name").asString();
      if (pj.has ("output") && pj.at ("output").has ("name")) output.name = pj.at ("output").at ("name").asString();
      if (pj.has ("meta")) metadata = pj.at ("meta");
    } else {
      input.readJson (pj.at ("input"));
      output.readJson (pj.at ("output"));
    }
  }
  void writeJson (ostream& out) const {   // seqpair.cpp:40-57
    out << "{\"input\":";
    input.writeJson (out);
    out << ",\"output\":";
    output.writeJson (out);
    if (alignment.size()) {
      out << ",\"alignment\":[";
      size_t n = 0;
      for (const auto& col: alignment) out << (n++ ? "," : "") << "[\"" << Json::escape (col.first) << "\",\"" << Json::escape (col.second) << "\"]";
      out << "]";
    }
    if (!metadata.isNull()) { out << ",\"meta\":"; metadata.write (out); }
    out << "}";
  }
  static SeqPair seqPairFromPath (const MachinePath& mp, const EvaluatedMachine& m, const char* inputName = "input", const char* outputName = "output");
};

struct SeqPairList {
  list<SeqPair> seqPairs;
  void readJson (const Json& pj) { for (const auto& j: pj.arr) { SeqPair sp; sp.readJson (j); seqPairs.push_back (sp); } }
  void writeJson (ostream& out) const {   // seqpair.cpp:251-259
    out << "[";
    size_t n = 0;
    for (const auto& sp: seqPairs) { out << (n++ ? ",\n " : ""); sp.writeJson (out); }
    out << "]";
  }
  static SeqPairList fromFile (const string& filename) {
    SeqPairList l;
    l.readJson (Json::parse (readTextFile (filename)));
    return l;
  }
};

// ---- Envelope (the role of src/seqpair.h:75-113, seqpair.cpp:100-229) ----
// The cells of a pair's matrices that may be used: on output row j the input positions inStart[j] <= i < inEnd[j]
// (row j = after j output symbols, position i = after i input symbols).  Three shapes, as in the reference:
//   full   every cell;
//   path   exactly the cells an alignment passes through: row j runs from the input position at which output
//          symbol j was emitted to the position at which symbol j+1 is about to be;
//   area   the band around an alignment that keeps, on each row, the cells between the match columns `width`
//          matches before and `width` matches after the row's own position in the alignment.
struct Envelope {
  typedef long InputIndex;
  typedef long OutputIndex;
  InputIndex inLen = 0;
  OutputIndex outLen = 0;
  vector<InputIndex> inStart, inEnd;

  Envelope() { setRows (0, 0); }
  Envelope (const SeqPair& sp) {
    if (sp.alignment.empty()) initFull (sp); else initPath (sp.alignment);
    requireFit (sp);
  }
  Envelope (const SeqPair& sp, size_t width) {
    if (sp.alignment.empty()) initFull (sp); else initPathArea (sp.alignment, width);
    requireFit (sp);
  }
  static Envelope fullEnvelope (const SeqPair& sp) { Envelope e; e.initFull (sp); return e; }

  void clear() { setRows (0, 0); }
  void initFull (const SeqPair& sp) { setRows ((InputIndex) sp.input.seq.size(), (OutputIndex) sp.output.seq.size()); }

  // One walk over the alignment columns.  `consumed` counts input symbols so far; a column with an output
  // symbol closes the current row just before it (a match column's own input symbol belongs to the next row)
  // and opens the next row just after it.
  void initPath (const SeqPair::AlignPath& cols) {
    inStart.assign (1, 0);
    inEnd.clear();
    InputIndex consumed = 0;
    for (const auto& col: cols) {
      const bool hasIn = !col.first.empty(), hasOut = !col.second.empty();
      if (hasOut) inEnd.push_back (consumed + 1);
      if (hasIn) ++consumed;
      if (hasOut) inStart.push_back (consumed);
    }
    inEnd.push_back (consumed + 1);
    inLen = consumed;
    outLen = (OutputIndex) inStart.size() - 1;
  }

  // matchAt[k] = input position just before the k-th match column; on row j, seen = matches at or before output
  // symbol j.  The row keeps everything after the match `width + 1` back and up to the match `width` ahead.
  void initPathArea (const SeqPair::AlignPath& cols, size_t width) {
    vector<InputIndex> matchAt;
    vector<size_t> seenOnRow (1, 0);
    InputIndex consumed = 0;
    for (const auto& col: cols) {
      const bool hasIn = !col.first.empty(), hasOut = !col.second.empty();
      if (hasIn && hasOut) matchAt.push_back (consumed);
      if (hasIn) ++consumed;
      if (hasOut) seenOnRow.push_back (matchAt.size());
    }
    setRows (consumed, (OutputIndex) seenOnRow.size() - 1);
    const size_t nMatch = matchAt.size();
    for (size_t j = 0; j < seenOnRow.size(); ++j) {
      const size_t seen = seenOnRow[j];
      if (seen > width) inStart[j] = matchAt[seen - width - 1] + 1;
      if (seen + width < nMatch) inEnd[j] = matchAt[seen + width] + 1;
    }
  }

  bool fits (const SeqPair& sp) const { return inLen == (InputIndex) sp.input.seq.size() && outLen == (OutputIndex) sp.output.seq.size(); }
  static bool overlapping (InputIndex s1, InputIndex e1, InputIndex s2, InputIndex e2) { return s1 < e2 && s2 < e1; }   // half-open intervals share a point
  // A path from (0, 0) to (inLen, outLen) exists inside the envelope's outline: the first row holds position 0,
  // the last row holds inLen, and each row reaches the previous one straight down or diagonally.
  bool connected() const {
    if (!(inStart[0] <= 0 && inEnd[0] > 0)) return false;
    for (OutputIndex j = 1; j <= outLen; ++j)
      if (!overlapping (inStart[j - 1], inEnd[j - 1] + 1, inStart[j], inEnd[j])) return false;
    return inStart[outLen] <= inLen && inEnd[outLen] > inLen;
  }
  bool isFull() const { for (OutputIndex j = 0; j <= outLen; ++j) if (inStart[j] != 0 || inEnd[j] != inLen + 1) return false; return true; }
  void writeJson (ostream& out) const {                 // [[start, end], ...] per output row (seqpair.cpp:224-229)
    out << "[";
    for (OutputIndex j = 0; j <= outLen; ++j) out << (j ? "," : "") << "[" << inStart[j] << "," << inEnd[j] << "]";
    out << "]";
  }

private:
  void setRows (InputIndex nIn, OutputIndex nOut) {     // every row of an nIn x nOut pair, unrestricted
    inLen = nIn; outLen = nOut;
    inStart.assign ((size_t) nOut + 1, 0);
    inEnd.assign ((size_t) nOut + 1, nIn + 1);
  }
  void requireFit (const SeqPair& sp) const { if (!fits (sp)) throw runtime_error ("Envelope/sequence mismatch"); }
};

inline list<Envelope> envelopes (const SeqPairList& l) { list<Envelope> e; for (const auto& sp: l.seqPairs) e.push_back (Envelope (sp)); return e; }                 // seqpair.cpp:231-236
inline list<Envelope> envelopes (const SeqPairList& l, size_t width) { list<Envelope> e; for (const auto& sp: l.seqPairs) e.push_back (Envelope (sp, width)); return e; }   // seqpair.cpp:238-243

// ---- EvaluatedMachine (src/eval.h:59-98) ----
struct EvaluatedMachineState {
  typedef size_t TransIndex;
  Json name;
  TransIndex nTransitions = 0, transOffset = 0;
  vector<LogWeight> logTransWeight;   // indexed by TransIndex
};

struct EvaluatedMachine {
  InputTokenizer inputTokenizer;
  OutputTokenizer outputTokenizer;
  vector<EvaluatedMachineState> state;
  EvaluatedMachineState::TransIndex nTransitions = 0;
  // flat form, enumeration order of eval.cpp:49-69
  vector<int32_t> src, dst, in, out;
  vector<double> logWeight;

  EvaluatedMachine() {}
  // transitions: (src, dest, input symbol, output symbol, log-weight), grouped by ascending src
  EvaluatedMachine (size_t nStates, const vector<InputSymbol>& inAlphabet, const vector<OutputSymbol>& outAlphabet,
                    const vector<MachineTransition>& transitions, const vector<Json>& stateNames = vector<Json>())
    : inputTokenizer (inAlphabet), outputTokenizer (outAlphabet), state (nStates)
  {
    for (size_t s = 0; s < stateNames.size() && s < nStates; ++s) state[s].name = stateNames[s];
    for (const auto& t: transitions) {
      src.push_back ((int32_t) t.src); dst.push_back ((int32_t) t.dest);
      in.push_back (inputTokenizer.sym2tok.at (t.in)); out.push_back (outputTokenizer.sym2tok.at (t.out));
      logWeight.push_back (t.logWeight);
    }
    index();
  }
  // {"nStates":..,"inAlphabet":[..],"outAlphabet":[..],"stateNames":[..],"trans":[[src,dst,inTok,outTok,logWeight,transIndex],..]}
  static EvaluatedMachine fromJson (const Json& j) {
    EvaluatedMachine m;
    vector<InputSymbol> ia;
    vector<OutputSymbol> oa;
    for (const auto& s: j.at ("inAlphabet").arr) ia.push_back (s.asString());
    for (const auto& s: j.at ("outAlphabet").arr) oa.push_back (s.asString());
    m.inputTokenizer = InputTokenizer (ia);
    m.outputTokenizer = OutputTokenizer (oa);
    m.state.resize ((size_t) j.at ("nStates").asInt());
    if (j.has ("stateNames"))
      for (size_t s = 0; s < j.at ("stateNames").size() && s < m.state.size(); ++s) m.state[s].name = j.at ("stateNames").at (s);
    for (const auto& t: j.at ("trans").arr) {
      m.src.push_back ((int32_t) t.at (0).asInt()); m.dst.push_back ((int32_t) t.at (1).asInt());
      m.in.push_back ((int32_t) t.at (2).asInt()); m.out.push_back ((int32_t) t.at (3).asInt());
      m.logWeight.push_back (t.at (4).asNumber());
    }
    m.index();
    return m;
  }
  static EvaluatedMachine fromFile (const string& filename) { return fromJson (Json::parse (readTextFile (filename))); }

  StateIndex nStates() const { return state.size(); }
  StateIndex startState() const { if (!nStates()) throw runtime_error ("EvaluatedMachine has no states"); return 0; }
  StateIndex endState() const { if (!nStates()) throw runtime_error ("EvaluatedMachine has no states"); return nStates() - 1; }
  bool canTokenize (const SeqPair& sp) const { return inputTokenizer.canTokenize (sp.input.seq) && outputTokenizer.canTokenize (sp.output.seq); }
  string stateNameJson (StateIndex s) const { return state[s].name.isNull() ? std::to_string (s) : state[s].name.dump(); }

  MachineTransition transition (int32_t id) const {
    MachineTransition t;
    t.id = id; t.src = (StateIndex) src[id]; t.dest = (StateIndex) dst[id];
    t.in = inputTokenizer.tok2sym[in[id]]; t.out = outputTokenizer.tok2sym[out[id]];
    t.transIndex = (size_t) id - state[src[id]].transOffset;
    t.logWeight = logWeight[id];
    return t;
  }

  // the role of EvaluatedMachineState::incoming (eval.h:68-76): ids of the transitions into `s` labelled
  // (inTok, outTok), by source state then transition index (= ascending id)
  vector<int32_t> incomingIds (StateIndex s, int inTok, int outTok) const {
    vector<int32_t> ids;
    for (size_t t = 0; t < dst.size(); ++t) if ((StateIndex) dst[t] == s && in[t] == inTok && out[t] == outTok) ids.push_back ((int32_t) t);
    return ids;
  }
  // the role of EvaluatedMachineState::outgoing: ids of the transitions out of `s` labelled (inTok, outTok), by destination
  // state, then transition index
  vector<int32_t> outgoingIds (StateIndex s, int inTok, int outTok) const {
    vector<int32_t> ids;
    for (size_t t = state[s].transOffset; t < state[s].transOffset + state[s].nTransitions; ++t) if (in[t] == inTok && out[t] == outTok) ids.push_back ((int32_t) t);
    std::stable_sort (ids.begin(), ids.end(), [&] (int32_t a, int32_t b) { return dst[a] < dst[b]; });
    return ids;
  }
  StateIndex transDest (int32_t id) const { return (StateIndex) dst[id]; }
  StateIndex transSource (int32_t id) const { return (StateIndex) src[id]; }
  double transLogWeight (int32_t id) const { return logWeight[id]; }

  // new log-weights for the same structure (what EvaluatedMachine(machine, params) recomputes per EM iteration)
  void setLogWeights (const vector<double>& lw) {
    if (lw.size() != logWeight.size()) throw runtime_error ("setLogWeights: size mismatch");
    logWeight = lw;
    for (auto& st: state) for (size_t t = 0; t < st.nTransitions; ++t) st.logTransWeight[t] = lw[st.transOffset + t];
    if (dev) mbCheck (mb_machine_update_weights (dev->h, logWeight.data()));
    if (gdev) mbCheck (mb_group_machine_update_weights (gdev->h, logWeight.data()));
  }

  mb_machine* handle() const {   // device copy, created on first use
    if (!dev) {
      std::shared_ptr<Dev> d (new Dev);
      mbCheck (mb_machine_create (&d->h, (int32_t) nStates(), (int32_t) inputTokenizer.tok2sym.size() - 1, (int32_t) outputTokenizer.tok2sym.size() - 1,
                                  (int64_t) src.size(), src.data(), dst.data(), in.data(), out.data(), logWeight.data()));
      dev = d;
    }
    return dev->h;
  }

  mb_gmachine* groupHandle (mb_group* g) const {   // one replica per device of the group, created on first use
    if (!gdev) {
      std::shared_ptr<GDev> d (new GDev);
      mbCheck (mb_group_machine_create (g, &d->h, (int32_t) nStates(), (int32_t) inputTokenizer.tok2sym.size() - 1, (int32_t) outputTokenizer.tok2sym.size() - 1,
                                        (int64_t) src.size(), src.data(), dst.data(), in.data(), out.data(), logWeight.data()));
      gdev = d;
    }
    return gdev->h;
  }

private:
  struct Dev { mb_machine* h = nullptr; ~Dev() { if (h) mb_machine_destroy (h); } };
  struct GDev { mb_gmachine* h = nullptr; ~GDev() { if (h) mb_group_machine_destroy (h); } };
  mutable std::shared_ptr<Dev> dev;
  mutable std::shared_ptr<GDev> gdev;
  void index() {
    nTransitions = src.size();
    for (size_t t = 0; t < src.size(); ++t) {
      if (src[t] < 0 || (size_t) src[t] >= state.size()) throw runtime_error ("EvaluatedMachine: transition source out of range");
      if (t && src[t] < src[t - 1]) throw runtime_error ("EvaluatedMachine: transitions must be grouped by ascending source state");
      state[src[t]].logTransWeight.push_back (logWeight[t]);
    }
    size_t cum = 0;
    for (auto& st: state) { st.nTransitions = st.logTransWeight.size(); st.transOffset = cum; cum += st.nTransitions; }
  }
};

inline void MachinePath::writeJson (ostream& out, const EvaluatedMachine& m) const {
  out << "{\"start\":" << m.startState();
  if (!m.state[m.startState()].name.isNull()) out << ",\"id\":" << m.state[m.startState()].name.dump();
  out << ",\"trans\":[";
  size_t n = 0;
  for (const auto& t: trans) {
    out << (n++ ? "," : "") << "{\"to\":" << t.dest;
    if (!m.state[t.dest].name.isNull()) out << ",\"id\":" << m.state[t.dest].name.dump();
    if (!t.inputEmpty()) out << ",\"in\":\"" << Json::escape (t.in) << "\"";
    if (!t.outputEmpty()) out << ",\"out\":\"" << Json::escape (t.out) << "\"";
    out << "}";
  }
  out << "]}";
}

inline SeqPair SeqPair::seqPairFromPath (const MachinePath& mp, const EvaluatedMachine& m, const char* inputName, const char* outputName) {
  SeqPair sp;   // seqpair.cpp:83-89
  sp.alignment = mp.alignment();
  sp.input.name = inputName;
  sp.output.name = outputName;
  for (const auto& col: sp.alignment) {
    if (col.first.size()) sp.input.seq.push_back (col.first);
    if (col.second.size()) sp.output.seq.push_back (col.second);
  }
  std::ostringstream p;
  mp.writeJson (p, m);
  Json meta;
  meta.type = Json::Object;
  meta.obj["path"] = Json::parse (p.str());   // like the reference, the path goes through a JSON object (keys sorted)
  sp.metadata = meta;
  return sp;
}

// ---- a tokenised SeqPairList on the device ----
class DeviceBatch {
public:
  DeviceBatch (const EvaluatedMachine& m, const vector<const SeqPair*>& pairs) : n ((int64_t) pairs.size()) {
    vector<uint8_t> x, y;
    vector<int64_t> xo (1, 0), yo (1, 0);
    for (const SeqPair* sp: pairs) {
      for (auto t: m.inputTokenizer.tokenize (sp->input.seq)) x.push_back ((uint8_t) t);     // throws on unknown symbols (eval.h:33-37)
      for (auto t: m.outputTokenizer.tokenize (sp->output.seq)) y.push_back ((uint8_t) t);
      xo.push_back ((int64_t) x.size());
      yo.push_back ((int64_t) y.size());
    }
    mbCheck (mb_batch_create (&h, n, x.data(), xo.data(), y.data(), yo.data()));
    // every matrix of a SeqPair that carries an alignment is restricted to the path envelope: the DPMatrix
    // constructors build their index mapper from Envelope(seqPair) (dpmatrix.defs.h:3,17, seqpair.cpp:104-110)
    bool any = false;
    for (const SeqPair* sp: pairs) any = any || sp->alignment.size();
    if (any) {
      vector<int64_t> rowOff (1, 0), st, en;
      for (const SeqPair* sp: pairs) {
        if (sp->alignment.size()) {
          const Envelope env (*sp);
          st.insert (st.end(), env.inStart.begin(), env.inStart.end());
          en.insert (en.end(), env.inEnd.begin(), env.inEnd.end());
        }
        rowOff.push_back ((int64_t) st.size());
      }
      mbCheck (mb_batch_set_envelopes (h, rowOff.data(), st.data(), en.data()));
    }
  }
  ~DeviceBatch() { if (h) mb_batch_destroy (h); }
  DeviceBatch (const DeviceBatch&) = delete;
  DeviceBatch& operator= (const DeviceBatch&) = delete;
  mb_batch* handle() const { return h; }
  int64_t size() const { return n; }
private:
  mb_batch* h = nullptr;
  int64_t n;
};

inline vector<const SeqPair*> pairPointers (const SeqPairList& l) {
  vector<const SeqPair*> v;
  for (const auto& sp: l.seqPairs) v.push_back (&sp);
  return v;
}

// ---- a SeqPairList over every GPU of the box ----
// The reference walks a list in one loop (counts.cpp:37-43, fitter.cpp:23-47, boss.cpp:796,826).  Here the list goes
// to the devices in one piece: with one visible GPU as a DeviceBatch, with several through the C ABI's group entry
// points (pairs dealt longest-first to the least loaded device, a host thread per device, the E-step's counts summed
// with an NCCL all-reduce).  hostGpuLimit() caps the devices used (0 = all visible; the CLI's --gpus).
inline int& hostGpuLimit() { static int limit = 0; return limit; }

inline mb_group* hostGroup() {      // null with a single device
  struct Holder { mb_group* g = nullptr; bool tried = false; ~Holder() { if (g) mb_group_destroy (g); } };
  static Holder h;
  if (!h.tried) {
    h.tried = true;
    int n = 0;
    mbCheck (mb_device_count (&n));
    if (hostGpuLimit() > 0 && hostGpuLimit() < n) n = hostGpuLimit();
    if (n > 1) {
      vector<int32_t> devs;
      for (int d = 0; d < n; ++d) devs.push_back (d);
      mbCheck (mb_group_create (&h.g, devs.data(), (int32_t) devs.size()));
    }
  }
  return h.g;
}

class ListBatch {
public:
  ListBatch (const EvaluatedMachine& m, const vector<const SeqPair*>& pairs) : machine (m), n ((int64_t) pairs.size()) {
    mb_group* g = pairs.size() > 1 ? hostGroup() : nullptr;
    if (!g) { single.reset (new DeviceBatch (m, pairs)); return; }
    vector<uint8_t> x, y;
    vector<int64_t> xo (1, 0), yo (1, 0), rowOff (1, 0), st, en;
    bool anyEnvelope = false;
    for (const SeqPair* sp: pairs) {
      for (auto t: m.inputTokenizer.tokenize (sp->input.seq)) x.push_back ((uint8_t) t);
      for (auto t: m.outputTokenizer.tokenize (sp->output.seq)) y.push_back ((uint8_t) t);
      xo.push_back ((int64_t) x.size());
      yo.push_back ((int64_t) y.size());
      if (sp->alignment.size()) {      // a pair that carries an alignment gets its path envelope, as in DeviceBatch
        const Envelope env (*sp);
        st.insert (st.end(), env.inStart.begin(), env.inStart.end());
        en.insert (en.end(), env.inEnd.begin(), env.inEnd.end());
        anyEnvelope = true;
      }
      rowOff.push_back ((int64_t) st.size());
    }
    x.push_back (0); y.push_back (0);
    mbCheck (mb_group_batch_create (g, &gb, n, x.data(), xo.data(), y.data(), yo.data()));
    if (anyEnvelope) mbCheck (mb_group_batch_set_envelopes (gb, rowOff.data(), st.data(), en.data()));
    gm = m.groupHandle (g);
  }
  ~ListBatch() { if (gb) mb_group_batch_destroy (gb); }
  ListBatch (const ListBatch&) = delete;
  ListBatch& operator= (const ListBatch&) = delete;
  int64_t size() const { return n; }
  bool sharded() const { return gb != nullptr; }
  void forward (double* ll) { if (gb) mbCheck (mb_group_forward (gm, gb, ll)); else mbCheck (mb_forward (machine.handle(), single->handle(), ll)); }
  void viterbi (double* score, int64_t* len) { if (gb) mbCheck (mb_group_viterbi (gm, gb, score, len)); else mbCheck (mb_viterbi (machine.handle(), single->handle(), score, len)); }
  void paths (void* ids, int bytesPerId, const int64_t* off) {
    if (gb) mbCheck (mb_group_viterbi_paths_narrow (gb, ids, bytesPerId, off)); else mbCheck (mb_viterbi_paths_narrow (single->handle(), ids, bytesPerId, off));
  }
  void counts (double* c, double* ll) { if (gb) mbCheck (mb_group_counts (gm, gb, c, ll)); else mbCheck (mb_counts (machine.handle(), single->handle(), c, ll)); }
  // c: [size()][nTransitions], pair k's counts in row k
  void pairCounts (double* c, double* ll) { if (gb) mbCheck (mb_group_pair_counts (gm, gb, c, ll)); else mbCheck (mb_pair_counts (machine.handle(), single->handle(), c, ll)); }
private:
  const EvaluatedMachine& machine;
  int64_t n;
  std::unique_ptr<DeviceBatch> single;
  mb_gbatch* gb = nullptr;
  mb_gmachine* gm = nullptr;
};

// ---- stored matrices: DPMatrix::cell (src/dpmatrix.h:128-146) and the stochastic traceback built on it ----
// The device keeps no matrix for a score; the first cell() fetches the pair's whole matrix (mb_matrix).
class StoredMatrix {
public:
  const EvaluatedMachine& machine;
  const SeqPair& seqPair;
  StoredMatrix (const EvaluatedMachine& m, const SeqPair& sp, int kind) : machine (m), seqPair (sp), kind (kind) {}
  // dpmatrix.h:136-146: -inf outside the matrix
  double cell (long inPos, long outPos, int state) const {
    const long Li = (long) seqPair.input.seq.size(), Lo = (long) seqPair.output.seq.size();
    if (inPos < 0 || inPos > Li || outPos < 0 || outPos > Lo || state < 0 || state >= (int) machine.nStates()) return -std::numeric_limits<double>::infinity();
    fetch();
    return cells[((size_t) outPos * (size_t) (Li + 1) + (size_t) inPos) * (size_t) machine.nStates() + (size_t) state];
  }
protected:
  int kind;
  mutable vector<double> cells;
  void fetch() const {
    if (!cells.empty()) return;
    const size_t Li = seqPair.input.seq.size(), Lo = seqPair.output.seq.size();
    cells.resize ((Li + 1) * (Lo + 1) * (size_t) machine.nStates());
    DeviceBatch b (machine, vector<const SeqPair*> (1, &seqPair));
    mbCheck (mb_matrix (machine.handle(), b.handle(), 0, kind, cells.data()));
  }
public:
  typedef long InputIndex;
  typedef long OutputIndex;
  // called with the cell and state a step starts from (traceBack: the step's source) and the transition's index in
  // that state's list; returning true ends the trace (dpmatrix.h:71)
  typedef std::function<bool (InputIndex, OutputIndex, StateIndex, size_t)> TraceTerminator;
  typedef std::function<size_t (const vector<double>&)> TransSelector;
  static size_t selectMaxTrans (const vector<double>& logWeights) {      // the FIRST maximum (dpmatrix.defs.h:171-174)
    return (size_t) std::distance (logWeights.begin(), std::max_element (logWeights.begin(), logWeights.end()));
  }
  // DPMatrix::traceBack (..., TraceTerminator, TransSelector) (dpmatrix.defs.h:82-110): from (inPos, outPos, s) towards the
  // origin.  Candidates in the reference's order: match, delete, insert, silent sources, each by source state then
  // transition index.  (This is the overload that honours the position; see SURVEY 8a row 10 for the others' quirk.)
  void traceBack (InputIndex i, OutputIndex o, StateIndex s, TraceTerminator stopTrace, TransSelector select = selectMaxTrans) const {
    if (!(cell (i, o, (int) s) > -std::numeric_limits<double>::infinity())) throw runtime_error ("Can't do traceback: no finite-weight paths");
    const vector<InputToken> inTok = machine.inputTokenizer.tokenize (seqPair.input.seq);
    const vector<OutputToken> outTok = machine.outputTokenizer.tokenize (seqPair.output.seq);
    while (i > 0 || o > 0 || s != 0) {
      vector<double> ll;
      vector<int32_t> ids;
      const int a = i ? inTok[i - 1] : 0, c = o ? outTok[o - 1] : 0;
      auto visit = [&] (int wantIn, int wantOut, long pi, long po) {
        for (int32_t id: machine.incomingIds (s, wantIn, wantOut)) { ids.push_back (id); ll.push_back (cell (pi, po, (int) machine.transSource (id)) + machine.transLogWeight (id)); }
      };
      if (i && o) visit (a, c, i - 1, o - 1);
      if (i) visit (a, 0, i - 1, o);
      if (o) visit (0, c, i, o - 1);
      visit (0, 0, i, o);
      if (ids.empty()) throw runtime_error ("traceback: dead end");
      const size_t best = select (ll);
      const MachineTransition t = machine.transition (ids[best < ids.size() ? best : ids.size() - 1]);
      if (!t.inputEmpty()) --i;
      if (!t.outputEmpty()) --o;
      s = t.src;
      if (stopTrace (i, o, s, t.transIndex)) break;
    }
  }
  // DPMatrix::traceForward (dpmatrix.defs.h:128-158) over a Backward matrix: from (inPos, outPos, s) towards the end
  void traceForward (InputIndex i, OutputIndex o, StateIndex s, TraceTerminator stopTrace, TransSelector select = selectMaxTrans) const {
    if (!(cell (i, o, (int) s) > -std::numeric_limits<double>::infinity())) throw runtime_error ("Can't do traceforward: no finite-weight paths");
    const vector<InputToken> inTok = machine.inputTokenizer.tokenize (seqPair.input.seq);
    const vector<OutputToken> outTok = machine.outputTokenizer.tokenize (seqPair.output.seq);
    const long Li = (long) inTok.size(), Lo = (long) outTok.size();
    while (i < Li || o < Lo || s != machine.nStates() - 1) {
      vector<double> ll;
      vector<int32_t> ids;
      const int a = i < Li ? inTok[i] : 0, c = o < Lo ? outTok[o] : 0;
      auto visit = [&] (int wantIn, int wantOut, long ni, long no) {
        for (int32_t id: machine.outgoingIds (s, wantIn, wantOut)) { ids.push_back (id); ll.push_back (cell (ni, no, (int) machine.transDest (id)) + machine.transLogWeight (id)); }
      };
      if (i < Li && o < Lo) visit (a, c, i + 1, o + 1);
      if (i < Li) visit (a, 0, i + 1, o);
      if (o < Lo) visit (0, c, i, o + 1);
      visit (0, 0, i, o);
      if (ids.empty()) throw runtime_error ("traceforward: dead end");
      const size_t best = select (ll);
      const MachineTransition t = machine.transition (ids[best < ids.size() ? best : ids.size() - 1]);
      if (stopTrace (i, o, s, t.transIndex)) break;
      if (!t.inputEmpty()) ++i;
      if (!t.outputEmpty()) ++o;
      s = t.dest;
    }
  }
protected:
  // the whole path from the end cell, as a MachinePath (ViterbiMatrix::path, ForwardMatrix::samplePath)
  template<class Selector>
  MachinePath traceBackWith (Selector select, int s) const {
    list<MachineTransition> rev;
    TraceTerminator collect = [&] (InputIndex, OutputIndex, StateIndex src, size_t ti) {
      rev.push_front (machine.transition ((int32_t) (machine.state[src].transOffset + ti)));
      return false;
    };
    traceBack ((long) seqPair.input.seq.size(), (long) seqPair.output.seq.size(), (StateIndex) s, collect, select);
    MachinePath p;
    p.trans.assign (rev.begin(), rev.end());
    return p;
  }
};

// ---- Forward (src/forward.h:8-28) ----
class ForwardMatrix : public StoredMatrix {
public:
  ForwardMatrix (const EvaluatedMachine& m, const SeqPair& sp) : StoredMatrix (m, sp, MB_MATRIX_FORWARD) { fill(); }
  ForwardMatrix (const EvaluatedMachine& m, const SeqPair& sp, const Envelope&) : StoredMatrix (m, sp, MB_MATRIX_FORWARD) { fill(); }
  double logLike() const { return ll; }
  // ForwardMatrix::samplePath (forward.cpp:17-23): stochastic traceback, candidate weights exp(cell + logWeight),
  // random_index over them with the caller's mt19937 (dpmatrix.defs.h:176-186, util.h:151-165)
  template<class AnyMachine> MachinePath samplePath (const AnyMachine&, std::mt19937& rng) const { return samplePath (rng); }
  // DPMatrix::randomTransSelector (dpmatrix.defs.h:176-186): draws a candidate in proportion to exp (log-weight)
  static TransSelector randomTransSelector (std::mt19937& rng) {
    return [&rng] (const vector<double>& logWeights) -> size_t {
      vector<double> w;
      double norm = 0;
      for (double lw: logWeights) { w.push_back (exp (lw)); norm += w.back(); }
      if (!(norm > 0)) throw runtime_error ("Zero weights in random_index");
      // random_double (util.h:102-106): generator() / (max + 1)
      double variate = (double) rng() / ((double) std::numeric_limits<std::mt19937::result_type>::max() + 1) * norm;
      for (size_t n = 0; n < w.size(); ++n) if ((variate -= w[n]) <= 0) return n;
      return w.size();
    };
  }
  MachinePath samplePath (std::mt19937& rng) const { return traceBackWith (randomTransSelector (rng), (int) machine.nStates() - 1); }
private:
  double ll = 0;
  void fill() {
    DeviceBatch b (machine, vector<const SeqPair*> (1, &seqPair));
    mbCheck (mb_forward (machine.handle(), b.handle(), &ll));
  }
};
typedef ForwardMatrix RollingOutputForwardMatrix;   // forward.h:28: same result, the device never stores the matrix

struct MachineCounts;

// ---- Backward (src/backward.h:10-56) ----
class BackwardMatrix : public StoredMatrix {
public:
  BackwardMatrix (const EvaluatedMachine& m, const SeqPair& sp) : StoredMatrix (m, sp, MB_MATRIX_BACKWARD) { fill(); }
  BackwardMatrix (const EvaluatedMachine& m, const SeqPair& sp, const Envelope&) : StoredMatrix (m, sp, MB_MATRIX_BACKWARD) { fill(); }
  double logLike() const { return ll; }
  void getCounts (const ForwardMatrix&, MachineCounts&) const;   // backward.cpp:58-60
  // ---- consumers of the stored matrices (backward.h:13-34, backward.cpp:52-56,62-108) ----
  // called per (source state, transition index, DESTINATION cell of the transition, posterior probability)
  typedef std::function<void (StateIndex, size_t, InputIndex, OutputIndex, double)> BackTransVisitor;
  struct PostTrans {
    InputIndex inPos;
    OutputIndex outPos;
    StateIndex src;
    size_t transIndex;
    double weight;
    bool operator< (const PostTrans& p) const { return weight < p.weight; }
  };
  typedef std::priority_queue<PostTrans> PostTransQueue;
  // BackwardMatrix::getCounts with a visitor (backward.cpp:62-87): every (cell, outgoing transition) posterior, cells from the
  // end to the origin, states descending, each state's match / delete / insert / silent lists in turn.  Host loop over the two
  // stored matrices (mb_matrix): the per-pair form; sums over a list belong in MachineCounts.
  void getCounts (const ForwardMatrix& forward, const BackTransVisitor& visit) const {
    const vector<InputToken> inTok = machine.inputTokenizer.tokenize (seqPair.input.seq);
    const vector<OutputToken> outTok = machine.outputTokenizer.tokenize (seqPair.output.seq);
    const long Li = (long) inTok.size(), Lo = (long) outTok.size();
    const double total = logLike();
    for (long o = Lo; o >= 0; --o)
      for (long i = Li; i >= 0; --i)
        for (long s = (long) machine.nStates() - 1; s >= 0; --s) {
          const double logOdds = forward.cell (i, o, (int) s) - total;
          auto group = [&] (int wantIn, int wantOut, long ni, long no) {
            for (int32_t id: machine.outgoingIds ((StateIndex) s, wantIn, wantOut))
              visit ((StateIndex) s, (size_t) id - machine.state[s].transOffset, ni, no, exp (logOdds + (cell (ni, no, (int) machine.transDest (id)) + machine.transLogWeight (id))));
          };
          const int a = i < Li ? inTok[i] : 0, c = o < Lo ? outTok[o] : 0;
          if (i < Li && o < Lo) group (a, c, i + 1, o + 1);
          if (i < Li) group (a, 0, i + 1, o);
          if (o < Lo) group (0, c, i, o + 1);
          group (0, 0, i, o);
        }
  }
  PostTransQueue postTransQueue (const ForwardMatrix& forward) const {      // backward.cpp:52-56
    PostTransQueue q;
    getCounts (forward, [&] (StateIndex s, size_t ti, InputIndex ip, OutputIndex op, double w) { q.push (PostTrans { ip, op, s, ti, w }); });
    return q;
  }
  // BackwardMatrix::traceFrom with a TraceTerminator (backward.cpp:98-108): back from (inPos, outPos, state) through the Forward
  // matrix, then the transition itself, then on through this matrix to the end
  void traceFrom (const ForwardMatrix& forward, InputIndex i, OutputIndex o, StateIndex s, size_t transIndex, TraceTerminator stopTrace) const;
private:
  double ll = 0;
  void fill() {
    DeviceBatch b (machine, vector<const SeqPair*> (1, &seqPair));
    mbCheck (mb_backward (machine.handle(), b.handle(), &ll));
  }
};

// ---- Viterbi (src/viterbi.h:8-17) ----
class ViterbiMatrix : public StoredMatrix {
public:
  ViterbiMatrix (const EvaluatedMachine& m, const SeqPair& sp) : StoredMatrix (m, sp, MB_MATRIX_VITERBI) { fill(); }
  ViterbiMatrix (const EvaluatedMachine& m, const SeqPair& sp, const Envelope&) : StoredMatrix (m, sp, MB_MATRIX_VITERBI) { fill(); }
  double logLike() const { return ll; }
  MachinePath path() const {   // viterbi.cpp:49-51 -> traceBack; asserts a finite end cell (dpmatrix.defs.h:84)
    if (!(ll > -std::numeric_limits<double>::infinity())) throw runtime_error ("Can't do traceback: no finite-weight paths");
    MachinePath p;
    for (int32_t id: ids) p.trans.push_back (machine.transition (id));
    return p;
  }
  template<class AnyMachine> MachinePath path (const AnyMachine&) const { return path(); }
private:
  double ll = 0;
  vector<int32_t> ids;
  void fill() {
    DeviceBatch b (machine, vector<const SeqPair*> (1, &seqPair));
    int64_t len = 0, off = 0;
    mbCheck (mb_viterbi (machine.handle(), b.handle(), &ll, &len));
    ids.resize ((size_t) len);
    if (len) mbCheck (mb_viterbi_paths (b.handle(), ids.data(), &off));
  }
};

// ---- E-step accumulator (src/counts.h:11-25, counts.cpp:24-71) ----
struct MachineCounts {
  vector<vector<double> > count;   // indexed: count[state][nTrans]
  double loglike = 0;
  MachineCounts() {}
  MachineCounts (const EvaluatedMachine& m) { init (m); }
  MachineCounts (const EvaluatedMachine& m, const SeqPair& sp) { init (m); (void) add (m, sp); }
  MachineCounts (const EvaluatedMachine& m, const SeqPairList& l, const list<Envelope>& = list<Envelope>()) {
    init (m);
    addBatch (m, pairPointers (l));   // one device call for the whole list (the reference loops, counts.cpp:41-42)
  }
  void init (const EvaluatedMachine& m) {
    loglike = 0;
    count = vector<vector<double> > (m.nStates());
    for (StateIndex s = 0; s < m.nStates(); ++s) count[s].assign (m.state[s].nTransitions, 0.);
  }
  double add (const EvaluatedMachine& m, const SeqPair& sp) { return addBatch (m, vector<const SeqPair*> (1, &sp)); }
  double add (const EvaluatedMachine& m, const SeqPair& sp, const Envelope&) { return add (m, sp); }
  double addBatch (const EvaluatedMachine& m, const vector<const SeqPair*>& pairs) {
    ListBatch b (m, pairs);
    vector<double> c (m.nTransitions ? m.nTransitions : 1, 0.), ll (pairs.size() ? pairs.size() : 1, 0.);
    b.counts (c.data(), ll.data());
    double total = 0;
    for (size_t k = 0; k < pairs.size(); ++k) total += ll[k];
    for (StateIndex s = 0; s < m.nStates(); ++s)
      for (size_t t = 0; t < count[s].size(); ++t) count[s][t] += c[m.state[s].transOffset + t];
    loglike += total;
    return total;
  }
  MachineCounts& operator+= (const MachineCounts& o) {
    for (size_t s = 0; s < count.size(); ++s) for (size_t t = 0; t < count[s].size(); ++t) count[s][t] += o.count[s][t];
    return *this;
  }
  void writeJson (ostream& outs) const {   // counts.cpp:73-78
    outs << "[";
    for (size_t s = 0; s < count.size(); ++s) {
      outs << (s ? ",\n " : "") << "[";
      for (size_t t = 0; t < count[s].size(); ++t) outs << (t ? "," : "") << count[s][t];
      outs << "]";
    }
    outs << "]" << std::endl;
  }
};

inline void BackwardMatrix::traceFrom (const ForwardMatrix& forward, InputIndex i, OutputIndex o, StateIndex s, size_t transIndex, TraceTerminator stopTrace) const {
  if (stopTrace (i, o, s, transIndex)) return;
  forward.traceBack (i, o, s, stopTrace);
  const MachineTransition t = machine.transition ((int32_t) (machine.state[s].transOffset + transIndex));
  traceForward (i + (t.inputEmpty() ? 0 : 1), o + (t.outputEmpty() ? 0 : 1), t.dest, stopTrace);
}

inline void BackwardMatrix::getCounts (const ForwardMatrix&, MachineCounts& counts) const {
  if (counts.count.empty()) counts.init (machine);
  const double before = counts.loglike;
  counts.add (machine, seqPair);
  counts.loglike = before;   // getCounts does not touch loglike (counts.cpp:61-62 adds it in add())
}

// ---- batched entry points (no reference equivalent: the reference loops over the list) ----
inline vector<double> forwardLogLikes (const EvaluatedMachine& m, const SeqPairList& l) {
  ListBatch b (m, pairPointers (l));
  vector<double> ll (l.seqPairs.size());
  if (ll.size()) b.forward (ll.data());
  return ll;
}

inline vector<double> viterbiLogLikes (const EvaluatedMachine& m, const SeqPairList& l, vector<MachinePath>* paths = nullptr) {
  ListBatch b (m, pairPointers (l));
  const size_t n = l.seqPairs.size();
  vector<double> sc (n);
  if (!n) return sc;
  if (!paths) { b.viterbi (sc.data(), nullptr); return sc; }
  vector<int64_t> len (n), off (n + 1, 0);
  b.viterbi (sc.data(), len.data());
  for (size_t k = 0; k < n; ++k) off[k + 1] = off[k] + len[k];
  paths->assign (n, MachinePath());
  if (m.nTransitions <= 256) {      // byte ids: a quarter of the device-to-host copy
    vector<uint8_t> ids ((size_t) off[n] ? (size_t) off[n] : 1);
    if (off[n]) b.paths (ids.data(), 1, off.data());
    for (size_t k = 0; k < n; ++k)
      for (int64_t q = off[k]; q < off[k + 1]; ++q) (*paths)[k].trans.push_back (m.transition ((int32_t) ids[q]));
    return sc;
  }
  vector<int32_t> ids ((size_t) off[n] ? (size_t) off[n] : 1);
  if (off[n]) b.paths (ids.data(), 4, off.data());
  for (size_t k = 0; k < n; ++k)
    for (int64_t q = off[k]; q < off[k + 1]; ++q) (*paths)[k].trans.push_back (m.transition (ids[q]));
  return sc;
}

// nSamples paths per pair drawn from the posterior on the device (mb_sample_paths): path j of pair k is keyed by (seed, k, j), so a
// list gives the same paths on every run and device.  (*loglike)[k] receives pair k's Forward log-likelihood; a pair without
// a finite path gets nSamples empty paths.  One device: the list is not dealt over the box's GPUs.  The reference's
// mt19937 draws are ForwardMatrix::samplePath's.
inline vector<vector<MachinePath> > posteriorPaths (const EvaluatedMachine& m, const SeqPairList& l, int nSamples, uint64_t seed, vector<double>* loglike = nullptr) {
  const size_t n = l.seqPairs.size();
  DeviceBatch b (m, pairPointers (l));
  vector<double> ll (n ? n : 1);
  const size_t nPaths = nSamples > 0 ? n * (size_t) nSamples : 0;
  vector<int64_t> len (nPaths ? nPaths : 1), off (nPaths + 1, 0);
  mbCheck (mb_sample_paths (m.handle(), b.handle(), nSamples, seed, ll.data(), len.data()));
  for (size_t r = 0; r < nPaths; ++r) off[r + 1] = off[r] + len[r];
  if (loglike) loglike->assign (ll.begin(), ll.begin() + n);
  vector<vector<MachinePath> > paths (n, vector<MachinePath> ((size_t) nSamples));
  auto unpack = [&] (const auto& ids) {
    for (size_t r = 0; r < nPaths; ++r)
      for (int64_t q = off[r]; q < off[r + 1]; ++q) paths[r / nSamples][r % nSamples].trans.push_back (m.transition ((int32_t) ids[q]));
  };
  if (m.nTransitions <= 256) {      // byte ids: a quarter of the device-to-host copy
    vector<uint8_t> ids ((size_t) off[nPaths] ? (size_t) off[nPaths] : 1);
    if (off[nPaths]) mbCheck (mb_sampled_paths (b.handle(), ids.data(), 1, off.data()));
    unpack (ids);
  } else {
    vector<int32_t> ids ((size_t) off[nPaths] ? (size_t) off[nPaths] : 1);
    if (off[nPaths]) mbCheck (mb_sampled_paths (b.handle(), ids.data(), 4, off.data()));
    unpack (ids);
  }
  return paths;
}

// The maximum expected accuracy path of each pair, computed for the whole list on the device (mb_mea; definitions in
// include/machineboss_b200.h): (*gain)[k] its gain (-inf, with an empty path, for a pair without a path), (*stepPost)[k] the
// posterior probability of each of its steps, (*loglike)[k] the Forward log-likelihood.  One device, like posteriorPaths.
inline vector<MachinePath> meaPaths (const EvaluatedMachine& m, const SeqPairList& l, vector<double>* gain = nullptr,
                                     vector<vector<double> >* stepPost = nullptr, vector<double>* loglike = nullptr) {
  const size_t n = l.seqPairs.size();
  DeviceBatch b (m, pairPointers (l));
  vector<double> g (n ? n : 1), ll (n ? n : 1);
  vector<int64_t> len (n ? n : 1), off (n + 1, 0);
  mbCheck (mb_mea (m.handle(), b.handle(), g.data(), ll.data(), len.data()));
  for (size_t k = 0; k < n; ++k) off[k + 1] = off[k] + len[k];
  vector<int32_t> ids ((size_t) off[n] ? (size_t) off[n] : 1);
  vector<double> post (ids.size());
  if (off[n]) mbCheck (mb_mea_paths (b.handle(), ids.data(), 4, off.data(), post.data()));
  if (gain) gain->assign (g.begin(), g.begin() + n);
  if (loglike) loglike->assign (ll.begin(), ll.begin() + n);
  if (stepPost) stepPost->assign (n, vector<double>());
  vector<MachinePath> paths (n);
  for (size_t k = 0; k < n; ++k)
    for (int64_t q = off[k]; q < off[k + 1]; ++q) {
      paths[k].trans.push_back (m.transition (ids[q]));
      if (stepPost) (*stepPost)[k].push_back (post[q]);
    }
  return paths;
}

// The posterior probability of each step of paths[k], a path of pair k of the list (mb_path_posteriors), one vector per path.
// One device.
inline vector<vector<double> > pathPosteriors (const EvaluatedMachine& m, const SeqPairList& l, const vector<MachinePath>& paths) {
  if (paths.size() != l.seqPairs.size()) throw runtime_error ("pathPosteriors: one path per pair of the list");
  const size_t n = paths.size();
  vector<vector<double> > out (n);
  if (!n) return out;
  DeviceBatch b (m, pairPointers (l));
  vector<int64_t> pairOf (n), off (n), len (n);
  vector<int32_t> ids;
  for (size_t k = 0; k < n; ++k) {
    pairOf[k] = (int64_t) k;
    off[k] = (int64_t) ids.size();
    for (const auto& t: paths[k].trans) ids.push_back ((int32_t) t.id);
    len[k] = (int64_t) ids.size() - off[k];
  }
  vector<double> post (ids.size() ? ids.size() : 1);
  if (ids.empty()) ids.push_back (0);
  mbCheck (mb_path_posteriors (m.handle(), b.handle(), (int64_t) n, pairOf.data(), ids.data(), off.data(), len.data(), post.data()));
  for (size_t k = 0; k < n; ++k) out[k].assign (post.begin() + off[k], post.begin() + off[k] + len[k]);
  return out;
}

// The MachineCounts of each pair of the list on its own, in list order, from one device call (mb_pair_counts; dealt over the
// box's GPUs like MachineCounts over a list): element k is MachineCounts (m, pair k), its loglike pair k's log-likelihood.
inline vector<MachineCounts> pairCounts (const EvaluatedMachine& m, const SeqPairList& l) {
  const size_t n = l.seqPairs.size(), T = (size_t) m.nTransitions;
  vector<MachineCounts> out (n, MachineCounts (m));
  if (!n) return out;
  ListBatch b (m, pairPointers (l));
  vector<double> c (n * T ? n * T : 1, 0.), ll (n, 0.);
  b.pairCounts (c.data(), ll.data());
  for (size_t k = 0; k < n; ++k) {
    for (StateIndex s = 0; s < m.nStates(); ++s)
      for (size_t t = 0; t < out[k].count[s].size(); ++t) out[k].count[s][t] = c[k * T + m.state[s].transOffset + t];
    out[k].loglike = ll[k];
  }
  return out;
}

// api.h:25-31 equivalents taking an already-evaluated machine
inline double forwardLogLike (const EvaluatedMachine& m, const SeqPair& sp) { return ForwardMatrix (m, sp).logLike(); }
inline double viterbiLogLike (const EvaluatedMachine& m, const SeqPair& sp) { return ViterbiMatrix (m, sp).logLike(); }
inline MachinePath viterbiAlign (const EvaluatedMachine& m, const SeqPair& sp) { return ViterbiMatrix (m, sp).path(); }
inline MachineCounts forwardBackwardCounts (const EvaluatedMachine& m, const SeqPair& sp) { return MachineCounts (m, sp); }
inline MachineCounts forwardBackwardCounts (const EvaluatedMachine& m, const SeqPairList& l) { return MachineCounts (m, l); }

}  // namespace MachineBoss

#endif
