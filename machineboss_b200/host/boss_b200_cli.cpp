// boss_b200_cli.cpp -- the `boss` verbs that reach the DP hot path (target/boss.cpp:725-848),
// running on the B200 engine:
//
//   boss_b200 --evaluated-machine M.json [data options] -L | -V | -A | -C
//   boss_b200 --machine M.json [-P params.json] [-N constraints.json] [-U] [data options] -L | -V | -A | -C | -T
//
//   --machine       a symbolic machine in the reference's basic JSON form (states, transitions with
//                   weight expressions, "defs", "cons"); machine algebra ("compose", ...) is rejected
//   -P, --params    parameter values;  -U, --use-defaults  fill missing ones from the constraints
//                   (boss.cpp:789);  -N, --constraints  for -T
//   -T, --train     Baum-Welch: E-step on the GPU, M-step on the host; prints the fitted parameters
//                   like boss.cpp:776-787
//   -C with --machine prints PARAMETER counts like `boss -C` (counts.cpp:80-106)
//
//   -L, --loglike   Forward log-likelihoods, printed like boss.cpp:792-808:  [["in","out",ll],...]
//   -V, --viterbi   Viterbi log-likelihoods, same layout                     (boss.cpp:819-848)
//   -A, --align     Viterbi alignments as a SeqPairList with meta.path       (boss.cpp:833,843-846)
//   -C, --counts    raw expected transition counts, MachineCounts::writeJson (counts.cpp:73-78)
//   -C --per-pair   a JSON array with one counts object per pair, in list order: each is what -C prints for that pair
//                   alone (pairCounts: the whole list in one device call)
//   --sample-paths SEED   one path per pair drawn from the posterior, ForwardMatrix::samplePath (forward.cpp:17-23)
//   --posterior-paths N [--posterior-seed S]   N paths per pair drawn from the posterior for the whole list at once on the
//                   device (posteriorPaths, default seed 1): [[[transition ids], ...N], ...], [] for a pair without a path
//   --mea           maximum expected accuracy paths for the whole list on the device (meaPaths), one object per pair in list
//                   order: {"input":..,"output":..,"gain":g,"path":[transition ids],"postProb":[posterior of each step]};
//                   "gain":"-Infinity" and empty arrays for a pair that cannot be tokenised or has no path
//   --viterbi-post-prob   per pair, the posterior probability of each step of its Viterbi path (pathPosteriors):
//                   [[p, ...], ...], [] for a pair without one
//                   (boss -C prints PARAMETER counts, which needs the symbolic weight derivatives
//                   of the Machine -- outside this path; see INTEGRATION.md)
//   data: -D/--data pairs.json (a SeqPairList) | --input-fasta X --output-fasta Y |
//         --input-chars S --output-chars S   (all inputs x all outputs, boss.cpp:763-765)
//
// The machine is given already evaluated (flat JSON: states, alphabets, numeric log-weights),
// because building it from a symbolic Machine + Params is the reference's job (INTEGRATION.md).
// Numbers are printed with the stream's default 6 significant digits, like boss (jsonio.h:19-21).
#include <unistd.h>

#include <cstring>
#include <fstream>
#include <iostream>

#include <chrono>

#include <sys/stat.h>
#include "boss_b200_fit.h"
#include "boss_b200_ingest.h"

using namespace MachineBoss;
using namespace std;

static vector<NamedSeq<string> > readFasta (const string& filename) {
  ifstream in (filename);
  if (!in) throw runtime_error ("File not found: " + filename);
  vector<NamedSeq<string> > seqs;
  string line;
  while (getline (in, line)) {
    if (line.size() && line[0] == '>') {
      NamedSeq<string> s;
      const size_t e = line.find_first_of (" \t", 1);
      s.name = line.substr (1, e == string::npos ? string::npos : e - 1);
      seqs.push_back (s);
    } else if (seqs.size())
      for (char c: line) if (!isspace ((unsigned char) c)) seqs.back().seq.push_back (string (1, c));   // splitToChars
  }
  return seqs;
}

static NamedSeq<string> fromChars (const string& s) {
  NamedSeq<string> n;
  n.name = s;
  for (char c: s) n.seq.push_back (string (1, c));
  return n;
}

// The machines of the BASELINE configs ship next to the executable, evaluated by the reference with `boss -U`
// default parameters (machineboss_b200/presets/NAME.eval.json[.gz], written by tools/make_presets.py): the symbolic
// preset library itself (src/preset.cpp) is outside the accelerated path.
static string presetFile (const string& name) {
  char exe[4096];
  const ssize_t n = readlink ("/proc/self/exe", exe, sizeof exe - 1);
  string dir = n > 0 ? string (exe, (size_t) n) : string (".");
  dir = dir.substr (0, dir.find_last_of ('/'));
  for (const char* ext: { ".eval.json", ".eval.json.gz" }) {
    const string path = dir + "/presets/" + name + ext;
    if (std::ifstream (path)) return path;
  }
  throw runtime_error ("no evaluated preset '" + name + "' under " + dir + "/presets (shipped: dnapsw, protpsw, prot2dna_dnapsw, PF00516, PF00516_protpsw)");
}

int main (int argc, char** argv) {
  try {
    string machineFile, symbolicFile, consFile, mstepFile;
    vector<string> dataFiles, paramFiles;
    bool useDefaults = false, doT = false;
    vector<NamedSeq<string> > inSeqs, outSeqs;
    bool doL = false, doV = false, doA = false, doC = false, doSample = false, useApi = false;
    string envMode;
    long long sampleSeed = 1;
    int posteriorN = 0;
    bool doMea = false, doViterbiPost = false;
    unsigned long long posteriorSeed = 1;
    int postTransTop = 0;
    bool doDownsample = false;
    double downsampleSize = 1., downsampleProb = 0.;
    int downsamplePaths = 0;      // > 0: stochastic, that many paths; -1: stochastic, up to nStates paths until the fraction is covered
    unsigned rngSeed = 5489u;     // mt19937's default seed
    string kernelCache;           // empty: none
    bool fastIngest = false, ingestOnly = false;
    bool perPair = false;         // -C: counts of each pair on its own
    string pairedFastaIn, pairedFastaOut;
    for (int a = 1; a < argc; ++a) {
      const string f = argv[a];
      auto next = [&] () -> string { if (a + 1 >= argc) throw runtime_error ("missing value for " + f); return argv[++a]; };
      if (f == "--evaluated-machine" || f == "-m") machineFile = next();
      else if (f == "--preset") machineFile = presetFile (next());      // boss --preset NAME (boss.cpp:247-249), already evaluated with -U defaults
      else if (f == "--machine") symbolicFile = next();
      else if (f == "-P" || f == "--params") paramFiles.push_back (next());
      else if (f == "-N" || f == "--constraints") consFile = next();
      else if (f == "-U" || f == "--use-defaults") useDefaults = true;
      else if (f == "-T" || f == "--train") doT = true;
      else if (f == "--mstep") mstepFile = next();   // one M-step from raw counts [[..],[..]] (no device needed)
      else if (f == "-D" || f == "--data") dataFiles.push_back (next());
      else if (f == "--input-fasta") { for (auto& s: readFasta (next())) inSeqs.push_back (s); }
      else if (f == "--output-fasta") { for (auto& s: readFasta (next())) outSeqs.push_back (s); }
      else if (f == "--input-chars") inSeqs.push_back (fromChars (next()));
      else if (f == "--output-chars") outSeqs.push_back (fromChars (next()));
      else if (f == "-L" || f == "--loglike") doL = true;
      else if (f == "-V" || f == "--viterbi") doV = true;
      else if (f == "-A" || f == "--align") doA = true;
      else if (f == "-C" || f == "--counts") doC = true;
      else if (f == "--per-pair") perPair = true;
      else if (f == "--envelope") envMode = next();      // full | path | <width>: print each pair's Envelope (t/src/testenv.cpp; no device needed)
      else if (f == "--sample-paths") { doSample = true; sampleSeed = atoll (next().c_str()); }
      else if (f == "--posterior-paths") { posteriorN = atoi (next().c_str()); if (posteriorN < 1) throw runtime_error ("--posterior-paths needs a count of at least 1"); }
      else if (f == "--posterior-seed") posteriorSeed = strtoull (next().c_str(), nullptr, 10);
      else if (f == "--mea") doMea = true;
      else if (f == "--viterbi-post-prob") doViterbiPost = true;
      else if (f == "--downsample-size") { doDownsample = true; downsampleSize = atof (next().c_str()); }      // boss.cpp:487-490: which transitions Machine::downsample keeps
      else if (f == "--downsample-prob") { doDownsample = true; downsampleProb = atof (next().c_str()); }
      else if (f == "--downsample-path") { doDownsample = true; downsamplePaths = atoi (next().c_str()); }      // boss.cpp:491-493: sample this many paths (seed: --seed)
      else if (f == "--downsample-frac") { doDownsample = true; downsamplePaths = -1; downsampleSize = atof (next().c_str()); }      // boss.cpp:494-497: sample until this fraction is covered
      else if (f == "--seed") rngSeed = (unsigned) atoll (next().c_str());
      else if (f == "--kernel-cache") kernelCache = next();      // keep the compiled kernels in this directory between runs (e.g. ~/.cache/machineboss_b200)
      else if (f == "--post-trans") postTransTop = atoi (next().c_str());      // the top of BackwardMatrix::postTransQueue and the trace from its first entry
      else if (f == "--device") mbCheck (mb_set_device (atoi (next().c_str())));
      else if (f == "--fast-ingest") fastIngest = true;      // -D lists go straight to packed tokens (boss_b200_ingest.h); -L / -V only
      else if (f == "--paired-fasta") { fastIngest = true; pairedFastaIn = next(); pairedFastaOut = next(); }      // record k of one file with record k of the other
      else if (f == "--ingest-only") { fastIngest = true; ingestOnly = true; }      // time the ingest, touch no device
      else if (f == "--api") useApi = true;      // route the verbs through the api.h free functions (Machine, Params, SeqPair), pair by pair
      else if (f == "--gpus") hostGpuLimit() = atoi (next().c_str());      // lists of pairs use this many GPUs (default: every visible one)
      else if (f == "-h" || f == "--help") { cout << "usage: boss_b200 --evaluated-machine M.json [-D pairs.json | --input-fasta X --output-fasta Y | --input-chars S --output-chars S] -L|-V|-A|-C" << endl; return 0; }
      else throw runtime_error ("unknown option " + f);
    }
    // The kernels a machine's structure is compiled into (NVRTC, seconds) are kept between runs of this program, as a command-line
    // call is one process per batch -- when --kernel-cache names a directory (the library caches nothing unless told to).
    if (!kernelCache.empty()) {
      string made;
      for (size_t q = 1; q <= kernelCache.size(); ++q)
        if (q == kernelCache.size() || kernelCache[q] == '/') { made = kernelCache.substr (0, q); mkdir (made.c_str(), 0755); }      // (errors show up as cache misses)
      mb_set_kernel_cache_dir (kernelCache.c_str());
    }
    if (envMode.size()) {
      SeqPairList data;
      for (const auto& df: dataFiles) { SeqPairList l = SeqPairList::fromFile (df); data.seqPairs.insert (data.seqPairs.end(), l.seqPairs.begin(), l.seqPairs.end()); }
      size_t k = 0;
      for (const auto& sp: data.seqPairs) {
        const Envelope env = envMode == "full" ? Envelope::fullEnvelope (sp) : envMode == "path" ? Envelope (sp) : Envelope (sp, (size_t) atoi (envMode.c_str()));
        if (!env.connected()) throw runtime_error ("Envelope is not connected");
        cout << (k++ ? "\n" : "");
        env.writeJson (cout);
      }
      cout << endl;
      return EXIT_SUCCESS;
    }
    if (machineFile.empty() && symbolicFile.empty()) throw runtime_error ("please specify --evaluated-machine or --machine");
    Machine machine;
    Params seed, params;
    Constraints constraints;
    const bool symbolic = !symbolicFile.empty();
    if (symbolic) {
      machine = Machine::fromFile (symbolicFile);
      for (const auto& pf: paramFiles) seed = seed.combine (Params::fromFile (pf));
      if (consFile.size()) constraints = Constraints::fromFile (consFile);
      params = machine.funcs.combine (seed).combine (machine.getParamDefs (useDefaults));    // boss.cpp:789
    } else if (doT) throw runtime_error ("-T needs a symbolic --machine");

    if (mstepFile.size()) {   // MachineObjective::optimize on given counts (counts.cpp:225-295)
      if (!symbolic) throw runtime_error ("--mstep needs a symbolic --machine");
      std::ifstream cf (mstepFile);
      if (!cf) throw runtime_error ("File not found: " + mstepFile);
      std::stringstream ss; ss << cf.rdbuf();
      const Json cj = Json::parse (ss.str());
      MachineCounts counts;
      for (const auto& row: cj.arr) { counts.count.push_back (vector<double>()); for (const auto& v: row.arr) counts.count.back().push_back (v.asNumber()); }
      if (counts.count.size() != machine.nStates()) throw runtime_error ("Number of states mismatch");
      const Params start = machine.cons.combine (constraints).defaultParams().combine (seed, true);
      const MachineObjective objective (machine, counts, constraints, machine.funcs);
      objective.optimize (start).writeJson (cout);
      cout << endl;
      return EXIT_SUCCESS;
    }

    if (doDownsample) {   // Machine::downsample's selection (machine.cpp:2036-2082) on a symbolic, toposorted, acyclic machine
      if (!symbolic) throw runtime_error ("--downsample-size / --downsample-prob need a symbolic --machine");
      Machine withParams = machine;
      withParams.funcs = machine.funcs.combine (seed, true);
      std::mt19937 rng (rngSeed);
      const vector<vector<bool>> allowed = downsamplePaths ? stochasticDownsampleTransitions (withParams, rng, downsampleSize, downsamplePaths > 0 ? downsamplePaths : (int) machine.nStates())
                                                           : downsampleTransitions (withParams, downsampleSize, downsampleProb);
      size_t kept = 0, total = 0;
      for (const auto& row: allowed) for (bool v: row) { ++total; if (v) ++kept; }
      cout << "{\"nTransitions\":" << total << ",\"kept\":" << kept << ",\"allowed\":[";
      for (size_t s = 0; s < allowed.size(); ++s) {
        cout << (s ? "," : "") << "[";
        for (size_t t = 0; t < allowed[s].size(); ++t) cout << (t ? "," : "") << (allowed[s][t] ? 1 : 0);
        cout << "]";
      }
      cout << "]}" << endl;
      return EXIT_SUCCESS;
    }

    EvaluatedMachine eval;
    if (!symbolic) eval = EvaluatedMachine::fromFile (machineFile);
    else if (!doT) eval = evaluate (machine, params);
    else {   // only the alphabets are needed to assemble the data
      Params any = machine.funcs.combine (seed).combine (machine.cons.combine (constraints).defaultParams(), false);
      eval = evaluate (machine, any);
    }

    if (fastIngest) {      // lists at scale: files -> packed tokens -> device, no SeqPair objects in between
      const auto t0 = std::chrono::steady_clock::now();
      PackedPairs pp;
      size_t fileBytes = 0;
      if (pairedFastaIn.size()) {
        const string a = readTextFile (pairedFastaIn), b = readTextFile (pairedFastaOut);
        fileBytes = a.size() + b.size();
        pp = packedFromFasta (a, b, eval);
      } else {
        if (dataFiles.size() != 1) throw runtime_error ("--fast-ingest takes one -D file (or --paired-fasta)");
        const string text = readTextFile (dataFiles[0]);
        fileBytes = text.size();
        pp = packedFromSeqPairListJson (text, eval);
      }
      const double secs = std::chrono::duration<double> (std::chrono::steady_clock::now() - t0).count();
      if (ingestOnly) {
        cout << "{\"pairs\":" << pp.size() << ",\"residues\":" << pp.residues() << ",\"file_bytes\":" << fileBytes << ",\"seconds\":" << secs
             << ",\"pairs_per_s\":" << (double) pp.size() / secs << ",\"MB_per_s\":" << (double) fileBytes / 1e6 / secs << "}" << endl;
        return EXIT_SUCCESS;
      }
      if (!(doL || doV) || doA || doC || doT) throw runtime_error ("--fast-ingest serves -L and -V");
      for (int pass = 0; pass < 2; ++pass) {
        if (!(pass ? doV : doL)) continue;
        const vector<double> sc = packedScores (eval, pp, pass == 1);
        cout << "[";
        for (size_t k = 0; k < pp.size(); ++k)
          cout << (k ? ",\n " : "") << "[\"" << Json::escape (pp.xName[k]) << "\",\"" << Json::escape (pp.yName[k]) << "\"," << toInfinitySafeString (sc[k]) << "]";
        cout << "]\n";
      }
      return EXIT_SUCCESS;
    }
    SeqPairList data;
    for (const auto& df: dataFiles) { SeqPairList l = SeqPairList::fromFile (df); data.seqPairs.insert (data.seqPairs.end(), l.seqPairs.begin(), l.seqPairs.end()); }
    const bool inputEmpty = eval.inputTokenizer.tok2sym.size() == 1, outputEmpty = eval.outputTokenizer.tok2sym.size() == 1;
    if (inSeqs.empty() && inputEmpty && !outSeqs.empty()) inSeqs.push_back (NamedSeq<string>());    // boss.cpp:757-760
    if (outSeqs.empty() && !inSeqs.empty() && outputEmpty) outSeqs.push_back (NamedSeq<string>());
    for (const auto& i: inSeqs) for (const auto& o: outSeqs) { SeqPair sp; sp.input = i; sp.output = o; data.seqPairs.push_back (sp); }
    if (data.seqPairs.empty() && inputEmpty && outputEmpty) data.seqPairs.push_back (SeqPair());   // boss.cpp:769-770
    if (data.seqPairs.empty()) throw runtime_error ("no sequence data given");
    if (!(doL || doV || doA || doC || doT || doSample || posteriorN || doMea || doViterbiPost || postTransTop)) throw runtime_error ("nothing to do: give -L, -V, -A, -C or -T");
    if (perPair && !doC) throw runtime_error ("--per-pair goes with -C");

    if (doT) {   // boss.cpp:776-787
      if (constraints.empty() && machine.cons.empty()) throw runtime_error ("To fit parameters, please specify a constraints file and (for machines with input/output) a data file");
      MachineFitter fitter;
      fitter.machine = machine;
      fitter.constraints = constraints;
      fitter.constants = machine.funcs;
      fitter.seed = fitter.allConstraints().defaultParams().combine (seed, true);
      if (getenv ("MB_VERBOSE"))
        fitter.onIteration = [] (int it, double ll, const Params&) { cerr << "Baum-Welch iteration #" << it << ": log-likelihood " << ll << endl; };
      params = fitter.fit (data);
      params.writeJson (cout);
      cout << endl;
      if (!(doL || doV || doA || doC)) return EXIT_SUCCESS;
      eval = evaluate (machine, machine.funcs.combine (params));
    }

    // pairs the machine cannot tokenise report -Infinity under -L/-V/-A (boss.cpp:798,826) ...
    SeqPairList ok;
    vector<int> okIndex;
    int n = 0;
    for (const auto& sp: data.seqPairs) { if (eval.canTokenize (sp)) { ok.seqPairs.push_back (sp); okIndex.push_back (n); } ++n; }
    const double ninf = -numeric_limits<double>::infinity();

    auto printScores = [&] (const vector<double>& okScores) {
      vector<double> all (data.seqPairs.size(), ninf);
      for (size_t k = 0; k < okScores.size(); ++k) all[okIndex[k]] = okScores[k];
      cout << "[";
      size_t k = 0;
      for (const auto& sp: data.seqPairs) {
        cout << (k ? ",\n " : "") << "[\"" << Json::escape (sp.input.name) << "\",\"" << Json::escape (sp.output.name) << "\"," << toInfinitySafeString (all[k]) << "]";
        ++k;
      }
      cout << "]\n";
    };

    if (useApi) {      // src/api.h:21-30, called the way a program written against the reference calls them
      if (!symbolic) throw runtime_error ("--api needs a symbolic --machine");
      const Params all = machine.funcs.combine (params);
      if (doL) { vector<double> v; for (const auto& sp: ok.seqPairs) v.push_back (forwardLogLike (machine, all, sp)); printScores (v); }
      if (doV) { vector<double> v; for (const auto& sp: ok.seqPairs) v.push_back (viterbiLogLike (machine, all, sp)); printScores (v); }
      if (doC) {
        const MachineCounts counts = forwardBackwardCounts (machine, all, data);
        cout << "{";
        size_t np = 0;
        for (const auto& nc: paramCounts (counts, machine, params)) cout << (np++ ? "," : "") << "\"" << Json::escape (nc.first) << "\":" << nc.second;
        cout << "}" << endl;
      }
      if (doA) {
        SeqPairList results;
        for (const auto& sp: ok.seqPairs)
          if (viterbiLogLike (machine, all, sp) > ninf) results.seqPairs.push_back (SeqPair::seqPairFromPath (viterbiAlign (machine, all, sp), eval, sp.input.name.c_str(), sp.output.name.c_str()));
        results.writeJson (cout);
        cout << endl;
      }
      return EXIT_SUCCESS;
    }
    if (doL) printScores (forwardLogLikes (eval, ok));
    if (doC) {
      // ... but -C does not test canTokenize (boss.cpp:811-816): an unknown symbol throws
      auto writeCounts = [&] (const MachineCounts& counts) {
        if (symbolic) {   // MachineCounts::writeParamCountsJson (counts.cpp:80-87)
          cout << "{";
          size_t np = 0;
          for (const auto& nc: paramCounts (counts, machine, params)) cout << (np++ ? "," : "") << "\"" << Json::escape (nc.first) << "\":" << nc.second;
          cout << "}";
        } else {
          std::ostringstream os;
          counts.writeJson (os);
          string js = os.str();
          while (js.size() && js.back() == '\n') js.pop_back();
          cout << js;
        }
      };
      if (perPair) {
        cout << "[";
        size_t k = 0;
        for (const auto& counts: pairCounts (eval, data)) { cout << (k++ ? ",\n " : ""); writeCounts (counts); }
        cout << "]" << endl;
      } else {
        writeCounts (MachineCounts (eval, data));
        cout << endl;
      }
    }
    if (postTransTop) {   // BackwardMatrix::postTransQueue (backward.cpp:52-56) and traceFrom (backward.cpp:98-108), per pair
      cout << "[";
      size_t k = 0;
      cout.precision (17);
      for (const auto& sp: data.seqPairs) {
        cout << (k++ ? ",\n " : "") << "{";
        if (eval.canTokenize (sp)) {
          const ForwardMatrix f (eval, sp);
          if (f.logLike() > ninf) {
            const BackwardMatrix b (eval, sp);
            BackwardMatrix::PostTransQueue q = b.postTransQueue (f);
            cout << "\"postTransCount\":" << q.size() << ",\"postTrans\":[";
            const BackwardMatrix::PostTrans first = q.top();
            for (int n = 0; n < postTransTop && !q.empty(); ++n) {
              const BackwardMatrix::PostTrans pt = q.top();
              q.pop();
              cout << (n ? "," : "") << "[" << pt.inPos << "," << pt.outPos << "," << (eval.state[pt.src].transOffset + pt.transIndex) << "," << pt.weight << "]";
            }
            const MachineTransition mt = eval.transition ((int32_t) (eval.state[first.src].transOffset + first.transIndex));
            cout << "],\"traceFrom\":[";
            size_t n = 0;
            b.traceFrom (f, first.inPos - (mt.inputEmpty() ? 0 : 1), first.outPos - (mt.outputEmpty() ? 0 : 1), first.src, first.transIndex,
                         [&] (long, long, StateIndex src, size_t ti) { cout << (n++ ? "," : "") << (eval.state[src].transOffset + ti); return false; });
            cout << "]";
          }
        }
        cout << "}";
      }
      cout << "]\n";
      cout.precision (6);
    }
    if (doSample) {   // ForwardMatrix::samplePath (forward.cpp:17-19), pair k drawn with mt19937 (seed + k): [[transition ids], ...]
      cout << "[";
      size_t k = 0;
      for (const auto& sp: data.seqPairs) {
        cout << (k ? ",\n " : "") << "[";
        if (eval.canTokenize (sp)) {
          const ForwardMatrix f (eval, sp);
          if (f.logLike() > ninf) {
            std::mt19937 rng ((unsigned) (sampleSeed + (long long) k));
            size_t n = 0;
            for (const auto& t: f.samplePath (rng).trans) cout << (n++ ? "," : "") << t.id;
          }
        }
        cout << "]";
        ++k;
      }
      cout << "]\n";
    }
    if (posteriorN) {   // the whole list in one device call; pairs that cannot be tokenised print []
      vector<double> ll;
      const vector<vector<MachinePath> > paths = posteriorPaths (eval, ok, posteriorN, (uint64_t) posteriorSeed, &ll);
      vector<int> okAt (data.seqPairs.size(), -1);
      for (size_t q = 0; q < okIndex.size(); ++q) okAt[okIndex[q]] = (int) q;
      cout << "[";
      for (size_t k = 0; k < data.seqPairs.size(); ++k) {
        cout << (k ? ",\n " : "") << "[";
        if (okAt[k] >= 0 && ll[okAt[k]] > ninf) {
          size_t j = 0;
          for (const auto& p: paths[okAt[k]]) {
            cout << (j++ ? "," : "") << "[";
            size_t n = 0;
            for (const auto& t: p.trans) cout << (n++ ? "," : "") << t.id;
            cout << "]";
          }
        }
        cout << "]";
      }
      cout << "]\n";
    }
    if (doMea || doViterbiPost) {   // the whole list in one device call; pairs that cannot be tokenised have no path
      vector<int> okAt (data.seqPairs.size(), -1);
      for (size_t q = 0; q < okIndex.size(); ++q) okAt[okIndex[q]] = (int) q;
      cout.precision (17);
      auto printList = [&] (const vector<double>& v) { cout << "["; size_t n = 0; for (double p: v) cout << (n++ ? "," : "") << p; cout << "]"; };
      if (doMea) {
        vector<double> gain;
        vector<vector<double> > post;
        const vector<MachinePath> paths = meaPaths (eval, ok, &gain, &post);
        cout << "[";
        size_t k = 0;
        for (const auto& sp: data.seqPairs) {
          const int q = okAt[k];
          const bool has = q >= 0 && gain[q] > ninf;
          cout << (k++ ? ",\n " : "") << "{\"input\":\"" << Json::escape (sp.input.name) << "\",\"output\":\"" << Json::escape (sp.output.name)
               << "\",\"gain\":";
          if (has) cout << gain[q]; else cout << toInfinitySafeString (ninf);
          cout << ",\"path\":[";
          size_t n = 0;
          if (has) for (const auto& t: paths[q].trans) cout << (n++ ? "," : "") << t.id;
          cout << "],\"postProb\":";
          printList (has ? post[q] : vector<double>());
          cout << "}";
        }
        cout << "]\n";
      }
      if (doViterbiPost) {
        vector<MachinePath> vpaths;
        const vector<double> sc = viterbiLogLikes (eval, ok, &vpaths);
        SeqPairList withPath;      // pairs without a Viterbi path have no steps to score
        vector<MachinePath> found;
        vector<int> foundAt (ok.seqPairs.size(), -1);
        size_t q = 0;
        for (const auto& sp: ok.seqPairs) {
          if (sc[q] > ninf) { foundAt[q] = (int) found.size(); withPath.seqPairs.push_back (sp); found.push_back (vpaths[q]); }
          ++q;
        }
        const vector<vector<double> > post = pathPosteriors (eval, withPath, found);
        cout << "[";
        for (size_t k = 0; k < data.seqPairs.size(); ++k) {
          const int f = okAt[k] >= 0 ? foundAt[okAt[k]] : -1;
          cout << (k ? ",\n " : "");
          printList (f >= 0 ? post[f] : vector<double>());
        }
        cout << "]\n";
      }
      cout.precision (6);
    }
    if (doA || doV) {
      vector<MachinePath> paths;
      const vector<double> sc = viterbiLogLikes (eval, ok, doA ? &paths : nullptr);
      if (doV) printScores (sc);
      if (doA) {
        SeqPairList results;
        size_t k = 0;
        for (const auto& sp: ok.seqPairs) {
          if (sc[k] > ninf) results.seqPairs.push_back (SeqPair::seqPairFromPath (paths[k], eval, sp.input.name.c_str(), sp.output.name.c_str()));
          ++k;
        }
        results.writeJson (cout);
        cout << endl;
      }
    }
  } catch (const std::exception& e) {
    cerr << e.what() << endl;
    return EXIT_FAILURE;   // boss.cpp:923-926
  }
  return EXIT_SUCCESS;
}
