// The parsimony bootstrap through the shim, timed (tools/bench_parsimony_bootstrap.py builds and drives it):
//   bench_parsimony_bootstrap <alignment> <R> <seed> <n_single>
// DNA alignment (one "name sequence" line per taxon) -> DistanceEstimation (JC69) -> BioNJ -> DRTreeParsimonyBootstrap (R
// replicates from the BIONJ tree).  First the first n_single replicates are searched one after another, each alone (every call
// a batch of one); then every tree goes back to the start and all R are searched in lockstep (OptimizationTools::
// optimizeTreeNNI).  Same driver, handle, patterns and kernels, so that the difference is what batching the replicates changes.  Prints the
// start tree (START) and one JSON line (RESULT) with the pattern count, the sampler's device time, both searches' wall and
// device time and calls, and every replicate's scores; exits 1 if a replicate's scores differ between the two.
#include <chrono>
#include <cstdio>
#include <fstream>
#include <memory>
#include <string>

#include "../bpp_phyl_b200/host/bppgpu_shim.hpp"

using namespace bppshim;
using namespace std;

static void newick(const Node* n, string& out) {
  if (!n->isLeaf()) {
    out += "(";
    for (size_t i = 0; i < n->getNumberOfSons(); ++i) {
      if (i) out += ",";
      newick(n->getSon(i), out);
    }
    out += ")";
  } else {
    out += n->getName();
  }
}

static double since(chrono::steady_clock::time_point t0) { return chrono::duration<double>(chrono::steady_clock::now() - t0).count(); }

int main(int argc, char** argv) {
  if (argc < 5) {
    fprintf(stderr, "usage: bench_parsimony_bootstrap <alignment> <R> <seed> <n_single>\n");
    return 2;
  }
  try {
    const DNA dna;
    VectorSiteContainer s(&dna);
    {
      ifstream in(argv[1]);
      string name, seq;
      while (in >> name >> seq) s.addSequence(BasicSequence(name, seq, &dna));
    }
    auto t0 = chrono::steady_clock::now();
    JCnuc model(&dna);
    GammaDiscreteRateDistribution rdist(1, 1.0);
    DistanceEstimation de(&model, &rdist, &s, 0, true);
    unique_ptr<DistanceMatrix> dm(de.getMatrix());
    BioNJ nj(*dm, false, true, false);
    unique_ptr<Tree> tree(nj.getTree());
    const double bionj_s = since(t0);
    t0 = chrono::steady_clock::now();
    DRTreeParsimonyBootstrap tb(*tree, s, (unsigned)atoi(argv[2]), strtoull(argv[3], nullptr, 10), false);
    const double create_s = since(t0);
    string start;
    newick(tb.getTree(0).getRootNode(), start);
    printf("START %s;\n", start.c_str());
    // the first n_single replicates searched alone, one after another, then every tree back at the start and all in lockstep
    const size_t n_single = min((size_t)atoi(argv[4]), tb.getNumberOfReplicates());
    const Tree start_tree(tb.getTree(0));
    vector<vector<int64_t> > single(n_single);
    t0 = chrono::steady_clock::now();
    for (size_t r = 0; r < n_single; ++r) {
      vector<vector<int64_t> > sc;
      const vector<size_t> only(1, r);
      OptimizationTools::optimizeTreeNNI(&tb, 0, &sc, &only);
      single[r] = sc[r];
    }
    const double single_s = since(t0);
    const double single_ms = tb.getDeviceMs();
    const size_t single_calls = tb.getNumberOfCalls();
    for (size_t r = 0; r < n_single; ++r) tb.setTree(r, start_tree);
    vector<vector<int64_t> > scores;
    t0 = chrono::steady_clock::now();
    OptimizationTools::optimizeTreeNNI(&tb, 0, &scores);
    const double search_s = since(t0);
    size_t rounds = 0;
    for (const auto& sc : scores) rounds = max(rounds, sc.size());   // the last round retires every replicate still active
    for (size_t r = 0; r < n_single; ++r)
      if (single[r] != scores[r]) throw Exception("replicate " + to_string(r) + ": searched alone, its scores differ from the lockstep's");
    printf("RESULT {\"patterns\": %zu, \"bionj_s\": %.4f, \"create_and_sample_s\": %.4f, \"sampler_device_ms\": %.4f, "
           "\"search_wall_s\": %.4f, \"search_device_ms\": %.3f, \"batched_calls\": %zu, \"rounds\": %zu, "
           "\"single\": {\"replicates\": %zu, \"search_wall_s\": %.4f, \"search_device_ms\": %.3f, \"calls\": %zu, "
           "\"scores_equal_lockstep\": true}, \"scores\": [",
           tb.getNumberOfPatterns(), bionj_s, create_s, tb.getSamplerMs(), search_s, tb.getDeviceMs() - single_ms,
           tb.getNumberOfCalls() - single_calls, rounds, n_single, single_s, single_ms, single_calls);
    for (size_t r = 0; r < scores.size(); ++r) {
      printf("%s[", r ? ", " : "");
      for (size_t i = 0; i < scores[r].size(); ++i) printf("%s%lld", i ? ", " : "", (long long)scores[r][i]);
      printf("]");
    }
    printf("]}\n");
    return 0;
  } catch (std::exception& e) {
    fprintf(stderr, "%s\n", e.what());
    return 1;
  }
}
