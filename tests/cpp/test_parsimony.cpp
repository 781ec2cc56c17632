// Parsimony through the shim (Parsimony/ of the reference): tests/test_parsimony.py and tools/bench_parsimony.py drive it.
//   test_parsimony search <alignment> <newick>   DNA alignment (one "name sequence" line per taxon): DistanceEstimation (JC69)
//                                                -> BioNJ -> DRTreeParsimonyScore -> OptimizationTools::optimizeTreeNNI.  Prints
//                                                the start tree (START), the score before and after every round (ROUND), the
//                                                smallest testNNI at the end (MIN_TEST_NNI), the sum of getScoreForEachSite
//                                                (SITE_SUM), the score of <newick> (TRUE) and the search's wall time (SEARCH_MS)
#include <chrono>
#include <cstdio>
#include <fstream>
#include <iostream>
#include <limits>
#include <memory>

#include "../../bpp_phyl_b200/host/bppgpu_shim.hpp"

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

int main(int argc, char** argv) {
  try {
    const string mode = argc > 1 ? argv[1] : "";
    if (mode == "search" && argc > 3) {
      const DNA dna;
      VectorSiteContainer s(&dna);
      ifstream in(argv[2]);
      string name, seq;
      while (in >> name >> seq) s.addSequence(BasicSequence(name, seq, &dna));
      JCnuc model(&dna);
      GammaDiscreteRateDistribution rdist(1, 1.0);
      DistanceEstimation de(&model, &rdist, &s, 0, true);
      unique_ptr<DistanceMatrix> dm(de.getMatrix());
      BioNJ nj(*dm, false, true, false);
      unique_ptr<Tree> tree(nj.getTree());
      DRTreeParsimonyScore tp(*tree, s, false);
      string start;
      newick(tp.getTree().getRootNode(), start);
      printf("START %s;\n", start.c_str());
      vector<int64_t> scores;
      const auto t0 = chrono::steady_clock::now();
      OptimizationTools::optimizeTreeNNI(&tp, 0, &scores);
      const double ms = 1e3 * chrono::duration<double>(chrono::steady_clock::now() - t0).count();
      printf("ROUND");
      for (int64_t x : scores) printf(" %lld", (long long)x);
      printf("\n");
      double best = numeric_limits<double>::infinity();
      for (const Node* v : tp.getTree().getNodes())
        if (v->hasFather() && v->getFather()->hasFather()) best = min(best, tp.testNNI(v->getId()));
      printf("MIN_TEST_NNI %lld\n", (long long)best);
      long long sum = 0;
      for (unsigned x : tp.getScoreForEachSite()) sum += x;
      printf("SITE_SUM %lld\n", sum);
      unique_ptr<Tree> truth(TreeTemplateTools::parenthesisToTree(argv[3]));
      DRTreeParsimonyScore tt(*truth, s, false);
      printf("TRUE %lld\nSEARCH_MS %.3f\n", (long long)tt.getScore(), ms);
      return 0;
    }
    cerr << "usage: test_parsimony search <alignment> <newick>" << endl;
    return 2;
  } catch (std::exception& e) {
    cerr << e.what() << endl;
    return 1;
  }
}
