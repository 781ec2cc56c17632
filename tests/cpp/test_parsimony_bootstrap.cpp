// The parsimony bootstrap through the shim (bppPars): tests/test_parsimony_bootstrap.py drives it.
//   test_parsimony_bootstrap lockstep <alignment> <newick> <R> <seed>
//       DRTreeParsimonyBootstrap from the tree <newick> (DNA alignment, one "name sequence" line per taxon), then the lockstep
//       OptimizationTools::optimizeTreeNNI.  Prints, per replicate r, its scores (SCORES r ...), its final tree (TREE r ...),
//       the sum of its weights (WEIGHT_SUM r), the number of batched calls (CALLS), and the scores of replicate 3 searched
//       alone (ALONE 3 ...).
//   test_parsimony_bootstrap support <alignment> <R> <seed>
//       DistanceEstimation (JC69) -> BioNJ -> DRTreeParsimonyScore -> optimizeTreeNNI gives the main tree; then
//       DRTreeParsimonyBootstrap (R replicates from the main tree) -> lockstep search -> TreeTools::computeBootstrapValues on
//       the main tree.  Prints the BIONJ start (START), the main tree (MAIN) and, per internal branch of the main tree, its
//       support and the leaves on the side of its split without the first leaf (SUPPORT value name,name,...).
//   test_parsimony_bootstrap values <main newick> <format> <replicate newick>...
//       TreeTools::computeBootstrapValues on hand-built trees (no device): per internal branch of the main tree, SUPPORT as
//       above, or THROWS and the message.
#include <cstdio>
#include <fstream>
#include <iostream>
#include <memory>
#include <set>

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

static string newick(const Tree& t) {
  string s;
  newick(t.getRootNode(), s);
  return s + ";";
}

static void leavesBelow(const Node* n, set<string>& out) {
  if (n->isLeaf()) out.insert(n->getName());
  for (size_t i = 0; i < n->getNumberOfSons(); ++i) leavesBelow(n->getSon(i), out);
}

// SUPPORT value and the leaves on the side of the branch's split without the first leaf, per internal non-root node
static void printSupports(const Tree& main) {
  const vector<string> all = main.getLeavesNames();
  const string first = *min_element(all.begin(), all.end());
  for (const Node* n : main.getNodes()) {
    if (n->isLeaf() || !n->hasFather()) continue;
    set<string> side;
    leavesBelow(n, side);
    if (side.count(first)) {
      set<string> other(all.begin(), all.end());
      for (const string& x : side) other.erase(x);
      side.swap(other);
    }
    printf("SUPPORT %.2f ", n->getBranchProperty(TreeTools::BOOTSTRAP));
    bool comma = false;
    for (const string& x : side) { printf("%s%s", comma ? "," : "", x.c_str()); comma = true; }
    printf("\n");
  }
}

int main(int argc, char** argv) {
  try {
    const string mode = argc > 1 ? argv[1] : "";
    const DNA dna;
    VectorSiteContainer s(&dna);
    if (argc > 2) {
      ifstream in(argv[2]);
      string name, seq;
      while (in >> name >> seq) s.addSequence(BasicSequence(name, seq, &dna));
    }
    if (mode == "values" && argc > 4) {
      unique_ptr<Tree> main(TreeTemplateTools::parenthesisToTree(argv[2]));
      vector<unique_ptr<Tree> > reps;
      vector<Tree*> ptrs;
      for (int i = 4; i < argc; ++i) {
        reps.emplace_back(TreeTemplateTools::parenthesisToTree(argv[i]));
        ptrs.push_back(reps.back().get());
      }
      try {
        TreeTools::computeBootstrapValues(*main, ptrs, false, atoi(argv[3]));
      } catch (Exception& e) {
        printf("THROWS %s\n", e.what());
        return 0;
      }
      printSupports(*main);
      return 0;
    }
    if (mode == "lockstep" && argc > 5) {
      unique_ptr<Tree> start(TreeTemplateTools::parenthesisToTree(argv[3]));
      DRTreeParsimonyBootstrap tb(*start, s, (unsigned)atoi(argv[4]), strtoull(argv[5], nullptr, 10));
      vector<vector<int64_t> > scores;
      OptimizationTools::optimizeTreeNNI(&tb, 0, &scores);
      for (size_t r = 0; r < tb.getNumberOfReplicates(); ++r) {
        printf("SCORES %zu", r);
        for (int64_t x : scores[r]) printf(" %lld", (long long)x);
        printf("\nTREE %zu %s\n", r, newick(tb.getTree(r)).c_str());
        if (tb.getScore(r) != scores[r].back()) throw Exception("getScore differs from the search's last score");
        long long sum = 0;
        for (unsigned w : tb.getWeights(r)) sum += w;
        printf("WEIGHT_SUM %zu %lld\n", r, sum);
      }
      printf("CALLS %zu\n", tb.getNumberOfCalls());
      // replicate 3 searched alone (every call a batch of one) on a second bootstrap of the same data and seed
      DRTreeParsimonyBootstrap alone(*start, s, (unsigned)atoi(argv[4]), strtoull(argv[5], nullptr, 10));
      vector<vector<int64_t> > sc;
      const vector<size_t> only(1, 3);
      OptimizationTools::optimizeTreeNNI(&alone, 0, &sc, &only);
      printf("ALONE 3");
      for (int64_t x : sc[3]) printf(" %lld", (long long)x);
      printf("\n");
      return 0;
    }
    if (mode == "support" && argc > 4) {
      JCnuc model(&dna);
      GammaDiscreteRateDistribution rdist(1, 1.0);
      DistanceEstimation de(&model, &rdist, &s, 0, true);
      unique_ptr<DistanceMatrix> dm(de.getMatrix());
      BioNJ nj(*dm, false, true, false);
      unique_ptr<Tree> tree(nj.getTree());
      DRTreeParsimonyScore tp(*tree, s, false);
      printf("START %s\n", newick(tp.getTree()).c_str());
      OptimizationTools::optimizeTreeNNI(&tp, 0);
      Tree main(tp.getTree());
      printf("MAIN %s\n", newick(main).c_str());
      DRTreeParsimonyBootstrap tb(main, s, (unsigned)atoi(argv[3]), strtoull(argv[4], nullptr, 10));
      OptimizationTools::optimizeTreeNNI(&tb, 0);
      TreeTools::computeBootstrapValues(main, tb.getTrees(), false, 2);
      printSupports(main);
      return 0;
    }
    cerr << "usage: test_parsimony_bootstrap lockstep <alignment> <newick> <R> <seed> | support <alignment> <R> <seed> | values "
            "<newick> <format> <newick>..." << endl;
    return 2;
  } catch (std::exception& e) {
    cerr << e.what() << endl;
    return 1;
  }
}
