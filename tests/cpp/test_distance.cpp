// Distance methods through the shim (Distance/ of the reference): tests/test_distances.py and tools/bench_distances.py drive it.
//   test_distance bionj <matrix file> [rooted] [positive]   BioNJ on a matrix ("n", then n lines "name d_0 ... d_n-1"); prints
//                                                            the tree in Newick with 17 significant digits and the host time
//   test_distance estimate                                   DistanceEstimation on test_likelihood.cpp's four sequences (T92
//                                                            kappa = 3, theta = .5, Gamma4 alpha = 1), BioNJ on it, the tree
//                                                            evaluated by DRHomogeneousTreeLikelihood and PseudoNewtonOptimizer
#include <chrono>
#include <cstdlib>
#include <cstdio>
#include <fstream>
#include <iostream>
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
  if (n->hasDistanceToFather()) {
    char b[64];
    snprintf(b, sizeof(b), ":%.17g", n->getDistanceToFather());
    out += b;
  }
}

static string toNewick(const Tree& t) {
  string s;
  newick(t.getRootNode(), s);
  return s + ";";
}

int main(int argc, char** argv) {
  try {
    const string mode = argc > 1 ? argv[1] : "";
    if (mode == "bionj" && argc > 2) {
      ifstream in(argv[2]);
      size_t n = 0;
      in >> n;
      vector<string> names(n);
      vector<double> d(n * n);
      for (size_t i = 0; i < n; ++i) {
        in >> names[i];
        for (size_t j = 0; j < n; ++j) {   // strtod: "nan" and "inf" are valid entries
          string tok;
          in >> tok;
          d[i * n + j] = strtod(tok.c_str(), nullptr);
        }
      }
      if (!in) throw Exception("bad matrix file");
      DistanceMatrix m(names);
      for (size_t i = 0; i < n; ++i)
        for (size_t j = 0; j < n; ++j) m(i, j) = d[i * n + j];
      const bool rooted = argc > 3 && string(argv[3]) == "1", positive = argc > 4 && string(argv[4]) == "1";
      const auto t0 = chrono::steady_clock::now();
      BioNJ nj(m, rooted, positive, false);
      const double ms = 1e3 * chrono::duration<double>(chrono::steady_clock::now() - t0).count();
      unique_ptr<Tree> tree(nj.getTree());
      printf("TREE %s\nBIONJ_MS %.3f\n", toNewick(*tree).c_str(), ms);
      return 0;
    }
    if (mode == "estimate") {
      const DNA dna;
      VectorSiteContainer s(&dna);
      s.addSequence(BasicSequence("A", "AAATGGCTGTGCACGTC", &dna));
      s.addSequence(BasicSequence("B", "GACTGGATCTGCACGTC", &dna));
      s.addSequence(BasicSequence("C", "CTCTGGATGTGCACGTG", &dna));
      s.addSequence(BasicSequence("D", "AAATGGCGGTGCGCCTA", &dna));
      T92 model(&dna, 3., .5);
      GammaDiscreteRateDistribution rdist(4, 1.0);
      DistanceEstimation de(&model, &rdist, &s, 0, true);
      unique_ptr<DistanceMatrix> dm(de.getMatrix());
      for (size_t i = 0; i < dm->size(); ++i) {
        printf("DIST %s", dm->getName(i).c_str());
        for (size_t j = 0; j < dm->size(); ++j) printf(" %.17g", (*dm)(i, j));
        printf("\n");
      }
      BioNJ nj(*dm, false, true, false);
      unique_ptr<Tree> tree(nj.getTree());
      printf("TREE %s\n", toNewick(*tree).c_str());
      DRHomogeneousTreeLikelihood tl(*tree, s, &model, &rdist);
      tl.initialize();
      printf("START %.15f\n", tl.getValue());
      PseudoNewtonOptimizer opt(&tl);
      opt.setTolerance(1e-6);
      opt.init(tl.getBranchLengthsParameters());
      int steps = 0;
      double prev;
      do {
        prev = opt.getFunctionValue();
        opt.step();
        ++steps;
      } while (fabs(opt.getFunctionValue() - prev) >= 1e-6 && steps < 200);
      printf("FINAL %.15f\n", opt.getFunctionValue());
      return 0;
    }
    cerr << "usage: test_distance bionj <file> [rooted] [positive] | estimate" << endl;
    return 2;
  } catch (std::exception& e) {
    cerr << e.what() << endl;
    return 1;
  }
}
