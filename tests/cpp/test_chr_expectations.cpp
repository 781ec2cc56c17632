// ChromosomeNumberMng::computeExpectations through the shim.
//   test_chr_expectations split   (no device) the class split of ChromosomeSubstitutionModel for several parameter sets, one
//                                 JSON document: tests/test_chr_expectations.py compares it with oracle/ref_mapping.py bit for bit
//   test_chr_expectations         the five-taxon ChromEvol case: DRNonHomogeneousTreeLikelihood -> marginal reconstruction ->
//                                 ComputeChromosomeTransitionsExp (1e5 paths), and the same estimator through the likelihood's
//                                 own bppgpu_expected_events call with the same seed
#include <cmath>
#include <cstdio>
#include <cstring>
#include <iostream>
#include <memory>

#include "../../bpp_phyl_b200/host/bppgpu_shim.hpp"

using namespace bppshim;
using namespace std;

typedef ChromosomeSubstitutionModel CSM;

static void print_split(const char* key, const CSM& m, bool comma) {
  const vector<double> R = m.getTypeRates();
  printf("\"%s\": {\"R\": [", key);
  for (size_t i = 0; i < R.size(); ++i) printf("%s%.17g", i ? ", " : "", R[i]);
  printf("], \"Q\": [");
  const size_t n = m.getNumberOfStates();
  for (size_t i = 0; i < n; ++i)
    for (size_t j = 0; j < n; ++j) printf("%s%.17g", i + j ? ", " : "", m.getGenerator()(i, j));
  printf("]}%s\n", comma ? "," : "");
}

int main(int argc, char** argv) {
  try {
    if (argc > 1 && !strcmp(argv[1], "split")) {
      // the parameter sets of test_chr_expectations.py::SPLIT_CASES, in that order
      ChromosomeAlphabet a30(1, 30), a12(3, 12), a40(1, 40);
      printf("{\n");
      print_split("linear", CSM(&a30, 0.7, 0.4, 0.2, 0.1, 0.03, 0.02, 0.01), true);
      print_split("exp", CSM(&a30, 0.7, 0.4, 0.2, 0.1, 0.03, -0.02, 0.01, (int)CSM::IgnoreParam, CSM::IgnoreParam, 0, CSM::EXP), true);
      print_split("demi_equal_dupl", CSM(&a12, 0.5, 0.3, 0.8, CSM::DemiEqualDupl), true);
      print_split("demi_ignored", CSM(&a12, 0.5, 0.3, 0.8, CSM::IgnoreParam), true);
      print_split("base_number", CSM(&a40, 0.6, 0.5, 0.3, 0.2, CSM::IgnoreParam, CSM::IgnoreParam, CSM::IgnoreParam, 4, 0.35, 13), true);
      print_split("clamped", CSM(&a12, 0.9, 0.2, 1.1, 0.7, CSM::IgnoreParam, CSM::IgnoreParam, CSM::IgnoreParam, 3, 0.25, 20), false);
      printf("}\n");
      return 0;
    }
    ChromosomeAlphabet chr(1, 30);
    unique_ptr<Tree> tree(TreeTemplateTools::parenthesisToTree("(((a:0.3,b:0.2):0.4,c:0.5):0.1,(d:0.3,e:0.6):0.2);"));
    VectorSiteContainer sites(&chr);
    sites.addSequence(BasicSequence("a", "7", &chr));
    sites.addSequence(BasicSequence("b", "8", &chr));
    sites.addSequence(BasicSequence("c", "14", &chr));
    sites.addSequence(BasicSequence("d", "9", &chr));
    sites.addSequence(BasicSequence("e", "X", &chr));
    CSM model(&chr, 0.7, 0.4, 0.2, 0.1, CSM::IgnoreParam, CSM::IgnoreParam, CSM::IgnoreParam, 3, 0.15, 6);
    ConstantRateDistribution cst;
    DRNonHomogeneousTreeLikelihood tl(*tree, sites, true, false, &model, &cst);
    tl.initialize();
    printf("LNL %.17g\n", tl.getLogLikelihood());
    MarginalNonRevAncestralStateReconstruction asr(&tl);
    asr.computePosteriorProbabilitiesOfNodesForEachStatePerSite();
    const int nSims = 100000;
    const uint64_t seed = 0x9E3779B97F4A7C15ull;
    ComputeChromosomeTransitionsExp exp(&tl, &model);
    exp.runSimulations(nSims, seed);
    exp.computeExpectationPerType();
    Vdouble direct, directUnreached;
    tl.getExpectedEvents(CSM::NUMTYPES, model.getTypeRates(), nSims, seed, direct, directUnreached);
    int mismatches = 0;
    for (int id : tl.getNodesId()) {
      for (int t = 0; t < CSM::NUMTYPES; ++t) {
        printf("EXP_%d_%d %.17g\n", id, t, exp.getExpectation(id, t));
        mismatches += exp.getExpectation(id, t) != direct[(size_t)id * CSM::NUMTYPES + t];
      }
      printf("UNREACHED_%d %.17g\n", id, exp.getUnreachedMass(id));
      mismatches += exp.getUnreachedMass(id) != directUnreached[(size_t)id];
    }
    for (int t = 0; t < CSM::NUMTYPES; ++t) printf("TOTAL_%d %.17g\n", t, exp.getTotalExpectation(t));
    printf("ABI_MISMATCHES %d\n", mismatches);
  } catch (std::exception& e) {
    cerr << e.what() << endl;
    return 1;
  }
  return 0;
}
