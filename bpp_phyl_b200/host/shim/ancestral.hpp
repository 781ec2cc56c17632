// bppgpu shim (see ../bppgpu_shim.hpp): ancestral reconstruction classes (joint ML, marginal, marginal non-reversible)
#pragma once
#include "likelihood.hpp"

namespace bppshim {

// ---- joint ML ancestral reconstruction (fork: Likelihood/MLAncestralStateReconstruction.{h,cpp}, Pupko et al. 2000) -------------
// The reference constructor takes the likelihood, its model, the root frequencies and its pxy_ map
// (MLAncestralStateReconstruction.h:88-103); here the device already holds that likelihood's tables, so `model` and `Pijt` are
// accepted for source compatibility only and `rootFrequencies` must be the likelihood's own.
class MLAncestralStateReconstruction {
 public:
  MLAncestralStateReconstruction(const AbstractHomogeneousTreeLikelihood* drl, const SubstitutionModel* model, const std::vector<double>& rootFrequencies,
                                 const void* Pijt = nullptr)
      : likelihood_(drl) {
    (void)model; (void)Pijt;
    const Vdouble& rf = drl->getRootFrequencies();
    if (rootFrequencies.size() != rf.size()) throw Exception("MLAncestralStateReconstruction: wrong number of root frequencies");
    for (size_t x = 0; x < rf.size(); ++x)
      if (std::fabs(rf[x] - rootFrequencies[x]) > 1e-12)
        throw Exception("MLAncestralStateReconstruction: root frequencies other than the likelihood's own are not supported");
  }
  void computeJointLikelihood() { likelihood_->getJointMLAncestralStates(states_, &bestLogLik_); computed_ = true; }
  // node id -> best state per distinct site (getAllAncestralStates, .cpp:136-141)
  std::map<int, std::vector<size_t> > getAllAncestralStates() const {
    if (!computed_) throw Exception("MLAncestralStateReconstruction: computeJointLikelihood() was not called");
    std::map<int, std::vector<size_t> > ancestors;
    const std::vector<int> ids = likelihood_->getNodesId();
    for (size_t n = 0; n < ids.size(); ++n) ancestors[ids[n]] = states_[n];
    return ancestors;
  }
  const Vdouble& getBestJointLogLikelihoodPerSite() const { return bestLogLik_; }   // not in the reference: log max joint likelihood

 private:
  const AbstractHomogeneousTreeLikelihood* likelihood_;   // not owned
  std::vector<std::vector<size_t> > states_;
  Vdouble bestLogLik_;
  bool computed_ = false;
};

// ---- marginal ancestral reconstruction (Likelihood/MarginalAncestralStateReconstruction.{h,cpp}) ---------------------------------
// getAncestralStatesForNode (.cpp:47-102): probs[i][x] = sum_c computeLikelihoodAtNode[i][c][x] r_c / l_i at an internal node --
// the device's marginal posterior table -- and the best (or a sampled) state per distinct site; a leaf gets the first maximum
// of its leaf likelihoods with probability one (:53-65).
class MarginalAncestralStateReconstruction {
 public:
  explicit MarginalAncestralStateReconstruction(const AbstractHomogeneousTreeLikelihood* drl)
      : likelihood_(drl), nbSites_(drl->getNumberOfSites()), nbDistinctSites_(drl->getNumberOfDistinctSites()),
        nbStates_(drl->getNumberOfStates()) {}
  std::vector<size_t> getAncestralStatesForNode(int nodeId, VVdouble& probs, bool sample = false) const {
    std::vector<size_t> ancestors(nbDistinctSites_, 0);
    if (likelihood_->getTree().getNode(nodeId)->isLeaf()) {
      const VVVdouble leaf = likelihood_->getPosteriorProbabilitiesForEachStateForEachRate(nodeId);   // leaf likelihoods x p_c / sum
      probs.assign(nbDistinctSites_, Vdouble(nbStates_, 0.0));
      for (size_t i = 0; i < nbDistinctSites_; ++i) {
        size_t j = 0;
        for (size_t x = 1; x < nbStates_; ++x) if (leaf[i][0][x] > leaf[i][0][j]) j = x;
        ancestors[i] = j;
        probs[i][j] = 1.0;
      }
      return ancestors;
    }
    likelihood_->getMarginalPosteriors(nodeId, probs, nullptr);
    for (size_t i = 0; i < nbDistinctSites_; ++i) {
      if (sample) {
        const double r = std::generate_canonical<double, 53>(rng_);
        double cum = 0;
        for (size_t j = 0; j < nbStates_; ++j) {
          cum += probs[i][j];
          if (r <= cum) { ancestors[i] = j; break; }
        }
      } else {
        ancestors[i] = (size_t)(std::max_element(probs[i].begin(), probs[i].end()) - probs[i].begin());
      }
    }
    return ancestors;
  }
  std::vector<size_t> getAncestralStatesForNode(int nodeId) const {
    VVdouble probs;
    return getAncestralStatesForNode(nodeId, probs, false);
  }
  // one state per distinct site for every node of the tree (recursiveMarginalAncestralStates)
  std::map<int, std::vector<size_t> > getAllAncestralStates() const {
    std::map<int, std::vector<size_t> > ancestors;
    for (int id : likelihood_->getNodesId()) ancestors[id] = getAncestralStatesForNode(id);
    return ancestors;
  }
  // the node's states site by site (getAncestralSequenceForNode without the Sequence wrapper): site -> pattern via getSiteIndex
  std::vector<size_t> getAncestralStatesPerSiteForNode(int nodeId, VVdouble* probs = nullptr, bool sample = false) const {
    VVdouble patterned;
    const std::vector<size_t> states = getAncestralStatesForNode(nodeId, patterned, sample);
    std::vector<size_t> all(nbSites_);
    if (probs) probs->resize(nbSites_);
    for (size_t i = 0; i < nbSites_; ++i) {
      all[i] = states[likelihood_->getSiteIndex(i)];
      if (probs) (*probs)[i] = patterned[likelihood_->getSiteIndex(i)];
    }
    return all;
  }

 private:
  const AbstractHomogeneousTreeLikelihood* likelihood_;   // not owned
  size_t nbSites_, nbDistinctSites_, nbStates_;
  mutable std::mt19937_64 rng_{20260101};
};

// ---- marginal ancestral reconstruction for non-reversible models (fork) --------------------------------------------------------
// Likelihood/MarginalNonRevAncestralStateReconstruction.h:66-207.  The reference re-runs the prefix pass once per root state
// (DRNonHomogeneousTreeLikelihood::computeLikelihoodPrefixConditionalOnRoot, .cpp:1026-1162: S full passes, S^2 work per
// (node, site, state) on top); the device computes the same tables in one pass per node from the resident arrays
// (bppgpu_get_marginal_posteriors).  Map keys follow the reference: node id -> distinct-site index -> state vector.
class MarginalNonRevAncestralStateReconstruction {
 public:
  explicit MarginalNonRevAncestralStateReconstruction(AbstractHomogeneousTreeLikelihood* drl)
      : likelihood_(drl), nbSites_(drl->getNumberOfSites()), nbDistinctSites_(drl->getNumberOfDistinctSites()),
        nbClasses_(drl->getNumberOfClasses()), nbStates_(drl->getNumberOfStates()) {}

  void computePosteriorProbabilitiesOfNodesForEachStatePerSite() {
    postProbNode_.reset(new std::map<int, std::map<size_t, std::vector<double> > >);
    jointProbabilities_.reset(new std::map<int, std::map<size_t, VVdouble> >);
    for (int id : likelihood_->getNodesId()) {
      VVdouble post;
      VVVdouble joint;
      likelihood_->getMarginalPosteriors(id, post, &joint);
      for (size_t i = 0; i < nbDistinctSites_; ++i) {
        (*postProbNode_)[id][i] = post[i];
        (*jointProbabilities_)[id][i] = joint[i];   // [nodeState][fatherState]; all zero at the root, like the reference
      }
    }
  }
  std::map<int, std::map<size_t, VVdouble> > getAllJointFatherNodeProbabilities() {
    if (!jointProbabilities_) computePosteriorProbabilitiesOfNodesForEachStatePerSite();
    return *jointProbabilities_;
  }
  std::map<int, std::map<size_t, std::vector<double> > >* getPosteriorProbForAllNodesAndStatesPerSite() {
    if (!postProbNode_) computePosteriorProbabilitiesOfNodesForEachStatePerSite();
    return postProbNode_.get();
  }
  // argmax state per SITE (.cpp:155-167).  The reference indexes the distinct-site tables with the site number, which is
  // only right when every site is its own pattern (ChromEvol: one site); here a site reads its pattern's entry.
  const std::map<int, std::vector<size_t> > getAllAncestralStates() const {
    if (!postProbNode_) throw Exception("MarginalNonRevAncestralStateReconstruction: posterior probabilities not computed");
    std::map<int, std::vector<size_t> > ancestors;
    for (const auto& kv : *postProbNode_) {
      std::vector<size_t>& a = ancestors[kv.first];
      a.reserve(nbSites_);
      for (size_t s = 0; s < nbSites_; ++s) {
        const std::vector<double>& p = kv.second.at(likelihood_->getSiteIndex(s));
        a.push_back((size_t)(std::max_element(p.begin(), p.end()) - p.begin()));   // VectorTools::whichMax: first maximum
      }
    }
    return ancestors;
  }
  // posterior of the root state at distinct site 0 (.cpp:139-153)
  std::vector<double> getRootPosteriorProb() const {
    VVdouble post;
    likelihood_->getMarginalPosteriors(likelihood_->getNodesId().back(), post, nullptr);
    return post.at(0);
  }

 private:
  AbstractHomogeneousTreeLikelihood* likelihood_;   // not owned
  size_t nbSites_, nbDistinctSites_, nbClasses_, nbStates_;
  std::unique_ptr<std::map<int, std::map<size_t, std::vector<double> > > > postProbNode_;
  std::unique_ptr<std::map<int, std::map<size_t, VVdouble> > > jointProbabilities_;
};

// ---- expected numbers of chromosome-number events per branch (fork) ----------------------------------------------------------
// ChromosomeNumberMng::computeExpectations: ComputeChromosomeTransitionsExp built from the fitted likelihood and its model.
// Stochastic mapping (Mayrose et al. 2010) with the estimator of bppgpu_expected_events (DESIGN §7b): numOfSimulations paths per
// start state over the branch lengths, combined with the (node, father) joint posteriors of
// MarginalNonRevAncestralStateReconstruction, which stay on the device.  The reference's random stream is not reproduced; a
// run depends only on the seed.  runSimulations does the device call (simulation and combination together);
// computeExpectationPerType forms the tree totals.
class ComputeChromosomeTransitionsExp {
 public:
  typedef ChromosomeSubstitutionModel::typeOfTransition typeOfTransition;
  ComputeChromosomeTransitionsExp(AbstractHomogeneousTreeLikelihood* tl, const ChromosomeSubstitutionModel* model)
      : likelihood_(tl), model_(model) {}

  void runSimulations(int numOfSimulations, uint64_t seed = 0) {
    if (numOfSimulations < 1) throw Exception("ComputeChromosomeTransitionsExp::runSimulations: need at least one simulation");
    likelihood_->getExpectedEvents(ChromosomeSubstitutionModel::NUMTYPES, model_->getTypeRates(), numOfSimulations, seed, expected_,
                                   unreached_);
    totals_.clear();
  }
  void computeExpectationPerType() {
    if (expected_.empty()) throw Exception("ComputeChromosomeTransitionsExp: runSimulations first");
    totals_.assign(ChromosomeSubstitutionModel::NUMTYPES, 0.0);
    for (size_t n = 0; n < unreached_.size(); ++n)
      for (int t = 0; t < ChromosomeSubstitutionModel::NUMTYPES; ++t) totals_[(size_t)t] += expected_[n * ChromosomeSubstitutionModel::NUMTYPES + (size_t)t];
  }
  // expected number of class-`type` events on the branch above nodeId (0 at the root)
  double getExpectation(int nodeId, int type) const {
    require();
    return expected_.at((size_t)nodeId * ChromosomeSubstitutionModel::NUMTYPES + (size_t)type);
  }
  // the tree's expected number of class-`type` events (computeExpectationPerType)
  double getTotalExpectation(int type) const {
    if (totals_.empty()) throw Exception("ComputeChromosomeTransitionsExp: computeExpectationPerType first");
    return totals_.at((size_t)type);
  }
  // posterior mass of the branch above nodeId whose (father, node) states no path reached: it contributes nothing to the
  // expectations, so a large value asks for more simulations
  double getUnreachedMass(int nodeId) const {
    require();
    return unreached_.at((size_t)nodeId);
  }

 private:
  void require() const { if (expected_.empty()) throw Exception("ComputeChromosomeTransitionsExp: runSimulations first"); }
  AbstractHomogeneousTreeLikelihood* likelihood_;   // not owned
  const ChromosomeSubstitutionModel* model_;         // not owned
  Vdouble expected_, unreached_, totals_;
};

// Likelihood/RNonHomogeneousMixedTreeLikelihood.{h,cpp}: mixed models on groups of branches.  The reference expands the set into one
// RNonHomogeneousTreeLikelihood per site path ("hyper-node") and adds their site likelihoods with the path probabilities
// (RNonHomogeneousMixedTreeLikelihood.cpp: getLikelihoodForASite = sum_paths p_path L_path); here every path is one point of a
// single device object: K x M model slots (path k, model m), one branch -> slot map per point, one evaluation for all paths.
class RNonHomogeneousMixedTreeLikelihood : public AbstractHomogeneousTreeLikelihood {
 public:
  RNonHomogeneousMixedTreeLikelihood(const Tree& tree, const VectorSiteContainer& data, MixedSubstitutionModelSet* modelSet,
                                     DiscreteDistribution* rDist, bool verbose = true, bool usePatterns = true, int device = 0)
      : AbstractHomogeneousTreeLikelihood(tree, modelSet->getModel(0)->getNModel(0), rDist, false, BPPGPU_FLAG_R_SEMANTICS, device),
        mixedSet_(modelSet) {
    (void)verbose; (void)usePatterns;
    for (size_t i = 0; i + 1 < nodes_.size(); ++i) mixedSet_->getModelIndexForNode(nodes_[i]->getId());   // throws if a branch has no model
    nPoints_ = (int)mixedSet_->getNumberOfPaths();
    nModelSlots_ = nPoints_ * (int)mixedSet_->getNumberOfModels();
    computeDerivatives_ = false;
    setData(data);
  }
  double getValue() const { requireInit(); return mixedMinusLogLik_; }
  double getLogLikelihood() const { return -getValue(); }
  double getLogLikelihoodForASite(size_t site) const { requireInit(); return mixedSiteLnl_[(size_t)siteIndex_[site]]; }
  void computeTreeLikelihood() { fireParameterChanged(); }

 protected:
  // "<Model>.<param>_<m>": parameter of the m-th mixed model of the set (1-based, like SubstitutionModelSet)
  bool applyBranchParameter(const std::string& name, double value) override {
    const size_t u = name.rfind('_');
    if (u == std::string::npos || name.compare(0, 5, "BrLen") == 0) return false;
    char* end = nullptr;
    const long m = std::strtol(name.c_str() + u + 1, &end, 10);
    if (*end != 0 || m < 1 || (size_t)m > mixedSet_->getNumberOfModels()) return false;
    mixedSet_->getModel((size_t)m - 1)->setParameterValue(name.substr(0, u), value);
    return true;
  }
  void uploadModel() override {
    if (!engine_) return;
    const size_t K = mixedSet_->getNumberOfPaths(), M = mixedSet_->getNumberOfModels();
    Vdouble r(rDist_->getNumberOfCategories()), p(r.size());
    for (size_t c = 0; c < r.size(); ++c) { r[c] = rDist_->getCategory(c); p[c] = rDist_->getProbability(c); }
    check(bppgpu_set_rates(engine_, r.data(), p.data()), "setRates");
    for (size_t k = 0; k < K; ++k) {
      for (size_t m = 0; m < M; ++m) {
        bppgpu_model_desc d;
        mixedSet_->getModel(m)->getNModel(k)->fillModelDesc(d);
        check(bppgpu_set_model(engine_, (int32_t)(k * M + m), &d), "setModel");
      }
      std::vector<int32_t> slot(nodes_.size(), 0);
      for (size_t i = 0; i + 1 < nodes_.size(); ++i) slot[i] = (int32_t)(k * M + mixedSet_->getModelIndexForNode(nodes_[i]->getId()));
      check(bppgpu_set_branch_models(engine_, (int32_t)k, slot.data()), "setBranchModels");
      // stationary set (nonhomogeneous.stationarity = yes): the root uses the equilibrium frequencies of the models
      const Vdouble f = mixedSet_->getModel(0)->getNModel(k)->getFrequencies();
      check(bppgpu_set_root_freqs(engine_, (int32_t)k, f.data()), "setRootFreqs");
    }
    rootFreqs_ = mixedSet_->getModel(0)->getNModel(0)->getFrequencies();
  }
  void fireParameterChanged() override {
    uploadModel();
    const size_t K = mixedSet_->getNumberOfPaths(), N = (size_t)nPatterns_;
    Vdouble t(nodes_.size(), 0.0);
    for (size_t i = 0; i < brLen_.size(); ++i) t[i] = brLen_[i];
    for (size_t k = 0; k < K; ++k) check(bppgpu_set_branch_lengths(engine_, (int32_t)k, t.data()), "applyParameters");
    Vdouble lnl(K, 0.0);
    check(bppgpu_eval(engine_, BPPGPU_EVAL_LNL, lnl.data(), nullptr, nullptr), "computeTreeLikelihood");
    numOfLikelihoodCalculations_ += (long)K;
    std::vector<Vdouble> sl(K, Vdouble(N));
    for (size_t k = 0; k < K; ++k) check(bppgpu_get_site_lnl(engine_, (int32_t)k, sl[k].data()), "getLogLikelihoodForEachSite");
    mixedSiteLnl_.assign(N, 0.0);
    for (size_t i = 0; i < N; ++i) {
      double mx = -std::numeric_limits<double>::infinity();
      for (size_t k = 0; k < K; ++k) if (mixedSet_->getPathProbability(k) > 0) mx = std::max(mx, sl[k][i]);
      double sum = 0;
      for (size_t k = 0; k < K; ++k) if (mixedSet_->getPathProbability(k) > 0) sum += mixedSet_->getPathProbability(k) * std::exp(sl[k][i] - mx);
      mixedSiteLnl_[i] = std::isfinite(mx) ? mx + std::log(sum) : mx;
    }
    Vdouble la(siteIndex_.size());   // getLogLikelihood (RHomogeneousTreeLikelihood.cpp:162-176): every site, sorted, summed
    for (size_t j = 0; j < la.size(); ++j) la[j] = mixedSiteLnl_[(size_t)siteIndex_[j]];
    std::sort(la.begin(), la.end());
    double ll = 0;
    for (size_t j = la.size(); j > 0; --j) ll += la[j - 1];
    mixedMinusLogLik_ = -ll;
    minusLogLik_ = mixedMinusLogLik_;
    siteLnl_ = mixedSiteLnl_;
    derivsValid_ = false;
    rootArraysValid_ = false;
  }

 private:
  MixedSubstitutionModelSet* mixedSet_;   // not owned
  Vdouble mixedSiteLnl_;
  double mixedMinusLogLik_ = 0;
};

}  // namespace bppshim
