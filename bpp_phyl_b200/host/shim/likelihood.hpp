// bppgpu shim (see ../bppgpu_shim.hpp): SitePatterns and the tree-likelihood classes (R / DR / NH / clock / point batch / mixtures)
#pragma once
#include "models.hpp"

namespace bppshim {

// ---- site patterns (SitePatterns.cpp:52-106 through the C ABI) -----------------------------------------------------------------
class SitePatterns {
 public:
  // sequences are taken in the order of `names` (PatternTools::getSequenceSubset re-orders to the tree's leaves)
  SitePatterns(const VectorSiteContainer& sites, const std::vector<std::string>& names) {
    const size_t n = sites.getNumberOfSites(), nt = names.size();
    std::vector<const BasicSequence*> seqs;
    for (const std::string& nm : names) seqs.push_back(&sites.getSequence(nm));
    size_t w = 1;
    for (const BasicSequence* s : seqs)
      for (size_t i = 0; i < n; ++i) w = std::max(w, (*s)[i].size());
    std::vector<uint8_t> cols(n * nt * w, 0);
    for (size_t i = 0; i < n; ++i)
      for (size_t t = 0; t < nt; ++t) std::memcpy(&cols[(i * nt + t) * w], (*seqs[t])[i].data(), (*seqs[t])[i].size());
    patternSite_.resize(n);
    weights_.resize(n);
    indices_.resize(n);
    int64_t np = 0;
    check(bppgpu_site_patterns(cols.data(), (int64_t)n, (int32_t)(nt * w), patternSite_.data(), weights_.data(), indices_.data(), &np),
          "SitePatterns");
    patternSite_.resize((size_t)np);
    weights_.resize((size_t)np);
  }
  const std::vector<unsigned int>& getWeights() const { return weights_; }
  const std::vector<int64_t>& getIndices() const { return indices_; }
  const std::vector<int64_t>& getPatternSites() const { return patternSite_; }

 private:
  std::vector<int64_t> patternSite_, indices_;
  std::vector<unsigned int> weights_;
};

// ---- sites -> patterns -> tip codes ------------------------------------------------------------------------------------------------
// What the engine and the distance routine consume: the global pattern compression of the sequences `names` (in that order), one
// code row per sequence (code = index of the distinct character, in order of first appearance) and the code table
// table[code][state] = model.getInitValue(state, character).
struct TipCodes {
  std::vector<unsigned int> weights;            // [patterns]
  std::vector<int64_t> siteIndex;               // [sites] -> pattern
  std::vector<std::vector<uint16_t> > codes;    // [names][patterns]
  std::vector<double> table;                    // [nCodes][S]
  size_t nCodes;
};
inline TipCodes encodeTipCodes(const VectorSiteContainer& sites, const std::vector<std::string>& names, const SubstitutionModel& model) {
  SitePatterns patterns(sites, names);
  TipCodes tc;
  const size_t np = patterns.getWeights().size();
  tc.weights = patterns.getWeights();
  tc.siteIndex = patterns.getIndices();
  std::map<std::string, int> codeOf;
  std::vector<std::string> chars;
  tc.codes.assign(names.size(), std::vector<uint16_t>(np));
  for (size_t t = 0; t < names.size(); ++t) {
    const BasicSequence& seq = sites.getSequence(names[t]);
    for (size_t k = 0; k < np; ++k) {
      const std::string& ch = seq[(size_t)patterns.getPatternSites()[k]];
      std::map<std::string, int>::iterator it = codeOf.find(ch);
      if (it == codeOf.end()) { it = codeOf.insert(std::make_pair(ch, (int)chars.size())).first; chars.push_back(ch); }
      tc.codes[t][k] = (uint16_t)it->second;
    }
  }
  const size_t S = model.getNumberOfStates();
  tc.nCodes = chars.size();
  tc.table.resize(chars.size() * S);
  for (size_t k = 0; k < chars.size(); ++k)
    for (size_t s = 0; s < S; ++s) tc.table[k * S + s] = model.getInitValue(s, chars[k]);
  return tc;
}

// ---- tree likelihood ---------------------------------------------------------------------------------------------------------------
struct Parameter {
  std::string name;
  double value;
};
typedef std::vector<Parameter> ParameterList;

// Common engine-backed implementation of {R,DR}HomogeneousTreeLikelihood and DRNonHomogeneousTreeLikelihood
class AbstractHomogeneousTreeLikelihood {
 public:
  virtual ~AbstractHomogeneousTreeLikelihood() { if (engine_) bppgpu_destroy(engine_); }
  AbstractHomogeneousTreeLikelihood(const AbstractHomogeneousTreeLikelihood&) = delete;
  AbstractHomogeneousTreeLikelihood& operator=(const AbstractHomogeneousTreeLikelihood&) = delete;

  // AbstractHomogeneousTreeLikelihood::initialize (:235-244)
  void initialize() {
    if (initialized_) throw Exception("Object already initialized.");
    if (!hasData_) throw Exception("Impossible to initialize, no data provided.");
    initialized_ = true;
    fireParameterChanged();
  }
  // value of the function = -lnL (RHomogeneousTreeLikelihood.cpp:287-291)
  double getValue() const {
    if (!initialized_) throw Exception("RHomogeneousTreeLikelihood::getValue(). Instance is not initialized.");
    return minusLogLik_;
  }
  double getLogLikelihood() const { return -getValue(); }
  double getLogLikelihoodForASite(size_t site) const { requireInit(); return siteLnl_[(size_t)siteIndex_[site]]; }
  double getLikelihoodForASite(size_t site) const { return std::exp(getLogLikelihoodForASite(site)); }
  Vdouble getLogLikelihoodForEachSite() const {
    requireInit();
    Vdouble v(siteIndex_.size());
    for (size_t i = 0; i < v.size(); ++i) v[i] = siteLnl_[(size_t)siteIndex_[i]];
    return v;
  }
  const Vdouble& getLogLikelihoodForEachDistinctSite() const { requireInit(); return siteLnl_; }
  size_t getNumberOfSites() const { return siteIndex_.size(); }
  size_t getNumberOfDistinctSites() const { return (size_t)nPatterns_; }
  size_t getSiteIndex(size_t site) const { return (size_t)siteIndex_[site]; }
  size_t getNumberOfStates() const { return model_->getNumberOfStates(); }
  size_t getNumberOfClasses() const { return rDist_->getNumberOfCategories(); }
  const Vdouble& getRootFrequencies() const { return rootFreqs_; }
  const Tree& getTree() const { return *tree_; }

  // "BrLen<i>": i-th node of the post-order list with the root dropped (init_ :155-157)
  ParameterList getBranchLengthsParameters() const {
    ParameterList pl;
    for (size_t i = 0; i < brLen_.size(); ++i) {
      if (reparametrizeRoot_ && ((int)i == root1_ || (int)i == root2_)) continue;
      pl.push_back({"BrLen" + std::to_string(i), brLen_[i]});
    }
    if (reparametrizeRoot_) {  // AbstractNonHomogeneousTreeLikelihood::initBranchLengthsParameters (:386-389)
      pl.push_back({"BrLenRoot", brLen_[(size_t)root1_] + brLen_[(size_t)root2_]});
      pl.push_back({"RootPosition", brLen_[(size_t)root1_] / (brLen_[(size_t)root1_] + brLen_[(size_t)root2_])});
    }
    return pl;
  }
  ParameterList getSubstitutionModelParameters() const {
    ParameterList pl;
    if (modelSet_) for (const std::string& n : modelSet_->getParameterNames()) pl.push_back({n, modelSet_->getParameterValue(n)});
    else for (const std::string& n : model_->getParameterNames()) pl.push_back({n, model_->getParameterValue(n)});
    return pl;
  }
  const SubstitutionModelSet* getSubstitutionModelSet() const { return modelSet_; }
  double getParameterValue(const std::string& name) const {
    if (reparametrizeRoot_ && name == "BrLenRoot") return brLen_[(size_t)root1_] + brLen_[(size_t)root2_];
    if (reparametrizeRoot_ && name == "RootPosition") return brLen_[(size_t)root1_] / (brLen_[(size_t)root1_] + brLen_[(size_t)root2_]);
    int b = brlenIndex(name);
    if (b < 0) throw ParameterNotFoundException("ParameterNotFoundException: " + name);
    return brLen_[(size_t)b];
  }
  // setParameters -> fireParameterChanged (RHomogeneousTreeLikelihood.cpp:255-283): P(t) of the changed branches (or
  // all of them when a model / rate-distribution parameter moved) are rebuilt and the whole tree is re-pruned
  void setParameterValue(const std::string& name, double value) { setParametersValues({{name, value}}); }
  void setParametersValues(const ParameterList& pl) {
    bool modelChanged = false;
    for (const Parameter& p : pl) {
      if (reparametrizeRoot_ && (p.name == "BrLenRoot" || p.name == "RootPosition")) {
        // applyParameters (AbstractNonHomogeneousTreeLikelihood.cpp:319-330): l1 = len * pos, l2 = len * (1 - pos)
        double len = brLen_[(size_t)root1_] + brLen_[(size_t)root2_], pos = brLen_[(size_t)root1_] / len;
        if (p.name == "BrLenRoot") len = p.value; else pos = p.value;
        brLen_[(size_t)root1_] = len * pos;
        brLen_[(size_t)root2_] = len * (1.0 - pos);
        continue;
      }
      if (applyBranchParameter(p.name, p.value)) continue;
      const int b = brlenIndex(p.name);
      if (b >= 0) brLen_[(size_t)b] = std::min(std::max(p.value, minimumBrLen_), maximumBrLen_);
      else {
        try { if (modelSet_) modelSet_->setParameterValue(p.name, p.value); else model_->setParameterValue(p.name, p.value); }
        catch (ParameterNotFoundException&) { rDist_->setParameterValue(p.name, p.value); }
        modelChanged = true;
      }
    }
    if (modelChanged) uploadModel();
    if (initialized_) fireParameterChanged();
  }
  void setParameters(const ParameterList& pl) { setParametersValues(pl); }
  // the model object was changed from outside (a mixed model re-deriving its sub-models): re-upload and re-evaluate
  void modelParametersChanged() { uploadModel(); if (initialized_) fireParameterChanged(); }

  // derivatives w.r.t. branch lengths of -lnL (RHomogeneousTreeLikelihood.cpp:346-361, DRHomogeneousTreeLikelihood.cpp:340-368)
  double getFirstOrderDerivative(const std::string& variable) const { return derivative(variable, 1); }
  double getSecondOrderDerivative(const std::string& variable) const { return derivative(variable, 2); }
  void enableDerivatives(bool yn) { computeDerivatives_ = yn; }
  // DRASDRTreeLikelihoodData::getDLikelihoodArray / getD2LikelihoodArray (nodeId): (dL_i / dt) / L_i and (d2L_i / dt2) / L_i per
  // distinct site, computed on the device from the resident DR arrays
  Vdouble getDLikelihoodArray(int nodeId) const { return siteDerivatives(nodeId, 1); }
  Vdouble getD2LikelihoodArray(int nodeId) const { return siteDerivatives(nodeId, 2); }
  const std::vector<unsigned int>& getWeights() const { return patternWeights_; }

  // pxy_[node][class][x][y] (getTransitionProbabilitiesPerRateClass)
  VVVdouble getTransitionProbabilitiesPerRateClass(int nodeId, size_t /*siteIndex*/ = 0) const {
    requireInit();
    const size_t S = getNumberOfStates(), C = getNumberOfClasses();
    std::vector<double> buf(C * S * S);
    check(bppgpu_get_transition_probabilities(engine_, 0, nodeId, BPPGPU_WANT_P, buf.data()), "getTransitionProbabilities");
    VVVdouble p(C, VVdouble(S, Vdouble(S)));
    for (size_t c = 0; c < C; ++c)
      for (size_t x = 0; x < S; ++x)
        for (size_t y = 0; y < S; ++y) p[c][x][y] = buf[(c * S + x) * S + y];
    return p;
  }
  // ---- DiscreteRatesAcrossSitesTreeLikelihood accessors (DiscreteRatesAcrossSitesTreeLikelihood.h:70-203) ---------------------------
  // All of them read the root arrays of the last evaluation (DRHomogeneousTreeLikelihood.cpp:203-227: rootSiteLikelihoods_[i][c] =
  // sum_x pi_x rootLikelihoods_[i][c][x]); they stay on the device until one of these is called, then come back once, scaled:
  // true value = array * 2^-exponent, and everything below is combined in log space so that sites under 1e-308 stay finite.
  double getLogLikelihoodForASiteForARateClass(size_t site, size_t rateClass) const {
    ensureRootArrays();
    return rootLogS_[(size_t)siteIndex_[site] * getNumberOfClasses() + rateClass];
  }
  double getLikelihoodForASiteForARateClass(size_t site, size_t rateClass) const { return std::exp(getLogLikelihoodForASiteForARateClass(site, rateClass)); }
  double getLogLikelihoodForASiteForARateClassForAState(size_t site, size_t rateClass, int state) const {
    ensureRootArrays();
    const size_t C = getNumberOfClasses(), S = getNumberOfStates(), row = (size_t)siteIndex_[site] * C + rateClass;
    return std::log(rootL_[row * S + (size_t)state]) - rootExp_[row] * 0.693147180559945309417232121458;
  }
  double getLikelihoodForASiteForARateClassForAState(size_t site, size_t rateClass, int state) const {
    ensureRootArrays();
    const size_t C = getNumberOfClasses(), S = getNumberOfStates(), row = (size_t)siteIndex_[site] * C + rateClass;
    return std::ldexp(rootL_[row * S + (size_t)state], -rootExp_[row]);
  }
  // AbstractDiscreteRatesAcrossSitesTreeLikelihood.cpp:110-133: sum_c p_c L[site][c][state]
  double getLikelihoodForASiteForAState(size_t site, int state) const {
    double l = 0;
    for (size_t c = 0; c < getNumberOfClasses(); ++c) l += getLikelihoodForASiteForARateClassForAState(site, c, state) * rDist_->getProbability(c);
    return l;
  }
  double getLogLikelihoodForASiteForAState(size_t site, int state) const { return std::log(getLikelihoodForASiteForAState(site, state)); }
  VVdouble getLikelihoodForEachSiteForEachRateClass() const { return eachSiteEachClass(false); }       // :92-106
  VVdouble getLogLikelihoodForEachSiteForEachRateClass() const { return eachSiteEachClass(true); }     // :137-151
  VVVdouble getLikelihoodForEachSiteForEachRateClassForEachState() const { return eachSiteEachClassEachState(false); }     // :155-174
  VVVdouble getLogLikelihoodForEachSiteForEachRateClassForEachState() const { return eachSiteEachClassEachState(true); }   // :178-197
  // :201-215  pb[i][c] = L[i][c] p_c / L[i]
  VVdouble getPosteriorProbabilitiesOfEachRate() const {
    ensureRootArrays();
    const size_t C = getNumberOfClasses();
    VVdouble pb(siteIndex_.size(), Vdouble(C));
    for (size_t i = 0; i < pb.size(); ++i) {
      const size_t k = (size_t)siteIndex_[i];
      for (size_t c = 0; c < C; ++c) pb[i][c] = std::exp(rootLogS_[k * C + c] - siteLnl_[k]) * rDist_->getProbability(c);
    }
    return pb;
  }
  // :219-234  sum_c (L[i][c] / L[i]) p_c r_c
  Vdouble getPosteriorRateOfEachSite() const {
    const VVdouble pb = getPosteriorProbabilitiesOfEachRate();
    Vdouble rates(pb.size(), 0.0);
    for (size_t i = 0; i < pb.size(); ++i)
      for (size_t c = 0; c < pb[i].size(); ++c) rates[i] += pb[i][c] * rDist_->getCategory(c);
    return rates;
  }
  // :238-248  whichMax of L[i][.] (first maximum; NOT weighted by p_c, like the reference)
  std::vector<size_t> getRateClassWithMaxPostProbOfEachSite() const {
    ensureRootArrays();
    const size_t C = getNumberOfClasses();
    std::vector<size_t> classes(siteIndex_.size(), 0);
    for (size_t i = 0; i < classes.size(); ++i) {
      const double* l = &rootLogS_[(size_t)siteIndex_[i] * C];
      for (size_t c = 1; c < C; ++c) if (l[c] > l[classes[i]]) classes[i] = c;
    }
    return classes;
  }
  Vdouble getRateWithMaxPostProbOfEachSite() const {   // :252-262
    const std::vector<size_t> cl = getRateClassWithMaxPostProbOfEachSite();
    Vdouble rates(cl.size());
    for (size_t i = 0; i < cl.size(); ++i) rates[i] = rDist_->getCategory(cl[i]);
    return rates;
  }

  // TreeLikelihood::getTransitionProbabilities(nodeId, siteIndex): the class tables averaged with the class probabilities
  // (AbstractDiscreteRatesAcrossSitesTreeLikelihood.cpp:310-329)
  VVdouble getTransitionProbabilities(int nodeId, size_t siteIndex = 0) const {
    const VVVdouble p3 = getTransitionProbabilitiesPerRateClass(nodeId, siteIndex);
    const size_t S = getNumberOfStates();
    VVdouble p2(S, Vdouble(S, 0.0));
    for (size_t i = 0; i < S; ++i)
      for (size_t j = 0; j < S; ++j)
        for (size_t k = 0; k < p3.size(); ++k) p2[i][j] += p3[k][i][j] * rDist_->getProbability(k);
    return p2;
  }
  // DRTreeLikelihood::computeLikelihoodAtNode-style access to the device-resident conditional likelihoods of an internal
  // node (subtree below it): true value = likelihoodArray[i][c][x] * 2^-scale[i][c]
  void getLikelihoodArray(int nodeId, VVVdouble& likelihoodArray, std::vector<std::vector<int> >& scale) const {
    requireInit();
    const size_t S = getNumberOfStates(), C = getNumberOfClasses(), N = (size_t)nPatterns_;
    std::vector<double> buf(N * C * S);
    std::vector<int32_t> ex(N * C);
    check(bppgpu_get_clv(engine_, 0, nodeId, 0, buf.data(), ex.data()), "getLikelihoodArray");
    likelihoodArray.assign(N, VVdouble(C, Vdouble(S)));
    scale.assign(N, std::vector<int>(C));
    for (size_t i = 0; i < N; ++i)
      for (size_t c = 0; c < C; ++c) {
        scale[i][c] = ex[i * C + c];
        for (size_t x = 0; x < S; ++x) likelihoodArray[i][c][x] = buf[(i * C + c) * S + x];
      }
  }
  // DRTreeLikelihood::computeLikelihoodAtNode(nodeId, VVVdouble&) (Likelihood/DRTreeLikelihood.h:92-102): the conditional
  // likelihood of ALL the data given the state at the node, computed on the device from the resident lower / upper
  // arrays; true value = likelihoodArray[i][c][x] * 2^-scale[i][c] (scale may be null: values are then de-scaled)
  void computeLikelihoodAtNode(int nodeId, VVVdouble& likelihoodArray, std::vector<std::vector<int> >* scale = nullptr) const {
    requireInit();
    ensureDerivativePass();
    const size_t S = getNumberOfStates(), C = getNumberOfClasses(), N = (size_t)nPatterns_;
    std::vector<double> buf(N * C * S);
    std::vector<int32_t> ex(N * C);
    check(bppgpu_get_node_posteriors(engine_, 0, nodeId, buf.data(), ex.data(), nullptr), "computeLikelihoodAtNode");
    likelihoodArray.assign(N, VVdouble(C, Vdouble(S)));
    if (scale) scale->assign(N, std::vector<int>(C));
    for (size_t i = 0; i < N; ++i)
      for (size_t c = 0; c < C; ++c) {
        if (scale) (*scale)[i][c] = ex[i * C + c];
        for (size_t x = 0; x < S; ++x)
          likelihoodArray[i][c][x] = scale ? buf[(i * C + c) * S + x] : std::ldexp(buf[(i * C + c) * S + x], -ex[i * C + c]);
      }
  }
  // DRTreeLikelihoodTools::getPosteriorProbabilitiesForEachStateForEachRate(drl, nodeId) (DRTreeLikelihoodTools.cpp:46-119)
  VVVdouble getPosteriorProbabilitiesForEachStateForEachRate(int nodeId) const {
    requireInit();
    ensureDerivativePass();
    const size_t S = getNumberOfStates(), C = getNumberOfClasses(), N = (size_t)nPatterns_;
    std::vector<double> buf(N * C * S);
    check(bppgpu_get_node_posteriors(engine_, 0, nodeId, nullptr, nullptr, buf.data()), "getPosteriorProbabilities");
    VVVdouble p(N, VVdouble(C, Vdouble(S)));
    for (size_t i = 0; i < N; ++i)
      for (size_t c = 0; c < C; ++c)
        for (size_t x = 0; x < S; ++x) p[i][c][x] = buf[(i * C + c) * S + x];
    return p;
  }
  // MarginalAncestralStateReconstruction::getAncestralStatesForNode: argmax_x sum_c posterior, one state per distinct site
  std::vector<size_t> getAncestralStatesForNode(int nodeId) const {
    const VVVdouble p = getPosteriorProbabilitiesForEachStateForEachRate(nodeId);
    std::vector<size_t> best(p.size(), 0);
    for (size_t i = 0; i < p.size(); ++i) {
      double bv = -1;
      for (size_t x = 0; x < p[i][0].size(); ++x) {
        double v = 0;
        for (size_t c = 0; c < p[i].size(); ++c) v += p[i][c][x];
        if (v > bv) { bv = v; best[i] = x; }
      }
    }
    return best;
  }
  // MarginalNonRevAncestralStateReconstruction's per-node tables (fork, MarginalNonRev...cpp:10-136) from the device-resident
  // arrays: post[i][x] = P(node = x | site i), joint[i][x][y] = P(node = x, father = y | site i) (null / ignored at the root)
  void getMarginalPosteriors(int nodeId, VVdouble& post, VVVdouble* joint) const {
    requireInit();
    const size_t S = getNumberOfStates(), N = (size_t)nPatterns_;
    const bool isRoot = nodeId == (int)nodes_.size() - 1;
    if (!isRoot) ensureDerivativePass();
    std::vector<double> pb(N * S), jb(joint && !isRoot ? N * S * S : 0);
    check(bppgpu_get_marginal_posteriors(engine_, 0, nodeId, pb.data(), jb.empty() ? nullptr : jb.data()), "MarginalNonRevAncestralStateReconstruction");
    post.assign(N, Vdouble(S));
    for (size_t i = 0; i < N; ++i)
      for (size_t x = 0; x < S; ++x) post[i][x] = pb[i * S + x];
    if (joint) {
      joint->assign(N, VVdouble(S, Vdouble(S, 0.0)));
      if (!isRoot)
        for (size_t i = 0; i < N; ++i)
          for (size_t x = 0; x < S; ++x)
            for (size_t y = 0; y < S; ++y) (*joint)[i][x][y] = jb[(i * S + x) * S + y];
    }
  }
  // MLAncestralStateReconstruction's result (fork): states[node][distinct site] of the joint ML assignment, computed on the
  // device with the transition probabilities and root frequencies of the last evaluation; bestLogLik[i] = its log joint likelihood
  void getJointMLAncestralStates(std::vector<std::vector<size_t> >& states, Vdouble* bestLogLik = nullptr) const {
    requireInit();
    const size_t N = (size_t)nPatterns_, nn = nodes_.size();
    std::vector<int32_t> buf(nn * N);
    Vdouble best(N);
    check(bppgpu_ml_ancestral_states(engine_, 0, buf.data(), best.data()), "MLAncestralStateReconstruction");
    states.assign(nn, std::vector<size_t>(N));
    for (size_t n = 0; n < nn; ++n)
      for (size_t i = 0; i < N; ++i) states[n][i] = (size_t)buf[n * N + i];
    if (bestLogLik) *bestLogLik = best;
  }
  std::vector<int> getNodesId() const {
    std::vector<int> ids;
    for (const Node* n : nodes_) ids.push_back(n->getId());
    return ids;
  }
  long getNumberOfLikelihoodCalculations() const { return numOfLikelihoodCalculations_; }  // fork: DRNonHomogeneousTreeLikelihood.h:75

 protected:
  AbstractHomogeneousTreeLikelihood(const Tree& tree, SubstitutionModel* model, DiscreteDistribution* rDist, bool checkRooted,
                                    unsigned engineFlags, int device)
      : tree_(new Tree(tree)), model_(model), rDist_(rDist), engine_(nullptr), engineFlags_(engineFlags), device_(device),
        initialized_(false), hasData_(false), computeDerivatives_(true), minusLogLik_(0), nPatterns_(0),
        minimumBrLen_(1e-6), maximumBrLen_(1e4), derivsValid_(false), numOfLikelihoodCalculations_(0) {
    // init_ (AbstractHomogeneousTreeLikelihood.cpp:140-166)
    if (checkRooted && tree_->isRooted()) tree_->unroot();
    tree_->resetNodesId();
    nodes_ = tree_->getNodes();
    for (size_t i = 0; i + 1 < nodes_.size(); ++i) {  // initBranchLengthsParameters (:305-337)
      double d = nodes_[i]->hasDistanceToFather() ? nodes_[i]->getDistanceToFather() : minimumBrLen_;
      d = std::min(std::max(d, minimumBrLen_), maximumBrLen_);
      nodes_[i]->setDistanceToFather(d);
      brLen_.push_back(d);
    }
  }

  // setData (RHomogeneousTreeLikelihood.cpp:131-146): sequences re-ordered to the leaves, global pattern compression, tip codes
  void setData(const VectorSiteContainer& sites) {
    if (sites.getNumberOfSequences() == 0 || sites.getNumberOfSites() == 0)
      throw Exception("DRASRTreeLikelihoodData::initLikelihoods. Can't use empty dataset (0 sequences or 0 sites).");
    const std::vector<std::string> leafNames = tree_->getLeavesNames();
    const TipCodes tc = encodeTipCodes(sites, leafNames, *model_);
    nPatterns_ = (int64_t)tc.weights.size();
    siteIndex_ = tc.siteIndex;
    const std::vector<std::vector<uint16_t> >& codes = tc.codes;
    const std::vector<double>& table = tc.table;
    const size_t S = model_->getNumberOfStates(), C = rDist_->getNumberOfCategories();
    // flattened topology: node id = post-order position
    const int nn = (int)nodes_.size();
    std::vector<int32_t> off(nn + 1, 0), children;
    for (int i = 0; i < nn; ++i) {
      for (size_t k = 0; k < nodes_[i]->getNumberOfSons(); ++k) children.push_back(nodes_[i]->getSon(k)->getId());
      off[i + 1] = (int32_t)children.size();
    }
    bppgpu_config cfg;
    std::memset(&cfg, 0, sizeof(cfg));
    cfg.n_states = (int32_t)S; cfg.n_cats = (int32_t)C; cfg.n_patterns = nPatterns_; cfg.n_nodes = nn; cfg.root = nn - 1;
    cfg.child_offsets = off.data(); cfg.children = children.data(); cfg.n_points = nPoints_;
    cfg.n_models = modelSet_ ? (int32_t)modelSet_->getNumberOfModels() : (nModelSlots_ > 0 ? nModelSlots_ : nPoints_);
    cfg.n_codes = (int32_t)tc.nCodes; cfg.code_bytes = tc.nCodes > 256 ? 2 : 1; cfg.code_table = table.data();
    // a batch of parameter points on one character keeps no per-node arrays: the engine may then apply P(t) in factored form
    cfg.device = device_; cfg.flags = engineFlags_ | ((nPoints_ > 1 && nPatterns_ == 1 && C == 1) ? 0u : (unsigned)BPPGPU_FLAG_KEEP_CLVS);
    if (engine_) { bppgpu_destroy(engine_); engine_ = nullptr; }
    check(bppgpu_create(&cfg, &engine_), "TreeLikelihood::setData");
    const std::vector<Node*> leaves = tree_->getLeaves();
    for (size_t t = 0; t < leaves.size(); ++t) {
      if (cfg.code_bytes == 1) {
        std::vector<uint8_t> c8(codes[t].begin(), codes[t].end());
        check(bppgpu_set_tip_codes(engine_, leaves[t]->getId(), c8.data()), "setData");
      } else {
        check(bppgpu_set_tip_codes(engine_, leaves[t]->getId(), codes[t].data()), "setData");
      }
    }
    check(bppgpu_set_pattern_weights(engine_, tc.weights.data()), "setData");
    patternWeights_ = tc.weights;
    hasData_ = true;
    uploadModel();
  }

  // hook for classes whose branch lengths are functions of other parameters (clock heights): true = name consumed
  virtual bool applyBranchParameter(const std::string&, double) { return false; }
  virtual Vdouble rootFrequencies() const { return modelSet_ ? modelSet_->getRootFrequencies() : model_->getFrequencies(); }

  virtual void uploadModel() {
    if (!engine_) return;
    bppgpu_model_desc d;
    if (modelSet_) {
      // AbstractNonHomogeneousTreeLikelihood::computeTransitionProbabilitiesForNode (.cpp:410-468): the branch above a node
      // uses modelSet_->getModelForNode(node id); one device slot per model of the set
      for (size_t k = 0; k < modelSet_->getNumberOfModels(); ++k) {
        modelSet_->getModel(k)->fillModelDesc(d);
        check(bppgpu_set_model(engine_, (int32_t)k, &d), "setModel");
      }
      std::vector<int32_t> slot(nodes_.size(), 0);
      for (size_t i = 0; i + 1 < nodes_.size(); ++i) slot[i] = (int32_t)modelSet_->getModelIndexForNode(nodes_[i]->getId());
      check(bppgpu_set_branch_models(engine_, 0, slot.data()), "setBranchModels");
    } else {
      model_->fillModelDesc(d);
      check(bppgpu_set_model(engine_, 0, &d), "setModel");
    }
    Vdouble r(rDist_->getNumberOfCategories()), p(r.size());
    for (size_t c = 0; c < r.size(); ++c) { r[c] = rDist_->getCategory(c); p[c] = rDist_->getProbability(c); }
    check(bppgpu_set_rates(engine_, r.data(), p.data()), "setRates");
    rootFreqs_ = rootFrequencies();
    check(bppgpu_set_root_freqs(engine_, 0, rootFreqs_.data()), "setRootFreqs");
  }

  // computeAllTransitionProbabilities + computeTreeLikelihood (+ the DR derivative passes) in one device evaluation
  virtual void fireParameterChanged() {
    Vdouble t(nodes_.size(), 0.0);
    for (size_t i = 0; i < brLen_.size(); ++i) t[i] = brLen_[i];
    check(bppgpu_set_branch_lengths(engine_, 0, t.data()), "applyParameters");
    double lnl = 0;
    check(bppgpu_eval(engine_, BPPGPU_EVAL_LNL, &lnl, nullptr, nullptr), "computeTreeLikelihood");
    ++numOfLikelihoodCalculations_;
    minusLogLik_ = -lnl;
    siteLnl_.resize((size_t)nPatterns_);
    check(bppgpu_get_site_lnl(engine_, 0, siteLnl_.data()), "getLogLikelihoodForEachSite");
    if (engineFlags_ & BPPGPU_FLAG_WEIGHTED_ROOT) check(bppgpu_get_root_freqs(engine_, 0, rootFreqs_.data()), "getRootFrequencies");
    derivsValid_ = false;
    rootArraysValid_ = false;
  }

  // the prefix (upper) arrays exist after an evaluation with derivatives
  void ensureDerivativePass() const {
    if (derivsValid_) return;
    d1_.assign(nodes_.size(), 0.0);
    d2_.assign(nodes_.size(), 0.0);
    double lnl = 0;
    check(bppgpu_eval(engine_, BPPGPU_EVAL_LNL | BPPGPU_EVAL_D1 | BPPGPU_EVAL_D2, &lnl, d1_.data(), d2_.data()), "computeTreeDLikelihoods");
    derivsValid_ = true;
  }
  double derivative(const std::string& variable, int order) const {
    requireInit();
    if (reparametrizeRoot_ && (variable == "BrLenRoot" || variable == "RootPosition")) {
      // DRNonHomogeneousTreeLikelihood.cpp:445-478 (first order), :576-867 (second order: needs the cross term of the two
      // root branches, rebuilt on the device)
      ensureDerivativePass();
      double o[4];
      check(bppgpu_get_root_reparam_derivatives(engine_, 0, o), "getSecondOrderDerivative");
      const int k = (order == 1 ? 0 : 2) + (variable == "BrLenRoot" ? 0 : 1);
      return -o[k];
    }
    const int b = brlenIndex(variable);
    if (b < 0) {
      for (const std::string& n : modelSet_ ? modelSet_->getParameterNames() : model_->getParameterNames())
        if (n == variable) throw Exception("Derivatives respective to substitution model parameters are not implemented.");
      throw ParameterNotFoundException("ParameterNotFoundException: " + variable);
    }
    if (!derivsValid_) {
      d1_.assign(nodes_.size(), 0.0);
      d2_.assign(nodes_.size(), 0.0);
      double lnl = 0;
      check(bppgpu_eval(engine_, BPPGPU_EVAL_LNL | BPPGPU_EVAL_D1 | BPPGPU_EVAL_D2, &lnl, d1_.data(), d2_.data()), "computeTreeDLikelihoods");
      derivsValid_ = true;
    }
    return order == 1 ? -d1_[(size_t)b] : -d2_[(size_t)b];
  }
  Vdouble siteDerivatives(int nodeId, int order) const {
    requireInit();
    ensureDerivativePass();
    Vdouble a((size_t)nPatterns_), b((size_t)nPatterns_);
    check(bppgpu_get_site_derivatives(engine_, 0, nodeId, a.data(), order == 2 ? b.data() : nullptr), "getDLikelihoodArray");
    return order == 1 ? a : b;
  }
  int brlenIndex(const std::string& name) const {
    if (name.compare(0, 5, "BrLen") != 0) return -1;
    char* end = nullptr;
    const long i = std::strtol(name.c_str() + 5, &end, 10);
    if (*end != 0 || i < 0 || (size_t)i >= brLen_.size()) return -1;
    return (int)i;
  }
  void requireInit() const { if (!initialized_) throw Exception("Instance is not initialized."); }
  // root arrays of the last evaluation: rootL_[i][c][x] (scaled), rootExp_[i][c], rootLogS_[i][c] = log sum_x pi_x L - exp ln 2
  void ensureRootArrays() const {
    requireInit();
    if (rootArraysValid_) return;
    const size_t S = getNumberOfStates(), C = getNumberOfClasses(), N = (size_t)nPatterns_;
    rootL_.resize(N * C * S);
    std::vector<int32_t> ex(N * C);
    check(bppgpu_get_clv(engine_, 0, (int32_t)nodes_.size() - 1, 0, rootL_.data(), ex.data()), "getRootLikelihoodArray");
    rootExp_.assign(ex.begin(), ex.end());
    rootLogS_.resize(N * C);
    for (size_t r = 0; r < N * C; ++r) {
      double s = 0;
      for (size_t x = 0; x < S; ++x) s += rootFreqs_[x] * rootL_[r * S + x];
      rootLogS_[r] = std::log(s) - rootExp_[r] * 0.693147180559945309417232121458;
    }
    rootArraysValid_ = true;
  }
  VVdouble eachSiteEachClass(bool logs) const {
    ensureRootArrays();
    const size_t C = getNumberOfClasses();
    VVdouble l(siteIndex_.size(), Vdouble(C));
    for (size_t i = 0; i < l.size(); ++i)
      for (size_t c = 0; c < C; ++c) {
        const double v = rootLogS_[(size_t)siteIndex_[i] * C + c];
        l[i][c] = logs ? v : std::exp(v);
      }
    return l;
  }
  VVVdouble eachSiteEachClassEachState(bool logs) const {
    const size_t C = getNumberOfClasses(), S = getNumberOfStates();
    VVVdouble l(siteIndex_.size(), VVdouble(C, Vdouble(S)));
    for (size_t i = 0; i < l.size(); ++i)
      for (size_t c = 0; c < C; ++c)
        for (size_t x = 0; x < S; ++x)
          l[i][c][x] = logs ? getLogLikelihoodForASiteForARateClassForAState(i, c, (int)x) : getLikelihoodForASiteForARateClassForAState(i, c, (int)x);
    return l;
  }

  std::unique_ptr<Tree> tree_;
  SubstitutionModel* model_;      // not owned (like the reference)
  SubstitutionModelSet* modelSet_ = nullptr;  // not owned; non-homogeneous classes: one model per branch group
  DiscreteDistribution* rDist_;   // not owned
  bppgpu_engine* engine_;
  unsigned engineFlags_;
  std::vector<unsigned int> patternWeights_;
  int device_;
  bool initialized_, hasData_, computeDerivatives_;
  double minusLogLik_;
  int64_t nPatterns_;
  std::vector<Node*> nodes_;
  Vdouble brLen_;
  double minimumBrLen_, maximumBrLen_;
  std::vector<int64_t> siteIndex_;
  Vdouble siteLnl_, rootFreqs_;
  mutable Vdouble d1_, d2_;
  mutable bool derivsValid_;
  mutable bool rootArraysValid_ = false;
  mutable Vdouble rootL_, rootLogS_;
  mutable std::vector<int> rootExp_;
  long numOfLikelihoodCalculations_;
  int nPoints_ = 1;  // parameter points evaluated per device call (LikelihoodPointBatch)
  int nModelSlots_ = 0;  // device model slots when they are not one per point (RNonHomogeneousMixedTreeLikelihood)
  bool reparametrizeRoot_ = false;  // BrLenRoot / RootPosition replace the two root branches (NH classes, rooted trees)
  int root1_ = -1, root2_ = -1;     // ids (= BrLen indices) of the root's first two sons
};

// Likelihood/RHomogeneousTreeLikelihood.h:108-138.  `usePatterns` (recursive per-subtree compression) changes only the
// memory layout of the reference, not its results; the device path always uses the global compression.
class RHomogeneousTreeLikelihood : public AbstractHomogeneousTreeLikelihood {
 public:
  RHomogeneousTreeLikelihood(const Tree& tree, const VectorSiteContainer& data, SubstitutionModel* model, DiscreteDistribution* rDist,
                             bool checkRooted = true, bool verbose = true, bool usePatterns = true, int device = 0)
      : AbstractHomogeneousTreeLikelihood(tree, model, rDist, checkRooted, BPPGPU_FLAG_R_SEMANTICS, device) {
    (void)verbose; (void)usePatterns;
    setData(data);
  }
};
// Likelihood/RHomogeneousClockTreeLikelihood.{h,cpp}: the same likelihood with the branch lengths of a rooted, bifurcating tree
// driven by node heights -- "TotalHeight" (height of the root: the longest path to a leaf, TreeTemplateTools::getHeights,
// TreeTemplateTools.cpp:173-186) and "HeightP<id>" (height / father's height) for every internal non-root node
// (initBranchLengthsParameters :121-157, computeBranchLengthsFromHeights :161-179, minimum branch length 0 :87).  No branch
// derivatives (getDerivableParameters is empty, :183-187).
class RHomogeneousClockTreeLikelihood : public RHomogeneousTreeLikelihood {
 public:
  RHomogeneousClockTreeLikelihood(const Tree& tree, const VectorSiteContainer& data, SubstitutionModel* model, DiscreteDistribution* rDist,
                                  bool checkRooted = true, bool verbose = true, int device = 0)
      : RHomogeneousTreeLikelihood(tree, data, model, rDist, false, verbose, true, device) {
    (void)checkRooted;
    if (!tree_->isRooted()) throw Exception("RHomogeneousClockTreeLikelihood::init_(). Tree is unrooted!");
    for (const Node* n : nodes_)
      if (n->getNumberOfSons() > 2) throw Exception("HomogeneousClockTreeLikelihood::init_(). Tree is multifurcating.");
    minimumBrLen_ = 0.0;
    std::vector<double> h(nodes_.size(), 0.0);
    for (size_t i = 0; i < nodes_.size(); ++i)   // post-order: sons first
      for (size_t k = 0; k < nodes_[i]->getNumberOfSons(); ++k) {
        const int s = nodes_[i]->getSon(k)->getId();
        h[i] = std::max(h[i], h[(size_t)s] + brLen_[(size_t)s]);
      }
    totalHeight_ = h.back();
    for (size_t i = 0; i + 1 < nodes_.size(); ++i)
      if (!nodes_[i]->isLeaf()) heightP_[(int)i] = h[i] / h[(size_t)nodes_[i]->getFather()->getId()];
    computeBranchLengthsFromHeights(nodes_.back(), totalHeight_);
  }
  ParameterList getBranchLengthsParameters() const {
    ParameterList pl;
    pl.push_back({"TotalHeight", totalHeight_});
    for (const auto& kv : heightP_) pl.push_back({"HeightP" + std::to_string(kv.first), kv.second});
    return pl;
  }
  double getParameterValue(const std::string& name) const {
    if (name == "TotalHeight") return totalHeight_;
    if (name.compare(0, 7, "HeightP") == 0) {
      std::map<int, double>::const_iterator it = heightP_.find(std::atoi(name.c_str() + 7));
      if (it != heightP_.end()) return it->second;
    }
    throw ParameterNotFoundException("ParameterNotFoundException: " + name);
  }
  ParameterList getDerivableParameters() const { requireInit(); return ParameterList(); }
  double getFirstOrderDerivative(const std::string& variable) const {
    throw Exception("RHomogeneousClockTreeLikelihood: no derivative with respect to " + variable + " (all parameters are non-derivable).");
  }
  double getSecondOrderDerivative(const std::string& variable) const { return getFirstOrderDerivative(variable); }

 protected:
  bool applyBranchParameter(const std::string& name, double value) override {
    if (name == "TotalHeight") totalHeight_ = value;
    else if (name.compare(0, 7, "HeightP") == 0 && heightP_.count(std::atoi(name.c_str() + 7))) heightP_[std::atoi(name.c_str() + 7)] = value;
    else if (name.compare(0, 5, "BrLen") == 0) throw ParameterNotFoundException("ParameterNotFoundException: " + name);
    else return false;
    computeBranchLengthsFromHeights(nodes_.back(), totalHeight_);
    return true;
  }

 private:
  void computeBranchLengthsFromHeights(const Node* node, double height) {
    for (size_t i = 0; i < node->getNumberOfSons(); ++i) {
      const Node* son = node->getSon(i);
      if (son->isLeaf()) brLen_[(size_t)son->getId()] = std::max(minimumBrLen_, height);
      else {
        const double sonHeight = heightP_.at(son->getId()) * height;
        brLen_[(size_t)son->getId()] = std::max(minimumBrLen_, height - sonHeight);
        computeBranchLengthsFromHeights(son, sonHeight);
      }
    }
  }
  double totalHeight_ = 0;
  std::map<int, double> heightP_;
};
// Likelihood/DRHomogeneousTreeLikelihood.h
class DRHomogeneousTreeLikelihood : public AbstractHomogeneousTreeLikelihood {
 public:
  DRHomogeneousTreeLikelihood(const Tree& tree, const VectorSiteContainer& data, SubstitutionModel* model, DiscreteDistribution* rDist,
                              bool checkRooted = true, bool verbose = true, int device = 0)
      : AbstractHomogeneousTreeLikelihood(tree, model, rDist, checkRooted, 0, device) {
    (void)verbose;
    setData(data);
  }
};
// Likelihood/DRNonHomogeneousTreeLikelihood.h:93-146, fork constructor (weightedRootFreq, calculateDerivatives); one model on
// every branch (what ChromosomeNumberOptimizer builds), the tree is kept rooted
class DRNonHomogeneousTreeLikelihood : public AbstractHomogeneousTreeLikelihood {
 public:
  DRNonHomogeneousTreeLikelihood(const Tree& tree, const VectorSiteContainer& data, bool weightedRootFreq, bool calculateDerivatives,
                                 SubstitutionModel* model, DiscreteDistribution* rDist, const Vdouble* rootFreqs = nullptr,
                                 bool verbose = true, int device = 0, bool reparametrizeRoot = false)
      : AbstractHomogeneousTreeLikelihood(tree, model, rDist, false,
                                          BPPGPU_FLAG_NH_DERIV | (weightedRootFreq ? BPPGPU_FLAG_WEIGHTED_ROOT : 0u), device) {
    (void)verbose;
    if (reparametrizeRoot) {  // AbstractNonHomogeneousTreeLikelihood::init_ (:162-189): root1_ / root2_ = the root's two sons
      const Node* root = nodes_.back();
      if (root->getNumberOfSons() != 2) throw Exception("reparametrizeRoot needs a rooted tree (a root with two sons)");
      root1_ = root->getSon(0)->getId();
      root2_ = root->getSon(1)->getId();
      reparametrizeRoot_ = true;
    }
    computeDerivatives_ = calculateDerivatives;
    if (rootFreqs) fixedRootFreqs_ = *rootFreqs;
    setData(data);
  }

  // Likelihood/DRNonHomogeneousTreeLikelihood.h:93-111: (tree, data, SubstitutionModelSet*, rDist, verbose, reparametrizeRoot)
  DRNonHomogeneousTreeLikelihood(const Tree& tree, const VectorSiteContainer& data, SubstitutionModelSet* modelSet,
                                 DiscreteDistribution* rDist, bool verbose = true, bool reparametrizeRoot = false, int device = 0,
                                 unsigned extraFlags = 0)
      : AbstractHomogeneousTreeLikelihood(tree, modelSet->getModel(0), rDist, false, BPPGPU_FLAG_NH_DERIV | extraFlags, device) {
    (void)verbose;
    // AbstractNonHomogeneousTreeLikelihood::setSubstitutionModelSet (.cpp:193-216)
    if (!modelSet->isFullySetUpFor(*tree_)) throw Exception("AbstractNonHomogeneousTreeLikelihood::init_(). Model set is not fully specified.");
    modelSet_ = modelSet;
    if (reparametrizeRoot) {
      const Node* root = nodes_.back();
      if (root->getNumberOfSons() != 2) throw Exception("reparametrizeRoot needs a rooted tree (a root with two sons)");
      root1_ = root->getSon(0)->getId();
      root2_ = root->getSon(1)->getId();
      reparametrizeRoot_ = true;
    }
    setData(data);
  }

 protected:
  Vdouble rootFrequencies() const {
    if (modelSet_) return modelSet_->getRootFrequencies();
    return fixedRootFreqs_.empty() ? model_->getFrequencies() : fixedRootFreqs_;
  }

 private:
  Vdouble fixedRootFreqs_;
};
// Likelihood/RNonHomogeneousTreeLikelihood.h: (tree, data, modelSet, rDist, verbose, usePatterns, reparametrizeRoot); the R
// classes' root reduction (non-positive terms dropped), same device path
class RNonHomogeneousTreeLikelihood : public DRNonHomogeneousTreeLikelihood {
 public:
  RNonHomogeneousTreeLikelihood(const Tree& tree, const VectorSiteContainer& data, SubstitutionModelSet* modelSet,
                                DiscreteDistribution* rDist, bool verbose = true, bool usePatterns = true, bool reparametrizeRoot = false,
                                int device = 0)
      : DRNonHomogeneousTreeLikelihood(tree, data, modelSet, rDist, verbose, reparametrizeRoot, device, BPPGPU_FLAG_R_SEMANTICS) {
    (void)usePatterns;
  }
};

// ---- batched front-end (SURVEY 8f-1) ------------------------------------------------------------------------------------------
// ChromosomeNumberOptimizer keeps a vector of DRNonHomogeneousTreeLikelihood objects, one per starting point, and evaluates
// and line-searches them one after the other (Likelihood/ChromosomeNumberOptimizer.cpp:58, :141-153, :472-517).  This class
// is that vector as ONE device object: same tree and data, one substitution model (and optionally one set of branch lengths)
// per point, every point's -lnL from a single bppgpu_eval (batched P(t) + one launch per node covering all points).
// Values are identical to what a DRNonHomogeneousTreeLikelihood built on models[k] returns.
class LikelihoodPointBatch : public AbstractHomogeneousTreeLikelihood {
 public:
  LikelihoodPointBatch(const Tree& tree, const VectorSiteContainer& data, bool weightedRootFreq,
                       const std::vector<SubstitutionModel*>& models, DiscreteDistribution* rDist, int device = 0,
                       bool checkRooted = false, unsigned engineFlags = BPPGPU_FLAG_NH_DERIV)
      : AbstractHomogeneousTreeLikelihood(tree, models.at(0), rDist, checkRooted,
                                          engineFlags | (weightedRootFreq ? BPPGPU_FLAG_WEIGHTED_ROOT : 0u), device),
        models_(models) {
    nPoints_ = (int)models.size();
    computeDerivatives_ = false;
    pointBrLen_.assign(models.size(), brLen_);
    values_.assign(models.size(), 0.0);
    setData(data);
  }
  size_t getNumberOfPoints() const { return models_.size(); }
  // a model parameter of point k moved (the caller changed models[k]): its eigensystem is re-uploaded before the next evaluation
  void modelChanged(size_t k) { dirty_.at(k) = 1; if (initialized_) fireParameterChanged(); }
  // several points changed: mark them all, then evaluate() once (one device call for every point)
  void markModelChanged(size_t k) { dirty_.at(k) = 1; }
  void evaluate() { requireInit(); fireParameterChanged(); }
  void setBranchLengths(size_t k, const Vdouble& brlen) {
    if (brlen.size() != brLen_.size()) throw Exception("LikelihoodPointBatch::setBranchLengths: wrong number of branch lengths");
    for (size_t i = 0; i < brlen.size(); ++i) pointBrLen_.at(k)[i] = std::min(std::max(brlen[i], minimumBrLen_), maximumBrLen_);
    if (initialized_) fireParameterChanged();
  }
  // -lnL of every point (getValue() of the k-th likelihood of the reference's vector)
  const Vdouble& getValues() const { requireInit(); return values_; }
  double getValue(size_t k) const { requireInit(); return values_.at(k); }
  // index of the best point (the reference sorts its vector with compareLikValues, ChromosomeNumberOptimizer.cpp:156)
  size_t getBestPoint() const {
    requireInit();
    size_t b = 0;
    for (size_t k = 1; k < values_.size(); ++k) if (values_[k] < values_[b]) b = k;
    return b;
  }

 protected:
  void uploadModel() override {
    if (!engine_) return;
    if (dirty_.size() != models_.size()) dirty_.assign(models_.size(), 1);
    Vdouble r(rDist_->getNumberOfCategories()), p(r.size());
    for (size_t c = 0; c < r.size(); ++c) { r[c] = rDist_->getCategory(c); p[c] = rDist_->getProbability(c); }
    check(bppgpu_set_rates(engine_, r.data(), p.data()), "setRates");
    for (size_t k = 0; k < models_.size(); ++k) {
      if (!dirty_[k]) continue;
      bppgpu_model_desc d;
      models_[k]->fillModelDesc(d);
      check(bppgpu_set_model(engine_, (int32_t)k, &d), "setModel");
      const Vdouble f = models_[k]->getFrequencies();
      check(bppgpu_set_root_freqs(engine_, (int32_t)k, f.data()), "setRootFreqs");
      dirty_[k] = 0;
    }
  }
  void fireParameterChanged() override {
    uploadModel();
    for (size_t k = 0; k < models_.size(); ++k) {
      Vdouble t(nodes_.size(), 0.0);
      for (size_t i = 0; i < brLen_.size(); ++i) t[i] = pointBrLen_[k][i];
      check(bppgpu_set_branch_lengths(engine_, (int32_t)k, t.data()), "applyParameters");
    }
    Vdouble lnl(models_.size(), 0.0);
    check(bppgpu_eval(engine_, BPPGPU_EVAL_LNL, lnl.data(), nullptr, nullptr), "computeTreeLikelihood");
    numOfLikelihoodCalculations_ += (long)models_.size();
    for (size_t k = 0; k < models_.size(); ++k) values_[k] = -lnl[k];
    minusLogLik_ = values_[0];
    derivsValid_ = false;
    rootArraysValid_ = false;
  }

 private:
  std::vector<SubstitutionModel*> models_;  // not owned
  std::vector<Vdouble> pointBrLen_;
  std::vector<char> dirty_;
  Vdouble values_;
};

// ---- mixture of substitution models (SURVEY 8f-3) ------------------------------------------------------------------------------
// RHomogeneousMixedTreeLikelihood keeps one RHomogeneousTreeLikelihood per sub-model of a MixedSubstitutionModel and combines
// them per site and rate class with the sub-model probabilities, L_site = sum_k probas_k L_k,site
// (Likelihood/RHomogeneousMixedTreeLikelihood.cpp:191-212; YNGP M-series, RELAX).  Here the sub-likelihoods are the points of one
// device object and the combination is a log-sum-exp over their per-site log-likelihoods.
class RHomogeneousMixedTreeLikelihood : public LikelihoodPointBatch {
 public:
  RHomogeneousMixedTreeLikelihood(const Tree& tree, const VectorSiteContainer& data, const std::vector<SubstitutionModel*>& subModels,
                                  const Vdouble& probas, DiscreteDistribution* rDist, int device = 0)
      : LikelihoodPointBatch(tree, data, false, subModels, rDist, device, /*checkRooted=*/true, /*engineFlags=*/0u), probas_(probas) {
    if (probas_.size() != subModels.size()) throw Exception("RHomogeneousMixedTreeLikelihood: one probability per sub-model");
  }
  // Likelihood/RHomogeneousMixedTreeLikelihood.h: (tree, data, model, rDist, checkRooted, verbose, usePatterns) with a mixed model
  RHomogeneousMixedTreeLikelihood(const Tree& tree, const VectorSiteContainer& data, MixedSubstitutionModel* model, DiscreteDistribution* rDist,
                                  bool checkRooted = true, bool verbose = true, bool usePatterns = true, int device = 0)
      : LikelihoodPointBatch(tree, data, false, subModelsOf(model), rDist, device, checkRooted, /*engineFlags=*/0u),
        probas_(model->getProbabilities()) { (void)verbose; (void)usePatterns; }
  static std::vector<SubstitutionModel*> subModelsOf(const MixedSubstitutionModel* m) {
    std::vector<SubstitutionModel*> v;
    for (size_t k = 0; k < m->getNumberOfModels(); ++k) v.push_back(m->getNModel(k));
    return v;
  }
  void setProbabilities(const Vdouble& p) { probas_ = p; if (initialized_) combine(); }
  double getValue() const { requireInit(); return mixedMinusLogLik_; }
  double getLogLikelihood() const { return -getValue(); }
  double getLogLikelihoodForASite(size_t site) const { requireInit(); return mixedSiteLnl_[(size_t)siteIndex_[site]]; }

 protected:
  void fireParameterChanged() override {
    LikelihoodPointBatch::fireParameterChanged();
    combine();
  }

 private:
  void combine() {
    const size_t K = getNumberOfPoints(), N = (size_t)nPatterns_;
    std::vector<Vdouble> sl(K, Vdouble(N));
    for (size_t k = 0; k < K; ++k) check(bppgpu_get_site_lnl(engine_, (int32_t)k, sl[k].data()), "getLogLikelihoodForEachSite");
    mixedSiteLnl_.assign(N, 0.0);
    for (size_t i = 0; i < N; ++i) {
      double m = -std::numeric_limits<double>::infinity();
      for (size_t k = 0; k < K; ++k) if (probas_[k] > 0) m = std::max(m, sl[k][i]);
      double s = 0;
      for (size_t k = 0; k < K; ++k) if (probas_[k] > 0) s += probas_[k] * std::exp(sl[k][i] - m);
      mixedSiteLnl_[i] = std::isfinite(m) ? m + std::log(s) : m;
    }
    // getLogLikelihood (RHomogeneousTreeLikelihood.cpp:162-176): every site, sorted, summed
    Vdouble la(siteIndex_.size());
    for (size_t j = 0; j < la.size(); ++j) la[j] = mixedSiteLnl_[(size_t)siteIndex_[j]];
    std::sort(la.begin(), la.end());
    double ll = 0;
    for (size_t j = la.size(); j > 0; --j) ll += la[j - 1];
    mixedMinusLogLik_ = -ll;
  }
  Vdouble probas_, mixedSiteLnl_;
  double mixedMinusLogLik_ = 0;
};

// Likelihood/DRHomogeneousMixedTreeLikelihood.{h,cpp}: one DRHomogeneousTreeLikelihood per sub-model of a mixed model
// (treeLikelihoodsContainer_, .cpp:60-78), combined with the sub-model probabilities:
//   L_i            = sum_j p_j L_j,i                                                   (getLogLikelihood :239-268)
//   d(-lnL)/dt_b   = - sum_i w_i sum_j p_j dL_j[i]                                      (getFirstOrderDerivative :399-437)
//   d2(-lnL)/dt_b2 = - sum_i w_i ( sum_j p_j d2L_j[i] - (sum_j p_j dL_j[i])^2 )         (getSecondOrderDerivative :462-508)
// where dL_j / d2L_j are sub-likelihood j's OWN relative arrays (getDLikelihoodArray: already divided by L_j,i) -- the
// reference's combination, reproduced literally.  Each sub-likelihood owns a device engine; per-site arrays come from
// bppgpu_get_site_lnl / bppgpu_get_site_derivatives.
class DRHomogeneousMixedTreeLikelihood {
 public:
  DRHomogeneousMixedTreeLikelihood(const Tree& tree, const VectorSiteContainer& data, MixedSubstitutionModel* model,
                                   DiscreteDistribution* rDist, bool checkRooted = true, bool verbose = true, bool rootArray = false,
                                   int device = 0)
      : model_(model) {
    (void)verbose; (void)rootArray;
    if (!model) throw Exception("Bad model: DRHomogeneousMixedTreeLikelihood needs a MixedTransitionModel.");
    for (size_t k = 0; k < model->getNumberOfModels(); ++k)
      subs_.emplace_back(new DRHomogeneousTreeLikelihood(tree, data, model->getNModel(k), rDist, checkRooted, false, device));
    probas_ = model->getProbabilities();
  }
  void initialize() {
    for (auto& s : subs_) s->initialize();
    initialized_ = true;
  }
  size_t getNumberOfModels() const { return subs_.size(); }
  const DRHomogeneousTreeLikelihood* getSubLikelihood(size_t k) const { return subs_.at(k).get(); }
  // parameters shared by every sub-likelihood (branch lengths, rate distribution); model parameters go through the mixed model
  void setParameterValue(const std::string& name, double value) {
    for (auto& s : subs_) s->setParameterValue(name, value);
  }
  void setParametersValues(const ParameterList& pl) {
    for (auto& s : subs_) s->setParametersValues(pl);
  }
  // fireParameterChanged (:170-192): the probabilities are re-read from the mixed model
  void modelChanged() {
    probas_ = model_->getProbabilities();
    for (size_t k = 0; k < subs_.size(); ++k) subs_[k]->modelParametersChanged();
  }
  ParameterList getBranchLengthsParameters() const { return subs_.at(0)->getBranchLengthsParameters(); }
  size_t getNumberOfSites() const { return subs_.at(0)->getNumberOfSites(); }
  double getLikelihoodForASite(size_t site) const {
    double r = 0;
    for (size_t k = 0; k < subs_.size(); ++k) r += subs_[k]->getLikelihoodForASite(site) * probas_[k];
    return r;
  }
  double getLogLikelihoodForASite(size_t site) const {
    double x = getLikelihoodForASite(site);
    if (x < 0) x = 0;
    return std::log(x);
  }
  double getLikelihoodForASiteForARateClass(size_t site, size_t rateClass) const {
    double r = 0;
    for (size_t k = 0; k < subs_.size(); ++k) r += subs_[k]->getLikelihoodForASiteForARateClass(site, rateClass) * probas_[k];
    return r;
  }
  double getLogLikelihood() const {
    requireInit();
    const std::vector<unsigned int>& w = subs_[0]->getWeights();
    const size_t N = w.size(), K = subs_.size();
    std::vector<Vdouble> sl(K);
    for (size_t k = 0; k < K; ++k) sl[k] = subs_[k]->getLogLikelihoodForEachDistinctSite();
    Vdouble la(N);
    for (size_t i = 0; i < N; ++i) {
      // log sum_j p_j L_j,i through the largest term: the per-site likelihoods of large trees are far below 1e-308
      double m = -std::numeric_limits<double>::infinity();
      for (size_t k = 0; k < K; ++k) if (probas_[k] > 0) m = std::max(m, sl[k][i]);
      double x = 0;
      for (size_t k = 0; k < K; ++k) if (probas_[k] > 0) x += probas_[k] * std::exp(sl[k][i] - m);
      la[i] = w[i] * (std::isfinite(m) ? m + std::log(x) : m);
    }
    std::sort(la.begin(), la.end());
    double ll = 0;
    for (size_t i = N; i > 0; --i) ll += la[i - 1];
    return ll;
  }
  double getValue() const { return -getLogLikelihood(); }
  double getFirstOrderDerivative(const std::string& variable) const {
    const int b = branch(variable);
    const std::vector<unsigned int>& w = subs_[0]->getWeights();
    std::vector<Vdouble> dl(subs_.size());
    for (size_t k = 0; k < subs_.size(); ++k) dl[k] = subs_[k]->getDLikelihoodArray(b);
    double d = 0;
    for (size_t i = 0; i < w.size(); ++i) {
      double x = 0;
      for (size_t k = 0; k < subs_.size(); ++k) x += dl[k][i] * probas_[k];
      d += w[i] * x;
    }
    return -d;
  }
  double getSecondOrderDerivative(const std::string& variable) const {
    const int b = branch(variable);
    const std::vector<unsigned int>& w = subs_[0]->getWeights();
    std::vector<Vdouble> dl(subs_.size()), d2l(subs_.size());
    for (size_t k = 0; k < subs_.size(); ++k) { dl[k] = subs_[k]->getDLikelihoodArray(b); d2l[k] = subs_[k]->getD2LikelihoodArray(b); }
    double d = 0;
    for (size_t i = 0; i < w.size(); ++i) {
      double x = 0, x2 = 0;
      for (size_t k = 0; k < subs_.size(); ++k) { x += dl[k][i] * probas_[k]; x2 += d2l[k][i] * probas_[k]; }
      d += w[i] * (x2 - x * x);
    }
    return -d;
  }

 private:
  void requireInit() const { if (!initialized_) throw Exception("Instance is not initialized."); }
  int branch(const std::string& variable) const {
    requireInit();
    if (variable.compare(0, 5, "BrLen") != 0) {
      for (const std::string& n : model_->getParameterNames())
        if (n == variable) throw Exception("Derivatives respective to substitution model parameters are not implemented.");
      throw ParameterNotFoundException("ParameterNotFoundException: " + variable);
    }
    return std::atoi(variable.c_str() + 5);
  }
  MixedSubstitutionModel* model_;
  std::vector<std::unique_ptr<DRHomogeneousTreeLikelihood> > subs_;
  Vdouble probas_;
  bool initialized_ = false;
};

}  // namespace bppshim
