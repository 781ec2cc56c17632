// bppgpu shim (see ../bppgpu_shim.hpp): DistanceMatrix, DistanceEstimation, BioNJ (Distance/DistanceMatrix.h,
// Distance/DistanceEstimation.cpp, Distance/BioNJ.cpp, Distance/NeighborJoining.cpp): a starting tree from the alignment alone
#pragma once
#include "likelihood.hpp"

namespace bppshim {

// Distance/DistanceMatrix.h: a named square matrix
class DistanceMatrix {
 public:
  explicit DistanceMatrix(const std::vector<std::string>& names) : names_(names), d_(names.size() * names.size(), 0.0) {}
  size_t size() const { return names_.size(); }
  const std::vector<std::string>& getNames() const { return names_; }
  const std::string& getName(size_t i) const { return names_.at(i); }
  double& operator()(size_t i, size_t j) { return d_[i * names_.size() + j]; }
  double operator()(size_t i, size_t j) const { return d_[i * names_.size() + j]; }

 private:
  std::vector<std::string> names_;
  std::vector<double> d_;
};

// DistanceEstimation::computeMatrix: the ML distance of every pair of sequences (one TwoTreeLikelihood per pair, rooted at the
// first sequence, branch length bounded to [1e-6, 1e4]).  All pairs are computed on the device in one call
// (bppgpu_pairwise_distances): the pairs' joint code counts as one integer matrix product, then a Newton search per pair.
// The model and rate parameters are taken as they are (the reference's optional parameter estimation is not done).
class DistanceEstimation {
 public:
  DistanceEstimation(SubstitutionModel* model, DiscreteDistribution* rDist, const VectorSiteContainer* sites, size_t verbose = 1,
                     bool computeMat = true, int device = 0)
      : model_(model), rDist_(rDist), sites_(sites), verbose_(verbose), device_(device) {
    if (computeMat) computeMatrix();
  }
  void computeMatrix() {
    const std::vector<std::string> names = sites_->getSequencesNames();
    if (names.size() < 2 || sites_->getNumberOfSites() == 0)
      throw Exception("DistanceEstimation::computeMatrix. Need at least two sequences and one site.");
    const TipCodes tc = encodeTipCodes(*sites_, names, *model_);
    const size_t L = names.size(), N = tc.weights.size();
    std::vector<uint8_t> c8(tc.nCodes <= 256 ? L * N : 0);
    std::vector<uint16_t> c16(tc.nCodes > 256 ? L * N : 0);
    for (size_t t = 0; t < L; ++t)
      for (size_t k = 0; k < N; ++k) {
        if (c8.empty()) c16[t * N + k] = tc.codes[t][k];
        else c8[t * N + k] = (uint8_t)tc.codes[t][k];
      }
    bppgpu_model_desc d;
    model_->fillModelDesc(d);
    Vdouble r(rDist_->getNumberOfCategories()), p(r.size());
    for (size_t c = 0; c < r.size(); ++c) { r[c] = rDist_->getCategory(c); p[c] = rDist_->getProbability(c); }
    std::vector<double> dist(L * L);
    check(bppgpu_pairwise_distances(device_, &d, model_->getFrequencies().data(), (int32_t)r.size(), r.data(), p.data(),
                                    (int32_t)tc.nCodes, c8.empty() ? 2 : 1, tc.table.data(), (int32_t)L, (int64_t)N,
                                    c8.empty() ? (const void*)c16.data() : (const void*)c8.data(), tc.weights.data(), dist.data(),
                                    nullptr, nullptr),
          "DistanceEstimation::computeMatrix");
    matrix_.reset(new DistanceMatrix(names));
    for (size_t i = 0; i < L; ++i)
      for (size_t j = 0; j < L; ++j) (*matrix_)(i, j) = dist[i * L + j];
  }
  // a new copy, owned by the caller (DistanceEstimation::getMatrix)
  DistanceMatrix* getMatrix() const { return matrix_ ? new DistanceMatrix(*matrix_) : nullptr; }
  size_t getVerbose() const { return verbose_; }

 private:
  SubstitutionModel* model_;
  DiscreteDistribution* rDist_;
  const VectorSiteContainer* sites_;
  size_t verbose_;
  int device_;
  std::unique_ptr<DistanceMatrix> matrix_;
};

// BioNJ (Gascuel 1997) as Bio++ runs it (Distance/BioNJ.cpp on Distance/NeighborJoining.cpp): at each step the pair maximising
// S_i + S_j - (n - 2) D_ij joins (first pair in row-major order of the remaining nodes on ties), its branch lengths are
// D_ij / 2 +- (S_i - S_j) / (2 (n - 2)), and the new node's distances and variances are the lambda-weighted BIONJ reduction.
// The per-row sums and criterion maxima run on the host cores (parallel_for); each row writes its own slot and rows are
// combined in order, so the tree does not depend on the thread count.
class BioNJ {
 public:
  explicit BioNJ(const DistanceMatrix& matrix, bool rooted = false, bool positiveLengths = false, bool verbose = true)
      : matrix_(matrix), rooted_(rooted), positive_(positiveLengths), verbose_(verbose) {
    computeTree();
  }
  void computeTree() {
    const size_t n0 = matrix_.size();
    if (n0 < (rooted_ ? 2u : 3u)) throw Exception("BioNJ::computeTree. Too few sequences.");
    std::vector<double> D(n0 * n0), V(n0 * n0);
    for (size_t i = 0; i < n0; ++i)
      for (size_t j = 0; j < n0; ++j) D[i * n0 + j] = V[i * n0 + j] = matrix_(i, j);
    std::vector<Node*> node(n0);
    for (size_t i = 0; i < n0; ++i) { node[i] = new Node(); node[i]->setName(matrix_.getName(i)); }
    std::vector<size_t> active(n0);
    for (size_t i = 0; i < n0; ++i) active[i] = i;
    auto clamp = [&](double x) { return positive_ ? std::max(x, 0.0) : x; };
    std::vector<double> S, rowBest;
    std::vector<size_t> rowArg;
    while (active.size() > (rooted_ ? 2u : 3u)) {
      const size_t m = active.size();
      S.assign(m, 0.0);
      linalg::parallel_for((int)m, 64, [&](int a) {
        double s = 0;
        for (size_t b = 0; b < m; ++b) s += D[active[(size_t)a] * n0 + active[b]];
        S[(size_t)a] = s;
      });
      rowBest.assign(m, -std::numeric_limits<double>::infinity());
      rowArg.assign(m, m);
      linalg::parallel_for((int)m, 64, [&](int a) {
        const double* Da = &D[active[(size_t)a] * n0];
        for (size_t b = (size_t)a + 1; b < m; ++b) {
          const double crit = S[(size_t)a] + S[b] - (double)(m - 2) * Da[active[b]];
          if (crit > rowBest[(size_t)a]) { rowBest[(size_t)a] = crit; rowArg[(size_t)a] = b; }
        }
      });
      size_t ba = 0;
      for (size_t a = 1; a + 1 < m; ++a)
        if (rowBest[a] > rowBest[ba]) ba = a;
      if (rowArg[ba] == m) {
        for (size_t x : active) delete node[x];
        throw Exception("BioNJ::computeTree. No pair has a finite criterion (NaN or infinite distances).");
      }
      const size_t bb = rowArg[ba], i = active[ba], j = active[bb];
      const double ratio = (S[ba] - S[bb]) / (double)(m - 2);
      const double di = clamp(0.5 * (D[i * n0 + j] + ratio)), dj = clamp(0.5 * (D[i * n0 + j] - ratio));
      double lambda = 0.5;
      if (V[i * n0 + j] != 0) {
        lambda = 0;
        for (size_t x : active)
          if (x != i && x != j) lambda += V[j * n0 + x] - V[i * n0 + x];
        lambda = lambda / (2.0 * (double)(m - 2) * V[i * n0 + j]) + 0.5;
      }
      lambda = std::min(std::max(lambda, 0.0), 1.0);
      Node* parent = new Node();
      node[i]->setDistanceToFather(di);
      node[j]->setDistanceToFather(dj);
      parent->addSon(node[i]);
      parent->addSon(node[j]);
      for (size_t x : active) {
        if (x == i || x == j) continue;
        const double dn = clamp(lambda * (D[i * n0 + x] - di) + (1 - lambda) * (D[j * n0 + x] - dj));
        const double vn = lambda * V[i * n0 + x] + (1 - lambda) * V[j * n0 + x] - lambda * (1 - lambda) * V[i * n0 + j];
        D[i * n0 + x] = D[x * n0 + i] = dn;
        V[i * n0 + x] = V[x * n0 + i] = vn;
      }
      node[i] = parent;
      node[j] = nullptr;
      active.erase(active.begin() + (std::ptrdiff_t)bb);
    }
    // NeighborJoining::finalStep
    Node* root = new Node();
    if (rooted_) {
      const size_t i = active[0], j = active[1];
      for (size_t x : active) { node[x]->setDistanceToFather(D[i * n0 + j] / 2); root->addSon(node[x]); }
    } else {
      const size_t i = active[0], j = active[1], k = active[2];
      node[i]->setDistanceToFather(clamp(D[i * n0 + j] + D[i * n0 + k] - D[j * n0 + k]) / 2);
      node[j]->setDistanceToFather(clamp(D[j * n0 + i] + D[j * n0 + k] - D[i * n0 + k]) / 2);
      node[k]->setDistanceToFather(clamp(D[k * n0 + i] + D[k * n0 + j] - D[i * n0 + j]) / 2);
      for (size_t x : active) root->addSon(node[x]);
    }
    tree_.reset(new TreeTemplate<Node>(root));
  }
  // a new copy, owned by the caller (AbstractAgglomerativeDistanceMethod::getTree)
  TreeTemplate<Node>* getTree() const { return new TreeTemplate<Node>(*tree_); }

 private:
  DistanceMatrix matrix_;
  bool rooted_, positive_, verbose_;
  std::unique_ptr<TreeTemplate<Node> > tree_;
};

}  // namespace bppshim
