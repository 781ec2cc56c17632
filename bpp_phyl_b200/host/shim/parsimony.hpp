// bppgpu shim (see ../bppgpu_shim.hpp): DRTreeParsimonyScore (Parsimony/DRTreeParsimonyScore.cpp) and
// OptimizationTools::optimizeTreeNNI for it: Fitch parsimony and an NNI search, every score and every NNI's change of score
// computed on the device (bppgpu_parsimony_*)
#pragma once
#include <cstdio>
#include <set>

#include "likelihood.hpp"

namespace bppshim {

// DRTreeParsimonyScore: Fitch's rule on bitsets over the site patterns.  A rooted tree is unrooted first.  A tip's set is the
// alphabet's resolved states of its character; with includeGaps, '-' is a state of its own (bit alphabet size).  Alphabets of
// more than 32 states (codons, chromosome counts) are refused.  The tip sets stay on the device; each score or NNI query sends
// the current topology.  Node ids persist across doNNI, as in the reference.
class DRTreeParsimonyScore {
 public:
  DRTreeParsimonyScore(const Tree& tree, const VectorSiteContainer& data, bool verbose = true, bool includeGaps = false,
                       int device = 0)
      : tree_(new Tree(tree)), verbose_(verbose) {
    if (tree_->isRooted()) tree_->unroot();
    const std::vector<std::string> names = tree_->getLeavesNames();
    const Alphabet* a = data.getAlphabet();
    const size_t S = a->getSize() + (includeGaps ? 1 : 0);
    const TipCodes tc = encodeTipCodes(data, names, S, [a, includeGaps](size_t s, const std::string& ch) {
      if (includeGaps && ch == "-") return s == a->getSize() ? 1.0 : 0.0;
      for (int x : a->getAlias(ch))
        if ((size_t)x == s) return 1.0;
      return 0.0;
    });
    siteIndex_ = tc.siteIndex;
    const size_t L = names.size(), N = tc.weights.size();
    nPatterns_ = N;
    std::vector<uint8_t> c8(tc.nCodes <= 256 ? L * N : 0);
    std::vector<uint16_t> c16(tc.nCodes > 256 ? L * N : 0);
    for (size_t t = 0; t < L; ++t) {
      rowOf_[names[t]] = (int)t;
      for (size_t k = 0; k < N; ++k) {
        if (c8.empty()) c16[t * N + k] = tc.codes[t][k];
        else c8[t * N + k] = (uint8_t)tc.codes[t][k];
      }
    }
    check(bppgpu_parsimony_create(device, (int32_t)S, (int32_t)tc.nCodes, c8.empty() ? 2 : 1, tc.table.data(), (int32_t)L,
                                  (int64_t)N, c8.empty() ? (const void*)c16.data() : (const void*)c8.data(), tc.weights.data(),
                                  0, &handle_),
          "DRTreeParsimonyScore");
  }
  ~DRTreeParsimonyScore() { bppgpu_parsimony_destroy(handle_); }
  DRTreeParsimonyScore(const DRTreeParsimonyScore&) = delete;
  DRTreeParsimonyScore& operator=(const DRTreeParsimonyScore&) = delete;

  const Tree& getTree() const { return *tree_; }
  // weighted over the site patterns = summed over the sites
  int64_t getScore() const { update_(); return score_; }
  unsigned int getScoreForSite(size_t site) const {
    update_();
    if (site >= siteIndex_.size()) throw Exception("IndexOutOfBoundsException: DRTreeParsimonyScore::getScoreForSite");
    return siteScores_[(size_t)siteIndex_[site]];
  }
  std::vector<unsigned int> getScoreForEachSite() const {
    update_();
    std::vector<unsigned int> v(siteIndex_.size());
    for (size_t i = 0; i < v.size(); ++i) v[i] = siteScores_[(size_t)siteIndex_[i]];
    return v;
  }
  double getTopologyValue() const { return (double)getScore(); }

  // NNISearchable::testNNI: score after the NNI of nodeId minus the current score (all NNIs come from one device call, cached
  // until the next doNNI)
  double testNNI(int nodeId) const {
    requireNni_(tree_->getNode(nodeId));
    if (!nniValid_) {
      Flat fl = flatten_();
      std::vector<int64_t> d(fl.nodes.size());
      check(bppgpu_parsimony_nni(handle_, (int32_t)fl.nodes.size(), fl.root, fl.off.data(), fl.ch.data(), fl.leafRow.data(), d.data(),
                                 nullptr),
            "DRTreeParsimonyScore::testNNI");
      delta_.clear();
      for (size_t i = 0; i < fl.nodes.size(); ++i) delta_[fl.nodes[i]->getId()] = d[i];
      nniValid_ = true;
    }
    return (double)delta_.at(nodeId);
  }
  // NNISearchable::doNNI: node and its uncle g.son(pos > 1 ? 0 : 1 - pos) change places (each appended to its new father's sons)
  void doNNI(int nodeId) {
    Node* v = tree_->getNode(nodeId);
    requireNni_(v);
    Node* f = v->getFather();
    Node* g = f->getFather();
    std::vector<Node*>& gs = g->sons();
    const size_t pos = (size_t)(std::find(gs.begin(), gs.end(), f) - gs.begin());
    Node* u = g->getSon(pos > 1 ? 0 : 1 - pos);
    std::vector<Node*>& fs = f->sons();
    fs.erase(std::find(fs.begin(), fs.end(), v));
    gs.erase(std::find(gs.begin(), gs.end(), u));
    f->addSon(u);
    g->addSon(v);
    scoreValid_ = nniValid_ = false;
  }
  // the NNI search restores a tree it rejected (node ids included)
  void setTopology(const Tree& t) {
    *tree_ = t;
    scoreValid_ = nniValid_ = false;
  }
  bool isVerbose() const { return verbose_; }

 private:
  struct Flat {
    std::vector<Node*> nodes;
    std::vector<int32_t> off, ch, leafRow;
    int32_t root;
  };
  // flattened ids are post-order positions of this call
  Flat flatten_() const {
    Flat fl;
    fl.nodes = tree_->getNodes();
    std::map<const Node*, int32_t> idx;
    for (size_t i = 0; i < fl.nodes.size(); ++i) idx[fl.nodes[i]] = (int32_t)i;
    fl.off.assign(1, 0);
    for (Node* n : fl.nodes) {
      for (size_t s = 0; s < n->getNumberOfSons(); ++s) fl.ch.push_back(idx[n->getSon(s)]);
      fl.off.push_back((int32_t)fl.ch.size());
      fl.leafRow.push_back(n->isLeaf() ? rowOf_.at(n->getName()) : -1);
    }
    fl.root = (int32_t)fl.nodes.size() - 1;
    return fl;
  }
  void update_() const {
    if (scoreValid_) return;
    Flat fl = flatten_();
    siteScores_.resize(nPatterns_);
    check(bppgpu_parsimony_score(handle_, (int32_t)fl.nodes.size(), fl.root, fl.off.data(), fl.ch.data(), fl.leafRow.data(), &score_,
                                 siteScores_.data()),
          "DRTreeParsimonyScore::computeScores");
    scoreValid_ = true;
  }
  static void requireNni_(const Node* v) {
    if (!v->hasFather() || !v->getFather()->hasFather())
      throw Exception("NodeException: DRTreeParsimonyScore: no NNI around a node whose father is the root (or around the root).");
  }

  std::unique_ptr<Tree> tree_;
  bool verbose_;
  bppgpu_parsimony* handle_ = nullptr;
  std::vector<int64_t> siteIndex_;
  size_t nPatterns_ = 0;
  std::map<std::string, int> rowOf_;
  mutable bool scoreValid_ = false, nniValid_ = false;
  mutable int64_t score_ = 0;
  mutable std::vector<uint32_t> siteScores_;
  mutable std::map<int, int64_t> delta_;
};

namespace OptimizationTools {
// optimizeTreeNNI for a parsimony score (OptimizationTools::optimizeTreeNNI(TreeParsimonyScore*) with NNITopologySearch), by
// the rule of DESIGN §7b: every NNI is scored in one device call; the improving ones are sorted by (change, post-order
// position) and taken greedily unless their {node, father, grandfather} meets one already taken; the k taken are applied in
// that order and the tree rescored; a round that does not lower the score is undone and retried with the first k / 2.  Stops
// at a tree no single NNI improves.  `scores` (may be null) receives the score before the first round and after each round.
inline DRTreeParsimonyScore* optimizeTreeNNI(DRTreeParsimonyScore* tp, unsigned int verbose = 1, std::vector<int64_t>* scores = nullptr) {
  int64_t cur = tp->getScore();
  if (scores) scores->assign(1, cur);
  for (int round = 1;; ++round) {
    const std::vector<Node*> nodes = tp->getTree().getNodes();
    std::vector<std::pair<double, size_t> > cand;   // (change, post-order position)
    for (size_t i = 0; i < nodes.size(); ++i) {
      const Node* v = nodes[i];
      if (!v->hasFather() || !v->getFather()->hasFather()) continue;
      const double d = tp->testNNI(v->getId());
      if (d < 0) cand.push_back(std::make_pair(d, i));
    }
    if (cand.empty()) break;
    std::sort(cand.begin(), cand.end());
    std::vector<int> taken;
    std::set<int> used;
    for (const auto& c : cand) {
      const Node* v = nodes[c.second];
      const int tri[3] = {v->getId(), v->getFather()->getId(), v->getFather()->getFather()->getId()};
      if (used.count(tri[0]) || used.count(tri[1]) || used.count(tri[2])) continue;
      used.insert(tri, tri + 3);
      taken.push_back(tri[0]);
    }
    const Tree before = tp->getTree();
    for (size_t k = taken.size();; k /= 2) {
      for (size_t j = 0; j < k; ++j) tp->doNNI(taken[j]);
      const int64_t s = tp->getScore();
      if (s < cur) {
        if (verbose) std::printf("optimizeTreeNNI: round %d, %zu NNIs, score %lld\n", round, k, (long long)s);
        cur = s;
        break;
      }
      if (k == 1) throw Exception("optimizeTreeNNI: a single improving NNI did not lower the score");
      tp->setTopology(before);
    }
    if (scores) scores->push_back(cur);
  }
  return tp;
}
}  // namespace OptimizationTools

}  // namespace bppshim
