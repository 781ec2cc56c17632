// bppgpu shim (see ../bppgpu_shim.hpp): DRTreeParsimonyScore (Parsimony/DRTreeParsimonyScore.cpp) and
// OptimizationTools::optimizeTreeNNI for it: Fitch parsimony and an NNI search, every score and every NNI's change of score
// computed on the device (bppgpu_parsimony_*); DRTreeParsimonyBootstrap and the lockstep search of its replicates (bppPars)
#pragma once
#include <cstdio>
#include <set>

#include "likelihood.hpp"

namespace bppshim {

// DRTreeParsimonyScore: Fitch's rule on bitsets over the site patterns.  A rooted tree is unrooted first.  A tip's set is the
// alphabet's resolved states of its character; with includeGaps, '-' is a state of its own (bit alphabet size).  Alphabets of
// more than 32 states (codons, chromosome counts) are refused.  The tip sets stay on the device; each score or NNI query sends
// the current topology.  Node ids persist across doNNI, as in the reference.
namespace parsimony_detail {
// DRTreeParsimonyScore's tip sets: `data` encoded for the leaves `names` (rows in that order) as the constructor does, the
// handle created with the pattern weights
inline bppgpu_parsimony* create(const VectorSiteContainer& data, const std::vector<std::string>& names, bool includeGaps, int device,
                                std::vector<int64_t>& siteIndex, std::map<std::string, int>& rowOf, size_t& nPatterns, const char* who) {
  const Alphabet* a = data.getAlphabet();
  const size_t S = a->getSize() + (includeGaps ? 1 : 0);
  const TipCodes tc = encodeTipCodes(data, names, S, [a, includeGaps](size_t s, const std::string& ch) {
    if (includeGaps && ch == "-") return s == a->getSize() ? 1.0 : 0.0;
    for (int x : a->getAlias(ch))
      if ((size_t)x == s) return 1.0;
    return 0.0;
  });
  siteIndex = tc.siteIndex;
  const size_t L = names.size(), N = tc.weights.size();
  nPatterns = N;
  std::vector<uint8_t> c8(tc.nCodes <= 256 ? L * N : 0);
  std::vector<uint16_t> c16(tc.nCodes > 256 ? L * N : 0);
  for (size_t t = 0; t < L; ++t) {
    rowOf[names[t]] = (int)t;
    for (size_t k = 0; k < N; ++k) {
      if (c8.empty()) c16[t * N + k] = tc.codes[t][k];
      else c8[t * N + k] = (uint8_t)tc.codes[t][k];
    }
  }
  bppgpu_parsimony* h = nullptr;
  check(bppgpu_parsimony_create(device, (int32_t)S, (int32_t)tc.nCodes, c8.empty() ? 2 : 1, tc.table.data(), (int32_t)L, (int64_t)N,
                                c8.empty() ? (const void*)c16.data() : (const void*)c8.data(), tc.weights.data(), 0, &h),
        who);
  return h;
}

// a topology as the C ABI takes it; flattened ids are post-order positions (Tree::getNodes order), the root last
struct Flat {
  std::vector<Node*> nodes;
  std::vector<int32_t> off, ch, leafRow;
  int32_t root;
};
inline Flat flatten(const Tree& tree, const std::map<std::string, int>& rowOf) {
  Flat fl;
  fl.nodes = tree.getNodes();
  std::map<const Node*, int32_t> idx;
  for (size_t i = 0; i < fl.nodes.size(); ++i) idx[fl.nodes[i]] = (int32_t)i;
  fl.off.assign(1, 0);
  for (Node* n : fl.nodes) {
    for (size_t s = 0; s < n->getNumberOfSons(); ++s) fl.ch.push_back(idx[n->getSon(s)]);
    fl.off.push_back((int32_t)fl.ch.size());
    fl.leafRow.push_back(n->isLeaf() ? rowOf.at(n->getName()) : -1);
  }
  fl.root = (int32_t)fl.nodes.size() - 1;
  return fl;
}

inline bool hasNNI(const Node* v) { return v->hasFather() && v->getFather()->hasFather(); }

// NNISearchable::doNNI: node and its uncle g.son(pos > 1 ? 0 : 1 - pos) change places (each appended to its new father's sons)
inline void doNNI(Tree& tree, int nodeId) {
  Node* v = tree.getNode(nodeId);
  if (!hasNNI(v))
    throw Exception("NodeException: DRTreeParsimonyScore: no NNI around a node whose father is the root (or around the root).");
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
}

// the improving NNIs of one round (DESIGN §7b): (change, post-order position) sorted, taken greedily unless their
// {node, father, grandfather} meets one already taken; returns the node ids in the order they are applied
inline std::vector<int> takeNNIs(const std::vector<Node*>& nodes, const std::vector<std::pair<double, size_t> >& improving) {
  std::vector<std::pair<double, size_t> > cand = improving;
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
  return taken;
}
}  // namespace parsimony_detail

class DRTreeParsimonyScore {
 public:
  DRTreeParsimonyScore(const Tree& tree, const VectorSiteContainer& data, bool verbose = true, bool includeGaps = false,
                       int device = 0)
      : tree_(new Tree(tree)), verbose_(verbose) {
    if (tree_->isRooted()) tree_->unroot();
    handle_ = parsimony_detail::create(data, tree_->getLeavesNames(), includeGaps, device, siteIndex_, rowOf_, nPatterns_,
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
    parsimony_detail::doNNI(*tree_, nodeId);
    scoreValid_ = nniValid_ = false;
  }
  // the NNI search restores a tree it rejected (node ids included)
  void setTopology(const Tree& t) {
    *tree_ = t;
    scoreValid_ = nniValid_ = false;
  }
  bool isVerbose() const { return verbose_; }

 private:
  typedef parsimony_detail::Flat Flat;
  Flat flatten_() const { return parsimony_detail::flatten(*tree_, rowOf_); }
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
    if (!parsimony_detail::hasNNI(v))
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

// DRTreeParsimonyBootstrap: bppPars's bootstrap.  The data are encoded as by DRTreeParsimonyScore (same tip codes, unrooting
// and gap rule); the weights of replicates 0 .. nbReplicates - 1 are drawn on the device from the site -> pattern indices
// (bppgpu_bootstrap_weights' sampler under `seed`) and stay there.  One tree per replicate, each starting from `start`; every
// score and NNI change of a batch of replicate trees comes from one device call (bppgpu_parsimony_*_replicates).
class DRTreeParsimonyBootstrap {
 public:
  DRTreeParsimonyBootstrap(const Tree& start, const VectorSiteContainer& data, unsigned int nbReplicates, uint64_t seed,
                           bool includeGaps = false, int device = 0)
      : seed_(seed), device_(device) {
    if (nbReplicates < 1) throw Exception("DRTreeParsimonyBootstrap: at least one replicate is needed");
    Tree t(start);
    if (t.isRooted()) t.unroot();
    handle_ = parsimony_detail::create(data, t.getLeavesNames(), includeGaps, device, siteIndex_, rowOf_, nPatterns_,
                                       "DRTreeParsimonyBootstrap");
    try {
      check(bppgpu_parsimony_draw_replicate_weights(handle_, (int64_t)siteIndex_.size(), siteIndex_.data(), 0, (int32_t)nbReplicates, seed),
            "DRTreeParsimonyBootstrap");
      check(bppgpu_parsimony_last_ms(handle_, &samplerMs_), "DRTreeParsimonyBootstrap");
    } catch (...) {
      bppgpu_parsimony_destroy(handle_);
      throw;
    }
    for (unsigned int r = 0; r < nbReplicates; ++r) trees_.emplace_back(new Tree(t));
    scores_.assign(nbReplicates, 0);
  }
  ~DRTreeParsimonyBootstrap() { bppgpu_parsimony_destroy(handle_); }
  DRTreeParsimonyBootstrap(const DRTreeParsimonyBootstrap&) = delete;
  DRTreeParsimonyBootstrap& operator=(const DRTreeParsimonyBootstrap&) = delete;

  size_t getNumberOfReplicates() const { return trees_.size(); }
  size_t getNumberOfPatterns() const { return nPatterns_; }
  const Tree& getTree(size_t r) const { return *trees_.at(r); }
  std::vector<Tree*> getTrees() const {
    std::vector<Tree*> v;
    for (const auto& t : trees_) v.push_back(t.get());
    return v;
  }
  // replicate r's score on its current tree (one batched call for all replicates, cached until a tree changes)
  int64_t getScore(size_t r) const {
    if (r >= trees_.size()) throw Exception("IndexOutOfBoundsException: DRTreeParsimonyBootstrap::getScore");
    if (!scoresValid_) {
      std::vector<size_t> all(trees_.size());
      std::vector<const Tree*> ts;
      for (size_t i = 0; i < all.size(); ++i) { all[i] = i; ts.push_back(trees_[i].get()); }
      scores_ = scoreTrees(all, ts);
      scoresValid_ = true;
    }
    return scores_[r];
  }
  // replicate r's pattern weights, drawn again on the device (a replicate depends only on the seed and its index)
  std::vector<unsigned int> getWeights(size_t r) const {
    if (r >= trees_.size()) throw Exception("IndexOutOfBoundsException: DRTreeParsimonyBootstrap::getWeights");
    std::vector<unsigned int> w(nPatterns_);
    check(bppgpu_bootstrap_weights(device_, (int64_t)siteIndex_.size(), siteIndex_.data(), (int64_t)nPatterns_, (int64_t)r, 1, seed_, w.data()),
          "DRTreeParsimonyBootstrap::getWeights");
    return w;
  }
  void setTree(size_t r, const Tree& t) {
    *trees_.at(r) = t;
    scoresValid_ = false;
  }

  // one device call: the score of trees[e] under replicate reps[e]'s weights
  std::vector<int64_t> scoreTrees(const std::vector<size_t>& reps, const std::vector<const Tree*>& trees) const {
    Batch b = batch_(reps, trees);
    std::vector<int64_t> s(reps.size());
    check(bppgpu_parsimony_score_replicates(handle_, (int32_t)reps.size(), b.rep.data(), b.nNodes, b.root, b.off.data(), b.ch.data(),
                                            b.leafRow.data(), s.data(), nullptr),
          "DRTreeParsimonyBootstrap::scoreTrees");
    account_();
    return s;
  }
  // one device call: every NNI change of trees[e] under replicate reps[e]'s weights, [e][post-order position]
  std::vector<std::vector<int64_t> > nniTrees(const std::vector<size_t>& reps, const std::vector<const Tree*>& trees) const {
    Batch b = batch_(reps, trees);
    std::vector<int64_t> d(reps.size() * (size_t)b.nNodes), s(reps.size());
    check(bppgpu_parsimony_nni_replicates(handle_, (int32_t)reps.size(), b.rep.data(), b.nNodes, b.root, b.off.data(), b.ch.data(),
                                          b.leafRow.data(), d.data(), s.data()),
          "DRTreeParsimonyBootstrap::nniTrees");
    account_();
    std::vector<std::vector<int64_t> > out(reps.size());
    for (size_t e = 0; e < reps.size(); ++e) out[e].assign(d.begin() + e * b.nNodes, d.begin() + (e + 1) * b.nNodes);
    return out;
  }
  // device time of the sampler, and of the batched calls so far with their number
  double getSamplerMs() const { return samplerMs_; }
  double getDeviceMs() const { return deviceMs_; }
  size_t getNumberOfCalls() const { return calls_; }

 private:
  struct Batch {
    std::vector<int32_t> rep, off, ch, leafRow;
    int32_t nNodes = 0, root = 0;
  };
  Batch batch_(const std::vector<size_t>& reps, const std::vector<const Tree*>& trees) const {
    if (reps.empty() || reps.size() != trees.size()) throw Exception("DRTreeParsimonyBootstrap: bad batch");
    Batch b;
    for (size_t e = 0; e < reps.size(); ++e) {
      const parsimony_detail::Flat fl = parsimony_detail::flatten(*trees[e], rowOf_);
      if (e == 0) { b.nNodes = (int32_t)fl.nodes.size(); b.root = fl.root; }
      if ((int32_t)fl.nodes.size() != b.nNodes) throw Exception("DRTreeParsimonyBootstrap: the trees of a batch differ in size");
      b.rep.push_back((int32_t)reps[e]);
      b.off.insert(b.off.end(), fl.off.begin(), fl.off.end());
      b.ch.insert(b.ch.end(), fl.ch.begin(), fl.ch.end());
      b.leafRow.insert(b.leafRow.end(), fl.leafRow.begin(), fl.leafRow.end());
    }
    return b;
  }
  void account_() const {
    double ms = 0;
    check(bppgpu_parsimony_last_ms(handle_, &ms), "DRTreeParsimonyBootstrap");
    deviceMs_ += ms;
    ++calls_;
  }

  uint64_t seed_;
  int device_;
  bppgpu_parsimony* handle_ = nullptr;
  std::vector<int64_t> siteIndex_;
  size_t nPatterns_ = 0;
  std::map<std::string, int> rowOf_;
  std::vector<std::unique_ptr<Tree> > trees_;
  mutable bool scoresValid_ = false;
  mutable std::vector<int64_t> scores_;
  double samplerMs_ = 0;
  mutable double deviceMs_ = 0;
  mutable size_t calls_ = 0;
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
    const std::vector<int> taken = parsimony_detail::takeNNIs(nodes, cand);
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

// optimizeTreeNNI for every replicate of a bootstrap, by the rule of DESIGN §7b applied to each replicate, in lockstep: each
// round is one nniTrees call over the replicates still active; each trial step is one scoreTrees call over the replicates
// whose trial is pending (a replicate whose trial did not lower its score retries with the first k / 2 in the next call).  A
// replicate retires at a tree no single NNI improves.  `scores` (may be null): scores[r] = replicate r's score before the
// first round and after each of its accepted rounds, as the single-replicate search with r's weights gives them.
// `replicates` (may be null: all) names the replicates to search; one of them alone is the single-replicate search, every
// call a batch of one.
inline DRTreeParsimonyBootstrap* optimizeTreeNNI(DRTreeParsimonyBootstrap* tb, unsigned int verbose = 1,
                                                 std::vector<std::vector<int64_t> >* scores = nullptr,
                                                 const std::vector<size_t>* replicates = nullptr) {
  const size_t R = tb->getNumberOfReplicates();
  std::vector<size_t> active;
  if (replicates) {
    active = *replicates;
    std::sort(active.begin(), active.end());
    active.erase(std::unique(active.begin(), active.end()), active.end());
    if (active.empty() || active.back() >= R) throw Exception("optimizeTreeNNI: bad replicate list");
  } else {
    for (size_t r = 0; r < R; ++r) active.push_back(r);
  }
  std::vector<const Tree*> trees;
  for (size_t r : active) trees.push_back(&tb->getTree(r));
  std::vector<int64_t> cur(R, 0);
  const std::vector<int64_t> first = tb->scoreTrees(active, trees);
  for (size_t e = 0; e < active.size(); ++e) cur[active[e]] = first[e];
  if (scores) {
    scores->assign(R, std::vector<int64_t>());
    for (size_t r : active) (*scores)[r].push_back(cur[r]);
  }
  struct Trial {
    size_t r;
    std::vector<int> taken;
    size_t k;
  };
  for (int round = 1; !active.empty(); ++round) {
    trees.clear();
    for (size_t r : active) trees.push_back(&tb->getTree(r));
    const std::vector<std::vector<int64_t> > delta = tb->nniTrees(active, trees);
    std::vector<Trial> pending;
    for (size_t e = 0; e < active.size(); ++e) {
      const std::vector<Node*> nodes = tb->getTree(active[e]).getNodes();
      std::vector<std::pair<double, size_t> > cand;   // (change, post-order position)
      for (size_t i = 0; i < nodes.size(); ++i)
        if (parsimony_detail::hasNNI(nodes[i]) && delta[e][i] < 0) cand.push_back(std::make_pair((double)delta[e][i], i));
      if (cand.empty()) continue;   // retires
      Trial t{active[e], parsimony_detail::takeNNIs(nodes, cand), 0};
      t.k = t.taken.size();
      pending.push_back(t);
    }
    std::vector<size_t> next;
    size_t accepted = 0;
    while (!pending.empty()) {
      std::vector<std::unique_ptr<Tree> > trial;
      std::vector<size_t> reps;
      trees.clear();
      for (const Trial& t : pending) {
        trial.emplace_back(new Tree(tb->getTree(t.r)));
        for (size_t j = 0; j < t.k; ++j) parsimony_detail::doNNI(*trial.back(), t.taken[j]);
        reps.push_back(t.r);
        trees.push_back(trial.back().get());
      }
      const std::vector<int64_t> s = tb->scoreTrees(reps, trees);
      std::vector<Trial> retry;
      for (size_t e = 0; e < pending.size(); ++e) {
        Trial& t = pending[e];
        if (s[e] < cur[t.r]) {
          tb->setTree(t.r, *trial[e]);
          cur[t.r] = s[e];
          if (scores) (*scores)[t.r].push_back(s[e]);
          next.push_back(t.r);
          ++accepted;
        } else {
          if (t.k == 1) throw Exception("optimizeTreeNNI: a single improving NNI did not lower the score");
          t.k /= 2;
          retry.push_back(t);
        }
      }
      pending.swap(retry);
    }
    std::sort(next.begin(), next.end());
    if (verbose) std::printf("optimizeTreeNNI (bootstrap): round %d, %zu of %zu replicates improved\n", round, accepted, active.size());
    active.swap(next);
  }
  return tb;
}
}  // namespace OptimizationTools

}  // namespace bppshim
