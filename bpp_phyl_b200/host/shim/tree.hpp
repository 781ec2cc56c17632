// bppgpu shim (see ../bppgpu_shim.hpp): Node, TreeTemplate, TreeTemplateTools (TreeTemplate.h, TreeTemplateTools.h), and
// BipartitionList / TreeTools::computeBootstrapValues (BipartitionList.h, TreeTools.h)
#pragma once
#include <cstdio>
#include <set>

#include "seq.hpp"

namespace bppshim {

// ---- trees (TreeTemplate.h, TreeTemplateTools.h) ---------------------------------------------------------------------
class Node {
 public:
  Node() : id_(-1), father_(nullptr), hasLen_(false), len_(0) {}
  ~Node() { for (Node* s : sons_) delete s; }
  int getId() const { return id_; }
  void setId(int i) { id_ = i; }
  bool isLeaf() const { return sons_.empty(); }
  bool hasFather() const { return father_ != nullptr; }
  Node* getFather() const { return father_; }
  size_t getNumberOfSons() const { return sons_.size(); }
  Node* getSon(size_t i) const { return sons_[i]; }
  void addSon(Node* s) { sons_.push_back(s); s->father_ = this; }
  bool hasDistanceToFather() const { return hasLen_; }
  double getDistanceToFather() const { return len_; }
  void setDistanceToFather(double d) { len_ = d; hasLen_ = true; }
  void deleteDistanceToFather() { hasLen_ = false; len_ = 0; }
  bool hasName() const { return !name_.empty(); }
  const std::string& getName() const { return name_; }
  void setName(const std::string& n) { name_ = n; }
  void removeFather() { father_ = nullptr; }
  std::vector<Node*>& sons() { return sons_; }
  // branch properties (the reference stores Clonable objects; here a number, e.g. TreeTools::BOOTSTRAP)
  void setBranchProperty(const std::string& name, double v) { branchProps_[name] = v; }
  bool hasBranchProperty(const std::string& name) const { return branchProps_.count(name) > 0; }
  double getBranchProperty(const std::string& name) const {
    auto it = branchProps_.find(name);
    if (it == branchProps_.end()) throw Exception("PropertyNotFoundException: Node::getBranchProperty: " + name);
    return it->second;
  }
  Node* cloneSubtree() const {
    Node* n = new Node();
    n->id_ = id_; n->hasLen_ = hasLen_; n->len_ = len_; n->name_ = name_; n->branchProps_ = branchProps_;
    for (Node* s : sons_) n->addSon(s->cloneSubtree());
    return n;
  }

 private:
  int id_;
  Node* father_;
  std::vector<Node*> sons_;
  bool hasLen_;
  double len_;
  std::string name_;
  std::map<std::string, double> branchProps_;
};

namespace TreeTemplateTools {
// post-order, root last (TreeTemplateTools.h:354-361)
inline void getNodes(Node* n, std::vector<Node*>& out) {
  for (size_t i = 0; i < n->getNumberOfSons(); ++i) getNodes(n->getSon(i), out);
  out.push_back(n);
}
// pre-order leaves (TreeTemplateTools.h:96-106)
inline void getLeaves(Node* n, std::vector<Node*>& out) {
  if (n->isLeaf()) out.push_back(n);
  for (size_t i = 0; i < n->getNumberOfSons(); ++i) getLeaves(n->getSon(i), out);
}
}  // namespace TreeTemplateTools

template <class N = Node>
class TreeTemplate {
 public:
  explicit TreeTemplate(N* root) : root_(root) { resetNodesId(); }
  TreeTemplate(const TreeTemplate& t) : root_(t.root_->cloneSubtree()) {}
  TreeTemplate& operator=(const TreeTemplate& t) { if (this != &t) { delete root_; root_ = t.root_->cloneSubtree(); } return *this; }
  ~TreeTemplate() { delete root_; }
  N* getRootNode() const { return root_; }
  bool isRooted() const { return root_->getNumberOfSons() == 2; }
  std::vector<N*> getNodes() const { std::vector<N*> v; TreeTemplateTools::getNodes(root_, v); return v; }
  std::vector<N*> getLeaves() const { std::vector<N*> v; TreeTemplateTools::getLeaves(root_, v); return v; }
  std::vector<std::string> getLeavesNames() const {
    std::vector<std::string> n;
    for (N* l : getLeaves()) n.push_back(l->getName());
    return n;
  }
  std::vector<int> getNodesId() const { std::vector<int> v; for (N* n : getNodes()) v.push_back(n->getId()); return v; }
  N* getNode(int id) const { for (N* n : getNodes()) if (n->getId() == id) return n; throw Exception("NodeNotFoundException: TreeTemplate::getNode(): Node with id not found."); }
  int getFatherId(int id) const { return getNode(id)->getFather()->getId(); }
  void resetNodesId() { int i = 0; for (N* n : getNodes()) n->setId(i++); }
  // TreeTemplate::unroot (TreeTemplate.h:244-284): keep son 0 as the new root, hang son 1 under it, sum the lengths
  bool unroot() {
    if (!isRooted()) throw Exception("UnrootedTreeException: Tree::unroot. Tree is already rooted.");
    N* s1 = root_->getSon(0);
    N* s2 = root_->getSon(1);
    if (s1->isLeaf() && s2->isLeaf()) return false;
    if (s1->isLeaf()) std::swap(s1, s2);
    if (s1->hasDistanceToFather()) {
      s2->setDistanceToFather(s2->hasDistanceToFather() ? s1->getDistanceToFather() + s2->getDistanceToFather() : s1->getDistanceToFather());
      s1->deleteDistanceToFather();
    }
    root_->sons().clear();
    delete root_;
    s1->removeFather();
    s1->addSon(s2);
    root_ = s1;
    return true;
  }

 private:
  N* root_;
};
typedef TreeTemplate<Node> Tree;

namespace TreeTemplateTools {
inline Node* parse_(const std::string& s, size_t& pos) {
  auto skip = [&]() { while (pos < s.size() && std::isspace((unsigned char)s[pos])) ++pos; };
  skip();
  Node* n = new Node();
  if (pos < s.size() && s[pos] == '(') {
    ++pos;
    for (;;) {
      n->addSon(parse_(s, pos));
      skip();
      if (pos < s.size() && s[pos] == ',') { ++pos; continue; }
      if (pos < s.size() && s[pos] == ')') { ++pos; break; }
      delete n;
      throw Exception("TreeTemplateTools::parenthesisToTree. Bad tree description: " + s);
    }
  }
  skip();
  size_t st = pos;
  while (pos < s.size() && std::string(",():;").find(s[pos]) == std::string::npos) ++pos;
  std::string nm = s.substr(st, pos - st);
  while (!nm.empty() && std::isspace((unsigned char)nm.back())) nm.pop_back();
  if (!nm.empty()) n->setName(nm);
  skip();
  if (pos < s.size() && s[pos] == ':') {
    ++pos;
    st = pos;
    while (pos < s.size() && std::string(",();").find(s[pos]) == std::string::npos) ++pos;
    n->setDistanceToFather(std::strtod(s.substr(st, pos - st).c_str(), nullptr));
  }
  return n;
}
inline TreeTemplate<Node>* parenthesisToTree(const std::string& description) {
  size_t pos = 0;
  return new TreeTemplate<Node>(parse_(description, pos));
}
}  // namespace TreeTemplateTools


// BipartitionList (BipartitionList.h), minimal: one bitset per branch (every non-root node) over the leaves in sorted-name
// order, normalised to the side without the first leaf, so that the two branches at the root of a rooted tree give one split
// and the split does not depend on son order or rooting.
class BipartitionList {
 public:
  explicit BipartitionList(const Tree& tree) {
    names_ = tree.getLeavesNames();
    std::sort(names_.begin(), names_.end());
    std::map<std::string, size_t> bit;
    for (size_t i = 0; i < names_.size(); ++i) bit[names_[i]] = i;
    std::map<const Node*, std::vector<bool> > below;
    for (Node* n : tree.getNodes()) {
      std::vector<bool>& b = below[n];
      b.assign(names_.size(), false);
      if (n->isLeaf()) b[bit.at(n->getName())] = true;
      for (size_t s = 0; s < n->getNumberOfSons(); ++s) {
        const std::vector<bool>& c = below[n->getSon(s)];
        for (size_t i = 0; i < b.size(); ++i) b[i] = b[i] || c[i];
      }
      if (!n->hasFather()) continue;
      std::vector<bool> side = b;
      if (side[0]) side.flip();
      splits_.push_back(side);
      nodes_.push_back(n);
    }
  }
  const std::vector<std::string>& getElementNames() const { return names_; }
  size_t getNumberOfBipartitions() const { return splits_.size(); }
  const std::vector<bool>& getBitBipartition(size_t i) const { return splits_[i]; }
  Node* getNode(size_t i) const { return nodes_[i]; }

 private:
  std::vector<std::string> names_;
  std::vector<std::vector<bool> > splits_;
  std::vector<Node*> nodes_;
};

namespace TreeTools {
static const std::string BOOTSTRAP = "bootstrap";
// computeBootstrapValues (TreeTools.cpp): for each internal branch of `tree`, the percentage of `trees` that contain its split,
// rounded half up to `format` decimals, stored as the branch property BOOTSTRAP.  Leaf branches get none.
inline void computeBootstrapValues(Tree& tree, const std::vector<Tree*>& trees, bool verbose = true, int format = 0) {
  if (trees.empty()) throw Exception("TreeTools::computeBootstrapValues: no replicate trees");
  const BipartitionList main(tree);
  std::map<std::vector<bool>, size_t> count;
  for (const Tree* t : trees) {
    const BipartitionList bl(*t);
    if (bl.getElementNames() != main.getElementNames())
      throw Exception("TreeTools::computeBootstrapValues: a replicate tree has another leaf set");
    std::set<std::vector<bool> > seen;
    for (size_t i = 0; i < bl.getNumberOfBipartitions(); ++i)
      if (seen.insert(bl.getBitBipartition(i)).second) ++count[bl.getBitBipartition(i)];
  }
  const double f = std::pow(10.0, format);
  for (size_t i = 0; i < main.getNumberOfBipartitions(); ++i) {
    Node* n = main.getNode(i);
    if (n->isLeaf()) continue;
    auto it = count.find(main.getBitBipartition(i));
    const double v = 100.0 * (it == count.end() ? 0 : it->second) / trees.size();
    n->setBranchProperty(BOOTSTRAP, std::floor(v * f + 0.5) / f);
  }
  if (verbose) std::printf("computeBootstrapValues: %zu trees, %zu branches\n", trees.size(), main.getNumberOfBipartitions());
}
}  // namespace TreeTools

}  // namespace bppshim
