// bppgpu shim (see ../bppgpu_shim.hpp): rate distributions, substitution models, omega mixtures, frequency sets, model sets
#pragma once
#include "io.hpp"

namespace bppshim {

// ---- rate distributions --------------------------------------------------------------------------------------------------
class DiscreteDistribution {
 public:
  virtual ~DiscreteDistribution() {}
  size_t getNumberOfCategories() const { return values_.size(); }
  double getCategory(size_t i) const { return values_[i]; }
  double getProbability(size_t i) const { return probs_[i]; }
  virtual void setParameterValue(const std::string& name, double v) { (void)name; (void)v; throw ParameterNotFoundException(name); }

 protected:
  Vdouble values_, probs_;
};
class ConstantRateDistribution : public DiscreteDistribution {
 public:
  ConstantRateDistribution() { values_.assign(1, 1.0); probs_.assign(1, 1.0); }
};
// Gamma(alpha, beta = alpha), K equiprobable classes, class value = class mean (bpp-core GammaDiscreteDistribution)
class GammaDiscreteRateDistribution : public DiscreteDistribution {
 public:
  GammaDiscreteRateDistribution(size_t n, double alpha = 1.0) : n_(n), alpha_(alpha) { discretize(); }
  void setParameterValue(const std::string& name, double v) {
    if (name != "alpha" && name != "Gamma.alpha") throw ParameterNotFoundException(name);
    alpha_ = v;
    discretize();
  }
  double getAlpha() const { return alpha_; }

 private:
  void discretize() {
    values_.assign(n_, 1.0);
    probs_.assign(n_, 1.0 / (double)n_);
    if (n_ == 1) return;
    const double beta = alpha_;
    std::vector<double> cdf1(n_ + 1, 0.0);
    cdf1[n_] = 1.0;
    for (size_t i = 1; i < n_; ++i) {
      const double q = linalg::gammp_inv(alpha_, (double)i / (double)n_) / beta;  // class bound
      cdf1[i] = linalg::gammp(alpha_ + 1.0, q * beta);
    }
    for (size_t i = 0; i < n_; ++i) values_[i] = (double)n_ * (alpha_ / beta) * (cdf1[i + 1] - cdf1[i]);
  }
  size_t n_;
  double alpha_;
};

// ---- substitution models -----------------------------------------------------------------------------------------------------
class SubstitutionModel {
 public:
  virtual ~SubstitutionModel() {}
  virtual std::string getName() const = 0;
  virtual const Alphabet* getAlphabet() const = 0;
  virtual size_t getNumberOfStates() const = 0;
  virtual const RowMatrix<double>& getPij_t(double t) const = 0;
  virtual const RowMatrix<double>& getdPij_dt(double t) const = 0;
  virtual const RowMatrix<double>& getd2Pij_dt2(double t) const = 0;
  virtual double Pij_t(size_t i, size_t j, double t) const { return getPij_t(t)(i, j); }
  virtual double dPij_dt(size_t i, size_t j, double t) const { return getdPij_dt(t)(i, j); }
  virtual double d2Pij_dt2(size_t i, size_t j, double t) const { return getd2Pij_dt2(t)(i, j); }
  virtual const RowMatrix<double>& getGenerator() const = 0;
  virtual const Vdouble& getEigenValues() const = 0;
  virtual const Vdouble& getIEigenValues() const = 0;
  virtual bool isDiagonalizable() const = 0;
  virtual bool isNonSingular() const = 0;
  virtual const RowMatrix<double>& getRowLeftEigenVectors() const = 0;
  virtual const RowMatrix<double>& getColumnRightEigenVectors() const = 0;
  virtual double getRate() const = 0;
  virtual void setRate(double r) = 0;
  virtual const Vdouble& getFrequencies() const = 0;
  virtual double getInitValue(size_t i, const std::string& ch) const = 0;
  virtual void setParameterValue(const std::string& name, double v) = 0;
  virtual std::vector<std::string> getParameterNames() const = 0;
  virtual void fillModelDesc(bppgpu_model_desc& d) const = 0;
  virtual SubstitutionModel* clone() const = 0;
  virtual double getParameterValue(const std::string& name) const { throw ParameterNotFoundException(name); }
};

class AbstractSubstitutionModel : public SubstitutionModel {
 public:
  AbstractSubstitutionModel(const Alphabet* alpha, size_t size)
      : alphabet_(alpha), size_(size), rate_(1.0), generator_(size, size), freq_(size, 1.0 / (double)size), eigenValues_(size),
        iEigenValues_(size, 0.0), isDiagonalizable_(false), isNonSingular_(false), isScalable_(true), reversible_(false),
        rightEigenVectors_(size, size), leftEigenVectors_(size, size), device_(0), extraFlags_(0), pijt_(size, size),
        dpijt_(size, size), d2pijt_(size, size) {}
  const Alphabet* getAlphabet() const { return alphabet_; }
  size_t getNumberOfStates() const { return size_; }
  const RowMatrix<double>& getGenerator() const { return generator_; }
  const Vdouble& getEigenValues() const { return eigenValues_; }
  const Vdouble& getIEigenValues() const { return iEigenValues_; }
  bool isDiagonalizable() const { return isDiagonalizable_; }
  bool isNonSingular() const { return isNonSingular_; }
  const RowMatrix<double>& getRowLeftEigenVectors() const { return leftEigenVectors_; }
  const RowMatrix<double>& getColumnRightEigenVectors() const { return rightEigenVectors_; }
  double getRate() const { return rate_; }
  void setRate(double r) { if (r <= 0) throw Exception("Bad value for rate: " + std::to_string(r)); rate_ = r; }
  const Vdouble& getFrequencies() const { return freq_; }
  void setDevice(int d) { device_ = d; }

  // AbstractTransitionModel::getInitValue (Model/AbstractSubstitutionModel.cpp:98-112)
  double getInitValue(size_t i, const std::string& ch) const {
    if (i >= size_) throw Exception("IndexOutOfBoundsException: AbstractTransitionModel::getInitValue");
    const std::vector<int> states = alphabet_->getAlias(ch);
    if (states.empty()) throw Exception("BadIntException: AbstractTransitionModel::getInitValue. Character " + ch + " is not allowed in model.");
    for (int s : states)
      if ((int)i == s) return 1.0;
    return 0.0;
  }

  // getPij_t / getdPij_dt / getd2Pij_dt2 (Model/AbstractSubstitutionModel.cpp:426-641): Interface 1 of the C ABI.
  // Like the reference the returned reference is to an internal buffer, valid until the next call.
  const RowMatrix<double>& getPij_t(double t) const { return ptable_(t, BPPGPU_WANT_P, pijt_); }
  const RowMatrix<double>& getdPij_dt(double t) const { return ptable_(t, BPPGPU_WANT_DP, dpijt_); }
  const RowMatrix<double>& getd2Pij_dt2(double t) const { return ptable_(t, BPPGPU_WANT_D2P, d2pijt_); }

  void fillModelDesc(bppgpu_model_desc& d) const {
    d.n_states = (int32_t)size_;
    d.flags = (isDiagonalizable_ ? BPPGPU_MODEL_DIAGONALIZABLE : 0u) | (isNonSingular_ ? BPPGPU_MODEL_NONSINGULAR : 0u) | extraFlags_;
    d.rate = rate_;
    d.right_eigen = rightEigenVectors_.data();
    d.left_eigen = leftEigenVectors_.data();
    d.eigen_re = eigenValues_.data();
    d.eigen_im = iEigenValues_.data();
    d.generator = generator_.data();
    d.taylor_epsilon = 1e-4;
  }

 protected:
  // AbstractSubstitutionModel::updateMatrices (Model/AbstractSubstitutionModel.cpp:175-421): null ("stop") lines are
  // stripped, the rest eigen-decomposed on the host, the ~0 eigenvalue pinned to 0 and (optionally) turned into the
  // equilibrium frequencies, then the generator is normalised to one substitution per unit time if scalable.
  void updateMatrices(bool computeFreq) {
    const int n = (int)size_;
    std::vector<char> vnull(n, 0);
    std::vector<int> ok;
    for (int i = 0; i < n; ++i) {
      bool null_ = std::fabs(generator_(i, i)) < NumConstants::TINY();
      for (int j = 0; null_ && j < n; ++j)
        if (std::fabs(generator_(j, i)) >= NumConstants::TINY()) null_ = false;
      vnull[i] = null_;
      if (!null_) ok.push_back(i);
    }
    const int m = (int)ok.size();
    std::vector<double> A((size_t)m * m), re, im, Vk;
    for (int i = 0; i < m; ++i)
      for (int j = 0; j < m; ++j) A[(size_t)i * m + j] = generator_(ok[i], ok[j]);
    bool eig_ok;
    if (reversible_) {
      // pi^1/2 Q pi^-1/2 is symmetric for a reversible generator
      std::vector<double> B((size_t)m * m), w, U;
      std::vector<double> sq(m);
      for (int i = 0; i < m; ++i) sq[i] = std::sqrt(freq_[ok[i]]);
      for (int i = 0; i < m; ++i)
        for (int j = 0; j < m; ++j) B[(size_t)i * m + j] = 0.5 * (sq[i] * A[(size_t)i * m + j] / sq[j] + sq[j] * A[(size_t)j * m + i] / sq[i]);
      linalg::jacobi_symmetric(B, m, w, U);
      re = w;
      im.assign(m, 0.0);
      Vk.assign((size_t)m * m, 0.0);
      for (int i = 0; i < m; ++i)
        for (int k = 0; k < m; ++k) Vk[(size_t)i * m + k] = U[(size_t)i * m + k] / sq[i];
      eig_ok = true;
    } else {
      eig_ok = linalg::eigen_general(A, m, re, im, Vk);
    }
    std::vector<double> V((size_t)n * n, 0.0), Vinv;
    eigenValues_.assign(n, 0.0);
    iEigenValues_.assign(n, 0.0);
    isNonSingular_ = false;
    isDiagonalizable_ = false;
    if (eig_ok) {
      for (int k = 0; k < m; ++k) { eigenValues_[k] = re[k]; iEigenValues_[k] = im[k]; }
      for (int i = 0; i < m; ++i)
        for (int k = 0; k < m; ++k) V[(size_t)ok[i] * n + k] = Vk[(size_t)i * m + k];
      int gi = 0;
      for (int i = 0; i < n; ++i)
        if (vnull[i]) V[(size_t)i * n + m + gi++] = 1.0;
      bool usable = linalg::invert(V, n, Vinv);
      if (usable) {
        // the eigen form must reproduce the generator; a (nearly) defective matrix does not and takes the series path,
        // as the reference does when MatrixTools::inv fails (:283-291)
        // V D with D block diagonal ([[re, im], [-im, re]] per conjugate pair): column work, then one product
        std::vector<double> VD((size_t)n * n);
        for (int k = 0; k < n; ++k) {
          const double re_k = eigenValues_[k], im_k = iEigenValues_[k];
          for (int i = 0; i < n; ++i) {
            double v = V[(size_t)i * n + k] * re_k;
            if (im_k > 0 && k + 1 < n) v -= V[(size_t)i * n + k + 1] * im_k;           // D[k+1][k] = -im
            else if (im_k < 0 && k >= 1 && iEigenValues_[k - 1] > 0) v += V[(size_t)i * n + k - 1] * iEigenValues_[k - 1];   // D[k-1][k] = +im
            VD[(size_t)i * n + k] = v;
          }
        }
        const std::vector<double> R = linalg::matmul(VD, Vinv, n);
        double err = 0.0, nrm = 0.0;
        for (int i = 0; i < n; ++i)
          for (int j = 0; j < n; ++j) {
            err = std::max(err, std::fabs(R[(size_t)i * n + j] - generator_(i, j)));
            nrm = std::max(nrm, std::fabs(generator_(i, j)));
          }
        if (!(err <= 1e-8 * std::max(nrm, 1e-300))) usable = false;
      }
      if (usable) {
        isDiagonalizable_ = true;
        if (!reversible_)
          for (int k = 0; k < n; ++k)
            if (std::fabs(iEigenValues_[k]) > NumConstants::TINY()) isDiagonalizable_ = false;
        // the unique ~0 eigenvalue (tolerance ladder, :306-315)
        std::vector<int> nullev;
        double fact = 0.1;
        while (nullev.empty() && fact < 1000) {
          fact *= 10;
          for (int k = 0; k < m; ++k)
            if (std::fabs(eigenValues_[k]) < fact * NumConstants::SMALL() && std::fabs(iEigenValues_[k]) < NumConstants::SMALL()) nullev.push_back(k);
        }
        int nulleigen = -1;
        if (nullev.size() == 1) nulleigen = nullev[0];
        else
          for (int cand : nullev) {  // :326-352: the one whose right vector is constant
            const double val = V[(size_t)ok[0] * n + cand];
            bool cst = val != 0.0;
            for (int i = 1; cst && i < m; ++i)
              if (std::fabs((V[(size_t)ok[i] * n + cand] - val) / val) > NumConstants::SMALL()) cst = false;
            if (cst) { nulleigen = cand; break; }
          }
        if (nulleigen >= 0) {
          isNonSingular_ = true;
          eigenValues_[nulleigen] = 0.0;
          iEigenValues_[nulleigen] = 0.0;
          if (computeFreq) {
            double sum = 0.0;
            for (int j = 0; j < n; ++j) sum += Vinv[(size_t)nulleigen * n + j];
            for (int j = 0; j < n; ++j) freq_[j] = Vinv[(size_t)nulleigen * n + j] / sum;
          }
        } else {
          isDiagonalizable_ = false;
        }
      }
    }
    if (!isNonSingular_) {
      // :386-410: rescale so the fastest state leaves at rate 1, frequencies from (I + Q)^256
      double mn = 0.0;
      for (int i = 0; i < n; ++i) mn = std::min(mn, generator_(i, i));
      if (isScalable_ && mn < 0) scaleGenerator(-1.0 / mn);
      if (computeFreq) {
        std::vector<double> T((size_t)n * n);
        for (int i = 0; i < n; ++i)
          for (int j = 0; j < n; ++j) T[(size_t)i * n + j] = generator_(i, j) + (i == j ? 1.0 : 0.0);
        for (int k = 0; k < 8; ++k) T = linalg::matmul(T, T, n);
        for (int j = 0; j < n; ++j) freq_[j] = T[j];
      }
      Vinv.assign((size_t)n * n, 0.0);
    }
    for (int i = 0; i < n; ++i)
      for (int j = 0; j < n; ++j) {
        rightEigenVectors_(i, j) = V[(size_t)i * n + j];
        leftEigenVectors_(i, j) = Vinv.empty() ? 0.0 : Vinv[(size_t)i * n + j];
      }
    if (isScalable_) {  // normalize(): -sum_i pi_i Q_ii = 1  (:645-652, :684-688)
      double sc = 0.0;
      for (int i = 0; i < n; ++i) sc -= freq_[i] * generator_(i, i);
      if (sc > 0) scaleGenerator(1.0 / sc);
    }
  }
  void scaleGenerator(double s) {
    for (size_t i = 0; i < size_; ++i) {
      for (size_t j = 0; j < size_; ++j) generator_(i, j) *= s;
      eigenValues_[i] *= s;
      iEigenValues_[i] *= s;
    }
  }
  void setDiagonal() {
    for (size_t i = 0; i < size_; ++i) {
      double s = 0.0;
      for (size_t j = 0; j < size_; ++j)
        if (j != i) s += generator_(i, j);
      generator_(i, i) = -s;
    }
  }

  const Alphabet* alphabet_;
  size_t size_;
  double rate_;
  RowMatrix<double> generator_;
  Vdouble freq_, eigenValues_, iEigenValues_;
  bool isDiagonalizable_, isNonSingular_, isScalable_, reversible_;
  RowMatrix<double> rightEigenVectors_, leftEigenVectors_;
  int device_;
  unsigned extraFlags_;

 private:
  const RowMatrix<double>& ptable_(double t, unsigned which, RowMatrix<double>& out) const {
    bppgpu_model_desc d;
    fillModelDesc(d);
    check(bppgpu_pt_batch(device_, &d, 1, &t, which, which == BPPGPU_WANT_P ? out.data() : nullptr,
                          which == BPPGPU_WANT_DP ? out.data() : nullptr, which == BPPGPU_WANT_D2P ? out.data() : nullptr),
          "getPij_t");
    return out;
  }
  mutable RowMatrix<double> pijt_, dpijt_, d2pijt_;
};

// AbstractReversibleSubstitutionModel::updateMatrices (:694-703): generator = exchangeability * frequencies
class AbstractReversibleSubstitutionModel : public AbstractSubstitutionModel {
 public:
  AbstractReversibleSubstitutionModel(const Alphabet* a, size_t n) : AbstractSubstitutionModel(a, n), exch_(n, n) { reversible_ = true; }

 protected:
  void updateReversible() {
    for (size_t i = 0; i < size_; ++i)
      for (size_t j = 0; j < size_; ++j) generator_(i, j) = i == j ? 0.0 : exch_(i, j) * freq_[j];
    setDiagonal();
    double sc = 0.0;
    for (size_t i = 0; i < size_; ++i) sc -= freq_[i] * generator_(i, i);
    scaleGenerator(1.0 / sc);
    const Vdouble keep = freq_;
    updateMatrices(false);
    freq_ = keep;
  }
  RowMatrix<double> exch_;
};

// Model/Nucleotide/GTR.cpp:84-124: exchangeabilities AC=d AG=1 AT=b CG=e CT=a GT=c; theta, theta1, theta2 frequencies
class GTR : public AbstractReversibleSubstitutionModel {
 public:
  GTR(const Alphabet* alpha, double a = 1., double b = 1., double c = 1., double d = 1., double e = 1., double piA = 0.25,
      double piC = 0.25, double piG = 0.25, double piT = 0.25)
      : AbstractReversibleSubstitutionModel(alpha, 4), a_(a), b_(b), c_(c), d_(d), e_(e) {
    freq_[0] = piA; freq_[1] = piC; freq_[2] = piG; freq_[3] = piT;
    update();
  }
  GTR* clone() const { return new GTR(*this); }
  std::string getName() const { return "GTR"; }
  std::vector<std::string> getParameterNames() const { return {"GTR.a", "GTR.b", "GTR.c", "GTR.d", "GTR.e"}; }
  double getParameterValue(const std::string& name) const {
    const std::string n = name.substr(name.find('.') == std::string::npos ? 0 : name.find('.') + 1);
    const std::map<std::string, const double*> m = {{"a", &a_}, {"b", &b_}, {"c", &c_}, {"d", &d_}, {"e", &e_}};
    const auto it = m.find(n);
    if (it == m.end()) throw ParameterNotFoundException(name);
    return *it->second;
  }
  void setParameterValue(const std::string& name, double v) {
    const std::string n = name.substr(name.find('.') == std::string::npos ? 0 : name.find('.') + 1);
    if (n == "a") a_ = v; else if (n == "b") b_ = v; else if (n == "c") c_ = v; else if (n == "d") d_ = v; else if (n == "e") e_ = v;
    else throw ParameterNotFoundException(name);
    update();
  }

 private:
  void update() {
    exch_.resize(4, 4);
    exch_(0, 1) = exch_(1, 0) = d_; exch_(0, 2) = exch_(2, 0) = 1.0; exch_(0, 3) = exch_(3, 0) = b_;
    exch_(1, 2) = exch_(2, 1) = e_; exch_(1, 3) = exch_(3, 1) = a_; exch_(2, 3) = exch_(3, 2) = c_;
    updateReversible();
  }
  double a_, b_, c_, d_, e_;
};

// Model/Nucleotide/HKY85.cpp:80-191 (generic eigen path instead of the closed form: identical P)
class HKY85 : public AbstractReversibleSubstitutionModel {
 public:
  HKY85(const Alphabet* alpha, double kappa = 1., double piA = 0.25, double piC = 0.25, double piG = 0.25, double piT = 0.25,
        const std::string& name = "HKY85")
      : AbstractReversibleSubstitutionModel(alpha, 4), kappa_(kappa), name_(name) {
    freq_[0] = piA; freq_[1] = piC; freq_[2] = piG; freq_[3] = piT;
    update();
  }
  HKY85* clone() const { return new HKY85(*this); }
  std::string getName() const { return name_; }
  std::vector<std::string> getParameterNames() const { return {name_ + ".kappa"}; }
  double getParameterValue(const std::string& name) const {
    if (name == "kappa" || name == name_ + ".kappa") return kappa_;
    throw ParameterNotFoundException(name);
  }
  void setParameterValue(const std::string& name, double v) {
    if (name != "kappa" && name != name_ + ".kappa") throw ParameterNotFoundException(name);
    kappa_ = v;
    update();
  }
  double getKappa() const { return kappa_; }

 protected:
  void update() {
    exch_.resize(4, 4);
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 4; ++j) exch_(i, j) = i == j ? 0.0 : 1.0;
    exch_(0, 2) = exch_(2, 0) = kappa_;
    exch_(1, 3) = exch_(3, 1) = kappa_;
    updateReversible();
  }
  double kappa_;
  std::string name_;
};
// Model/Nucleotide/T92.cpp:81-187: HKY85 with pi = ((1-theta)/2, theta/2, theta/2, (1-theta)/2)
class T92 : public HKY85 {
 public:
  T92(const Alphabet* alpha, double kappa = 1., double theta = 0.5)
      : HKY85(alpha, kappa, (1 - theta) / 2, theta / 2, theta / 2, (1 - theta) / 2, "T92"), theta_(theta) {}
  T92* clone() const { return new T92(*this); }
  std::vector<std::string> getParameterNames() const { return {"T92.kappa", "T92.theta"}; }
  double getParameterValue(const std::string& name) const {
    if (name == "theta" || name == "T92.theta") return theta_;
    return HKY85::getParameterValue(name);
  }
  void setParameterValue(const std::string& name, double v) {
    if (name == "theta" || name == "T92.theta") {   // T92::updateMatrices (T92.cpp:81-94): piA = piT = (1 - theta) / 2, piC = piG = theta / 2
      theta_ = v;
      freq_[0] = freq_[3] = (1 - v) / 2;
      freq_[1] = freq_[2] = v / 2;
      update();
    } else HKY85::setParameterValue(name, v);
  }

 private:
  double theta_;
};
class K80 : public HKY85 {
 public:
  K80(const Alphabet* alpha, double kappa = 1.) : HKY85(alpha, kappa, .25, .25, .25, .25, "K80") {}
  K80* clone() const { return new K80(*this); }
};
class JCnuc : public HKY85 {
 public:
  explicit JCnuc(const Alphabet* alpha) : HKY85(alpha, 1.0, .25, .25, .25, .25, "JC69") {}
  JCnuc* clone() const { return new JCnuc(*this); }
};

// Model/Protein/LG08.cpp:53-62 + the published Le & Gascuel 2008 constants
#include "../lg08_data.inc"
class LG08 : public AbstractReversibleSubstitutionModel {
 public:
  explicit LG08(const Alphabet* alpha) : AbstractReversibleSubstitutionModel(alpha, 20) {
    int k = 0;
    for (int i = 1; i < 20; ++i)
      for (int j = 0; j < i; ++j) exch_(i, j) = exch_(j, i) = LG08_LOWER[k++];
    for (int i = 0; i < 20; ++i) freq_[i] = LG08_FREQ[i];
    updateReversible();
  }
  LG08* clone() const { return new LG08(*this); }
  std::string getName() const { return "LG08"; }
  std::vector<std::string> getParameterNames() const { return {}; }
  void setParameterValue(const std::string& name, double) { throw ParameterNotFoundException(name); }
};

// Model/Codon/YN98.cpp:51-77: K80 rate / 3 on single-nucleotide changes, x omega if non-synonymous, x target codon
// frequency, stop codons zeroed (AbstractCodonSubstitutionModel.cpp:174-191), then normalised
class YN98 : public AbstractSubstitutionModel {
 public:
  YN98(const Alphabet* alpha, double kappa = 1., double omega = 1., const Vdouble* codonFreq = nullptr)
      : AbstractSubstitutionModel(alpha, 64), kappa_(kappa), omega_(omega) {
    if (codonFreq) freq_ = *codonFreq;
    else {
      double n = 0;
      for (int i = 0; i < 64; ++i) { freq_[i] = CodonAlphabet::isStop(i) ? 0.0 : 1.0; n += freq_[i]; }
      for (int i = 0; i < 64; ++i) freq_[i] /= n;
    }
    reversible_ = false;  // the reference runs the general EigenValue path for word models
    update();
  }
  YN98* clone() const { return new YN98(*this); }
  std::string getName() const { return "YN98"; }
  double getParameterValue(const std::string& name) const {
    if (name == "kappa" || name == "YN98.kappa") return kappa_;
    if (name == "omega" || name == "YN98.omega") return omega_;
    throw ParameterNotFoundException(name);
  }
  std::vector<std::string> getParameterNames() const { return {"YN98.kappa", "YN98.omega"}; }
  void setParameterValue(const std::string& name, double v) {
    if (name == "kappa" || name == "YN98.kappa") kappa_ = v;
    else if (name == "omega" || name == "YN98.omega") omega_ = v;
    else throw ParameterNotFoundException(name);
    update();
  }

 private:
  void update() {
    for (int i = 0; i < 64; ++i)
      for (int j = 0; j < 64; ++j) {
        generator_(i, j) = 0.0;
        if (i == j) continue;
        const int di[3] = {i / 16, (i / 4) % 4, i % 4}, dj[3] = {j / 16, (j / 4) % 4, j % 4};
        int ndiff = 0, p = -1;
        for (int k = 0; k < 3; ++k)
          if (di[k] != dj[k]) { ++ndiff; p = k; }
        if (ndiff != 1 || CodonAlphabet::isStop(i) || CodonAlphabet::isStop(j)) continue;
        const bool ts = (di[p] == 0 && dj[p] == 2) || (di[p] == 2 && dj[p] == 0) || (di[p] == 1 && dj[p] == 3) || (di[p] == 3 && dj[p] == 1);
        double r = (ts ? kappa_ : 1.0) / (kappa_ + 2.0) / 3.0;
        r *= (CodonAlphabet::aminoAcid(i) == CodonAlphabet::aminoAcid(j) ? 1.0 : omega_) * freq_[j];
        generator_(i, j) = r;
      }
    setDiagonal();
    const Vdouble keep = freq_;
    // reversible w.r.t. the codon frequencies: use the symmetric solver on the sense codons
    reversible_ = true;
    updateMatrices(false);
    reversible_ = false;
    freq_ = keep;
  }
  double kappa_, omega_;
};

// Grantham (1974) amino-acid distances, what bpp-seq's GranthamAAChemicalDistance::getIndex returns in its default symmetric
// mode (GY94.h:45,88).  bpp-seq is not under /root/reference, so the published table is restated here in Grantham's own order
// (Ser Arg Leu Pro Thr Ala Val Gly Ile Phe Tyr Cys His Gln Asn Lys Asp Glu Met Trp), upper triangle by rows.
inline double granthamDistance(char a, char b) {
  static const char* order = "SRLPTAVGIFYCHQNKDEMW";
  static const int upper[190] = {
      110, 145, 74, 58, 99, 124, 56, 142, 155, 144, 112, 89, 68, 46, 121, 65, 80, 135, 177,
      102, 103, 71, 112, 96, 125, 97, 97, 77, 180, 29, 43, 86, 26, 96, 54, 91, 101,
      98, 92, 96, 32, 138, 5, 22, 36, 198, 99, 113, 153, 107, 172, 138, 15, 61,
      38, 27, 68, 42, 95, 114, 110, 169, 77, 76, 91, 103, 108, 93, 87, 147,
      58, 69, 59, 89, 103, 92, 149, 47, 42, 65, 78, 85, 65, 81, 128,
      64, 60, 94, 113, 112, 195, 86, 91, 111, 106, 126, 107, 84, 148,
      109, 29, 50, 55, 192, 84, 96, 133, 97, 152, 121, 21, 88,
      135, 153, 147, 159, 98, 87, 80, 127, 94, 98, 127, 184,
      21, 33, 198, 94, 109, 149, 102, 168, 134, 10, 61,
      22, 205, 100, 116, 158, 102, 177, 140, 28, 40,
      194, 83, 99, 143, 85, 160, 122, 36, 37,
      174, 154, 139, 202, 154, 170, 196, 215,
      24, 68, 32, 81, 40, 87, 115,
      46, 53, 61, 29, 101, 130,
      94, 23, 42, 142, 174,
      101, 56, 95, 110,
      45, 160, 181,
      126, 152,
      67};
  int i = -1, j = -1;
  for (int k = 0; k < 20; ++k) {
    if (order[k] == a) i = k;
    if (order[k] == b) j = k;
  }
  if (i < 0 || j < 0) throw Exception("granthamDistance: not an amino acid");
  if (i == j) return 0.0;
  if (i > j) std::swap(i, j);
  // row i starts after sum_{r<i} (19 - r) entries
  return (double)upper[i * 19 - i * (i - 1) / 2 + (j - i - 1)];
}

// Model/Codon/GY94.cpp:49-71 = CodonDistanceFrequenciesSubstitutionModel over K80 with the Grantham distance:
// K80 rate / 3 on single-nucleotide changes (AbstractWordSubstitutionModel::fillBasicGenerator), x exp(-d(aa_i, aa_j) / V) when
// non-synonymous (beta = gamma = 1, AbstractCodonDistanceSubstitutionModel.cpp:80-88), x target codon frequency, stop codons
// zeroed (AbstractCodonSubstitutionModel.cpp:174-191), then normalised.  Parameters "GY94.kappa" (1) and "GY94.V" (10000).
class GY94 : public AbstractSubstitutionModel {
 public:
  GY94(const Alphabet* alpha, double kappa = 1., double V = 10000., const Vdouble* codonFreq = nullptr)
      : AbstractSubstitutionModel(alpha, 64), kappa_(kappa), V_(V) {
    if (codonFreq) freq_ = *codonFreq;
    else {
      double n = 0;
      for (int i = 0; i < 64; ++i) { freq_[i] = CodonAlphabet::isStop(i) ? 0.0 : 1.0; n += freq_[i]; }
      for (int i = 0; i < 64; ++i) freq_[i] /= n;
    }
    reversible_ = false;
    update();
  }
  GY94* clone() const { return new GY94(*this); }
  std::string getName() const { return "GY94"; }
  double getParameterValue(const std::string& name) const {
    if (name == "kappa" || name == "GY94.kappa") return kappa_;
    if (name == "V" || name == "GY94.V") return V_;
    throw ParameterNotFoundException(name);
  }
  std::vector<std::string> getParameterNames() const { return {"GY94.kappa", "GY94.V"}; }
  void setParameterValue(const std::string& name, double v) {
    if (name == "kappa" || name == "GY94.kappa") kappa_ = v;
    else if (name == "V" || name == "GY94.V") V_ = v;
    else throw ParameterNotFoundException(name);
    update();
  }
  double getCodonsMulRate(size_t i, size_t j) const {
    const char ai = CodonAlphabet::aminoAcid((int)i), aj = CodonAlphabet::aminoAcid((int)j);
    return ai == aj ? 1.0 : std::exp(-granthamDistance(ai, aj) / V_);
  }

 private:
  void update() {
    for (int i = 0; i < 64; ++i)
      for (int j = 0; j < 64; ++j) {
        generator_(i, j) = 0.0;
        if (i == j) continue;
        const int di[3] = {i / 16, (i / 4) % 4, i % 4}, dj[3] = {j / 16, (j / 4) % 4, j % 4};
        int ndiff = 0, p = -1;
        for (int k = 0; k < 3; ++k)
          if (di[k] != dj[k]) { ++ndiff; p = k; }
        if (ndiff != 1 || CodonAlphabet::isStop(i) || CodonAlphabet::isStop(j)) continue;
        const bool ts = (di[p] == 0 && dj[p] == 2) || (di[p] == 2 && dj[p] == 0) || (di[p] == 1 && dj[p] == 3) || (di[p] == 3 && dj[p] == 1);
        generator_(i, j) = (ts ? kappa_ : 1.0) / (kappa_ + 2.0) / 3.0 * getCodonsMulRate(i, j) * freq_[j];
      }
    setDiagonal();
    const Vdouble keep = freq_;
    reversible_ = true;   // reversible w.r.t. the codon frequencies: symmetric solver on the sense codons
    updateMatrices(false);
    reversible_ = false;
    freq_ = keep;
  }
  double kappa_, V_;
};

// Model/ChromosomeSubstitutionModel.cpp:431-802 (gain / loss / duplication / demi-duplication / base number)
class ChromosomeSubstitutionModel : public AbstractSubstitutionModel {
 public:
  static constexpr double IgnoreParam = -999.0;   // ChromosomeSubstitutionModel.h:15-23
  static constexpr double DemiEqualDupl = -2.0;
  enum rateChangeFunc { LINEAR = 0, EXP = 1 };
  ChromosomeSubstitutionModel(const ChromosomeAlphabet* alpha, double gain, double loss, double dupl, double demi,
                              double gainR = IgnoreParam, double lossR = IgnoreParam, double duplR = IgnoreParam,
                              int baseNum = (int)IgnoreParam, double baseNumR = IgnoreParam, unsigned maxChrRange = 0,
                              rateChangeFunc rc = LINEAR)
      : AbstractSubstitutionModel(alpha, alpha->getSize()), chr_(alpha), gain_(gain), loss_(loss), dupl_(dupl), demi_(demi),
        gainR_(gainR), lossR_(lossR), duplR_(duplR), baseNum_(baseNum), baseNumR_(baseNumR), maxChrRange_(maxChrRange), rc_(rc) {
    isScalable_ = false;  // :58
    extraFlags_ = BPPGPU_MODEL_CLAMP01 | BPPGPU_MODEL_CHR_DERIV | BPPGPU_MODEL_CHR_TAYLOR;
    update();
  }
  ChromosomeSubstitutionModel* clone() const { return new ChromosomeSubstitutionModel(*this); }
  std::string getName() const { return "Chromosome"; }
  std::vector<std::string> getParameterNames() const { return {"Chromosome.gain", "Chromosome.loss", "Chromosome.dupl", "Chromosome.demi"}; }
  double getParameterValue(const std::string& name) const {
    const std::string n = name.substr(name.find('.') == std::string::npos ? 0 : name.find('.') + 1);
    const std::map<std::string, double> m = {{"gain", gain_}, {"loss", loss_}, {"dupl", dupl_}, {"demi", demi_}, {"gainR", gainR_},
                                             {"lossR", lossR_}, {"duplR", duplR_}, {"baseNumR", baseNumR_}};
    if (!m.count(n)) throw ParameterNotFoundException(name);
    return m.at(n);
  }
  void setParameterValue(const std::string& name, double v) {
    const std::string n = name.substr(name.find('.') == std::string::npos ? 0 : name.find('.') + 1);
    if (n == "gain") gain_ = v; else if (n == "loss") loss_ = v; else if (n == "dupl") dupl_ = v; else if (n == "demi") demi_ = v;
    else if (n == "gainR") gainR_ = v; else if (n == "lossR") lossR_ = v; else if (n == "duplR") duplR_ = v; else if (n == "baseNumR") baseNumR_ = v;
    else throw ParameterNotFoundException(name);
    update();
  }
  // event classes of ComputeChromosomeTransitionsExp, in the order of their rate terms in update()
  enum typeOfTransition { GAIN_T = 0, LOSS_T = 1, DUPL_T = 2, DEMIPLOIDY_T = 3, BASENUM_T = 4, NUMTYPES = 5 };
  // the generator's off-diagonal split by the rate term that produced it: [NUMTYPES][S][S], zero diagonal.  Added in class order
  // the five matrices give getGenerator()'s off-diagonal bit for bit (what bppgpu_expected_events takes as type_rates).
  std::vector<double> getTypeRates() const {
    const size_t n = size_;
    std::vector<double> R(NUMTYPES * n * n, 0.0);
    forEachRateTerm([&](int t, int r, int c, double v) { R[((size_t)t * n + (size_t)r) * n + (size_t)c] += v; });
    return R;
  }

 private:
  double rate_(int i, double c, double lin) const {  // getRate (:504-526)
    if (c == IgnoreParam && lin == IgnoreParam) return 0.0;
    const double total = c == IgnoreParam ? lin : c;
    if (lin == IgnoreParam) return total;
    return rc_ == LINEAR ? total + lin * (i - 1) : total * std::exp(lin * (i - 1));
  }
  // every rate term of the generator in the order update() adds them: add(class, row, column, rate), class 0..4 = gain, loss,
  // dupl, demi, baseNum.  A clamped jump keeps its class; the two demi / 2 targets at odd i are both demi.
  template <class F>
  void forEachRateTerm(F add) const {
    const int mn = (int)chr_->getMin(), mx = (int)chr_->getMax();
    const double demi = demi_ == DemiEqualDupl ? dupl_ : demi_;
    for (int i = mn; i <= mx; ++i) {
      const int r = i - mn;
      if (i + 1 <= mx) add(GAIN_T, r, r + 1, rate_(i, gain_, gainR_));
      if (i - 1 >= mn) add(LOSS_T, r, r - 1, rate_(i, loss_, lossR_));
      if (2 * i <= mx) add(DUPL_T, r, 2 * i - mn, rate_(i, dupl_, duplR_));
      else if (i != mx) add(DUPL_T, r, mx - mn, rate_(i, dupl_, duplR_));
      if (demi != IgnoreParam && i != mx) {  // :533-560
        if (i % 2 == 0 && (int)(i * 1.5) <= mx) add(DEMIPLOIDY_T, r, (int)(i * 1.5) - mn, demi);
        else if (i % 2 != 0 && (int)std::ceil(i * 1.5) <= mx) {
          if (i == 1) add(DEMIPLOIDY_T, r, (int)std::ceil(i * 1.5) - mn, demi);
          else {
            add(DEMIPLOIDY_T, r, (int)std::ceil(i * 1.5) - mn, demi / 2);
            add(DEMIPLOIDY_T, r, (int)std::floor(i * 1.5) - mn, demi / 2);
          }
        } else add(DEMIPLOIDY_T, r, mx - mn, demi);
      }
      if (i < mx && baseNum_ != (int)IgnoreParam)  // :562-577
        for (int j = i + 1; j <= mx; ++j) {
          if (j == mx) { if ((unsigned)(j - i) <= maxChrRange_) add(BASENUM_T, r, j - mn, baseNumR_); }
          else if ((j - i) % baseNum_ == 0 && (unsigned)(j - i) <= maxChrRange_) add(BASENUM_T, r, j - mn, baseNumR_);
        }
    }
  }
  void update() {
    const int n = (int)size_;
    for (int i = 0; i < n; ++i)
      for (int j = 0; j < n; ++j) generator_(i, j) = 0.0;
    forEachRateTerm([this](int, int r, int c, double v) { generator_(r, c) += v; });
    setDiagonal();
    updateMatrices(false);
    for (size_t i = 0; i < size_; ++i) freq_[i] = 1.0 / (double)size_;
  }
  const ChromosomeAlphabet* chr_;
  double gain_, loss_, dupl_, demi_, gainR_, lossR_, duplR_;
  int baseNum_;
  double baseNumR_;
  unsigned maxChrRange_;
  rateChangeFunc rc_;
};

// ---- mixtures of one model over a parameter (Model/MixedSubstitutionModel.h, MixtureOfASubstitutionModel) ---------------------------
class MixedSubstitutionModel {
 public:
  virtual ~MixedSubstitutionModel() {}
  virtual std::string getName() const = 0;
  virtual size_t getNumberOfModels() const = 0;
  virtual SubstitutionModel* getNModel(size_t i) const = 0;
  virtual double getNProbability(size_t i) const = 0;
  virtual std::vector<std::string> getParameterNames() const = 0;
  virtual double getParameterValue(const std::string& name) const = 0;
  virtual void setParameterValue(const std::string& name, double v) = 0;
  Vdouble getProbabilities() const {
    Vdouble p(getNumberOfModels());
    for (size_t i = 0; i < p.size(); ++i) p[i] = getNProbability(i);
    return p;
  }
};

// The omega mixtures of the YNGP wrappers: three YN98 that differ in omega, class probabilities from the simplex parameters
// theta1, theta2 (SimpleDiscreteDistribution: p0 = theta1, p1 = (1 - theta1) theta2, p2 = the rest), and the homogenisation of the
// synonymous rate (YNGP_M2::updateMatrices, Model/Codon/YNGP_M2.cpp:134-146): sub-model k gets the relative rate
// 1 / Q_k(synfrom, synto) for the first synonymous pair with non-zero rates, normalised to mean 1 under the probabilities
// (MixtureOfASubstitutionModel::setVRates).
class OmegaMixture_ : public MixedSubstitutionModel {
 public:
  size_t getNumberOfModels() const { return 3; }
  SubstitutionModel* getNModel(size_t i) const { return sub_.at(i).get(); }
  double getNProbability(size_t i) const { return probs_.at(i); }

 protected:
  OmegaMixture_(const Alphabet* alpha, const Vdouble* codonFreq) : alpha_(alpha) { if (codonFreq) codonFreq_ = *codonFreq; }
  void rebuild(double kappa, const double omega[3], double theta1, double theta2) {
    probs_ = {theta1, (1 - theta1) * theta2, (1 - theta1) * (1 - theta2)};
    // the sub-model OBJECTS are kept over parameter moves: likelihood objects hold pointers to them (getNModel)
    if (sub_.size() != 3) {
      sub_.clear();
      for (int k = 0; k < 3; ++k) sub_.emplace_back(new YN98(alpha_, kappa, omega[k], codonFreq_.empty() ? nullptr : &codonFreq_));
    } else {
      for (int k = 0; k < 3; ++k) {
        sub_[k]->setRate(1.0);
        sub_[k]->setParameterValue("kappa", kappa);
        sub_[k]->setParameterValue("omega", omega[k]);
      }
    }
    size_t from = 0, to = 0;
    bool found = false;
    for (size_t f = 1; f < 64 && !found; ++f)
      for (size_t t = 0; t < f && !found; ++t)
        if (CodonAlphabet::aminoAcid((int)f) == CodonAlphabet::aminoAcid((int)t) && !CodonAlphabet::isStop((int)f) &&
            sub_[0]->getGenerator()(f, t) != 0 && sub_[1]->getGenerator()(f, t) != 0) {
          from = f;
          to = t;
          found = true;
        }
    if (!found) throw Exception("Impossible to find synonymous codons");
    double r[3], mean = 0;
    for (int k = 0; k < 3; ++k) { r[k] = 1.0 / sub_[k]->getGenerator()(from, to); mean += probs_[k] * r[k]; }
    for (int k = 0; k < 3; ++k) sub_[k]->setRate(r[k] / mean);
  }
  const Alphabet* alpha_;
  Vdouble codonFreq_;
  std::vector<std::unique_ptr<YN98> > sub_;
  Vdouble probs_;
};
// Model/Codon/YNGP_M2.cpp:52-146: omega in {omega0 < 1, 1, omega2 > 1}
class YNGP_M2 : public OmegaMixture_ {
 public:
  YNGP_M2(const Alphabet* alpha, double kappa = 1., double omega0 = 0.5, double omega2 = 2., double theta1 = 0.333333, double theta2 = 0.5,
          const Vdouble* codonFreq = nullptr)
      : OmegaMixture_(alpha, codonFreq), kappa_(kappa), omega0_(omega0), omega2_(omega2), theta1_(theta1), theta2_(theta2) { update(); }
  std::string getName() const { return "YNGP_M2"; }
  std::vector<std::string> getParameterNames() const { return {"YNGP_M2.kappa", "YNGP_M2.omega0", "YNGP_M2.omega2", "YNGP_M2.theta1", "YNGP_M2.theta2"}; }
  double getParameterValue(const std::string& name) const { return *slot(name); }
  void setParameterValue(const std::string& name, double v) { *const_cast<double*>(slot(name)) = v; update(); }

 private:
  const double* slot(const std::string& name) const {
    const std::string n = name.substr(name.find('.') == std::string::npos ? 0 : name.find('.') + 1);
    const std::map<std::string, const double*> m = {{"kappa", &kappa_}, {"omega0", &omega0_}, {"omega2", &omega2_}, {"theta1", &theta1_}, {"theta2", &theta2_}};
    if (!m.count(n)) throw ParameterNotFoundException(name);
    return m.at(n);
  }
  void update() { const double w[3] = {omega0_, 1.0, omega2_}; rebuild(kappa_, w, theta1_, theta2_); }
  double kappa_, omega0_, omega2_, theta1_, theta2_;
};
// fork, Model/Codon/RELAX.cpp:52-218: omegas ((p omega1)^k, omega1^k, omega2^k), floored at 0.001 / capped at 999 (:176-205)
class RELAX : public OmegaMixture_ {
 public:
  RELAX(const Alphabet* alpha, double kappa = 1., double p = 0.5, double omega1 = 1., double omega2 = 2., double k = 1.,
        double theta1 = 0.333333, double theta2 = 0.5, const Vdouble* codonFreq = nullptr)
      : OmegaMixture_(alpha, codonFreq), kappa_(kappa), p_(p), omega1_(omega1), omega2_(omega2), k_(k), theta1_(theta1), theta2_(theta2) { update(); }
  std::string getName() const { return "RELAX"; }
  std::vector<std::string> getParameterNames() const {
    return {"RELAX.kappa", "RELAX.p", "RELAX.omega1", "RELAX.omega2", "RELAX.k", "RELAX.theta1", "RELAX.theta2"};
  }
  double getParameterValue(const std::string& name) const { return *slot(name); }
  void setParameterValue(const std::string& name, double v) { *const_cast<double*>(slot(name)) = v; update(); }

 private:
  const double* slot(const std::string& name) const {
    const std::string n = name.substr(name.find('.') == std::string::npos ? 0 : name.find('.') + 1);
    const std::map<std::string, const double*> m = {{"kappa", &kappa_}, {"p", &p_}, {"omega1", &omega1_}, {"omega2", &omega2_},
                                                     {"k", &k_}, {"theta1", &theta1_}, {"theta2", &theta2_}};
    if (!m.count(n)) throw ParameterNotFoundException(name);
    return m.at(n);
  }
  void update() {
    const double w[3] = {std::max(std::pow(p_ * omega1_, k_), 0.001), std::max(std::pow(omega1_, k_), 0.001), std::min(std::pow(omega2_, k_), 999.0)};
    rebuild(kappa_, w, theta1_, theta2_);
  }
  double kappa_, p_, omega1_, omega2_, k_, theta1_, theta2_;
};

// Model/MixedSubstitutionModelSet.h: mixed models on groups of branches; the site paths ("hyper-nodes") supported here are the
// ones test/test_relax.cpp:100-102 sets up -- sub-model k of every model travels together, with the first model's probability.
class MixedSubstitutionModelSet {
 public:
  explicit MixedSubstitutionModelSet(const Alphabet* alpha) : alphabet_(alpha) {}
  void addModel(MixedSubstitutionModel* model, const std::vector<int>& nodesId) {   // owns the model
    if (!models_.empty() && model->getNumberOfModels() != models_[0]->getNumberOfModels()) {
      delete model;
      throw Exception("MixedSubstitutionModelSet: every model needs the same number of sub-models for linked site paths");
    }
    for (int id : nodesId) nodeToModel_[id] = models_.size();
    models_.emplace_back(model);
  }
  size_t getNumberOfModels() const { return models_.size(); }
  MixedSubstitutionModel* getModel(size_t i) const { return models_.at(i).get(); }
  size_t getNumberOfPaths() const { return models_.at(0)->getNumberOfModels(); }
  double getPathProbability(size_t k) const { return models_.at(0)->getNProbability(k); }
  size_t getModelIndexForNode(int nodeId) const {
    std::map<int, size_t>::const_iterator it = nodeToModel_.find(nodeId);
    if (it == nodeToModel_.end()) throw Exception("MixedSubstitutionModelSet: no model associated to node with id " + std::to_string(nodeId));
    return it->second;
  }
  const Alphabet* getAlphabet() const { return alphabet_; }

 private:
  const Alphabet* alphabet_;
  std::vector<std::unique_ptr<MixedSubstitutionModel> > models_;
  std::map<int, size_t> nodeToModel_;
};

// ---- root frequency sets and non-homogeneous model sets ---------------------------------------------------------------------------
// Model/FrequencySet/NucleotideFrequencySet.h: GCFrequencySet (one parameter theta = G+C content), FixedFrequencySet
class FrequencySet {
 public:
  virtual ~FrequencySet() {}
  virtual FrequencySet* clone() const = 0;
  virtual const Vdouble& getFrequencies() const = 0;
  virtual std::vector<std::string> getParameterNames() const = 0;
  virtual double getParameterValue(const std::string& name) const = 0;
  virtual void setParameterValue(const std::string& name, double v) = 0;
};
class GCFrequencySet : public FrequencySet {
 public:
  explicit GCFrequencySet(const Alphabet* = nullptr, double theta = 0.5) : freq_(4) { set(theta); }
  GCFrequencySet* clone() const { return new GCFrequencySet(*this); }
  const Vdouble& getFrequencies() const { return freq_; }
  std::vector<std::string> getParameterNames() const { return {"GC.theta"}; }
  double getParameterValue(const std::string& name) const { if (name != "GC.theta" && name != "theta") throw ParameterNotFoundException(name); return theta_; }
  void setParameterValue(const std::string& name, double v) { if (name != "GC.theta" && name != "theta") throw ParameterNotFoundException(name); set(v); }

 private:
  void set(double theta) { theta_ = theta; freq_[0] = freq_[3] = (1 - theta) / 2; freq_[1] = freq_[2] = theta / 2; }
  double theta_;
  Vdouble freq_;
};
class FixedFrequencySet : public FrequencySet {
 public:
  explicit FixedFrequencySet(const Vdouble& f) : freq_(f) {}
  FixedFrequencySet* clone() const { return new FixedFrequencySet(*this); }
  const Vdouble& getFrequencies() const { return freq_; }
  std::vector<std::string> getParameterNames() const { return {}; }
  double getParameterValue(const std::string& name) const { throw ParameterNotFoundException(name); }
  void setParameterValue(const std::string& name, double) { throw ParameterNotFoundException(name); }

 private:
  Vdouble freq_;
};

// Model/SubstitutionModelSet.h: models attached to the branches above given node ids, root frequencies, parameters named
// "<model parameter>_<model index + 1>" with aliases (SubstitutionModelSet::aliasParameters).  The set owns its models and
// its root frequency set, like the reference.
class SubstitutionModelSet {
 public:
  explicit SubstitutionModelSet(const Alphabet* alpha) : alphabet_(alpha) {}
  SubstitutionModelSet(const SubstitutionModelSet& o) : alphabet_(o.alphabet_), nodeToModel_(o.nodeToModel_), aliases_(o.aliases_) {
    for (const auto& m : o.models_) models_.emplace_back(m->clone());
    if (o.rootFreqs_) rootFreqs_.reset(o.rootFreqs_->clone());
  }
  SubstitutionModelSet& operator=(const SubstitutionModelSet&) = delete;
  SubstitutionModelSet* clone() const { return new SubstitutionModelSet(*this); }
  const Alphabet* getAlphabet() const { return alphabet_; }
  void setRootFrequencies(FrequencySet* f) { rootFreqs_.reset(f); }
  const FrequencySet* getRootFrequencySet() const { return rootFreqs_.get(); }
  bool isStationary() const { return !rootFreqs_; }
  // SubstitutionModelSet::getRootFrequencies: the root set, or (stationary sets) the first model's equilibrium frequencies
  Vdouble getRootFrequencies() const { return rootFreqs_ ? rootFreqs_->getFrequencies() : models_.at(0)->getFrequencies(); }
  void addModel(SubstitutionModel* model, const std::vector<int>& nodesId) {
    std::unique_ptr<SubstitutionModel> own(model);
    if (!models_.empty() && model->getNumberOfStates() != models_[0]->getNumberOfStates())
      throw Exception("SubstitutionModelSet::addModel. A Substitution Model cannot be added to a Model Set if it does not have the same number of states.");
    for (int id : nodesId) {
      if (nodeToModel_.count(id)) throw Exception("SubstitutionModelSet::addModel. Node " + std::to_string(id) + " already has a model.");
      nodeToModel_[id] = models_.size();
    }
    models_.push_back(std::move(own));
  }
  size_t getNumberOfModels() const { return models_.size(); }
  size_t getNumberOfStates() const { return models_.at(0)->getNumberOfStates(); }
  SubstitutionModel* getModel(size_t i) const { return models_.at(i).get(); }
  size_t getModelIndexForNode(int nodeId) const {
    std::map<int, size_t>::const_iterator it = nodeToModel_.find(nodeId);
    if (it == nodeToModel_.end()) throw Exception("SubstitutionModelSet::getModelIndexForNode(). No model associated to node with id " + std::to_string(nodeId));
    return it->second;
  }
  SubstitutionModel* getModelForNode(int nodeId) const { return getModel(getModelIndexForNode(nodeId)); }
  std::vector<int> getNodesWithModel(size_t i) const {
    std::vector<int> v;
    for (const auto& kv : nodeToModel_) if (kv.second == i) v.push_back(kv.first);
    return v;
  }
  // every node of the tree but the root has a model, and only those (SubstitutionModelSet::isFullySetUpFor)
  bool isFullySetUpFor(const Tree& tree) const {
    const std::vector<Node*> nodes = tree.getNodes();
    for (size_t i = 0; i + 1 < nodes.size(); ++i) if (!nodeToModel_.count(nodes[i]->getId())) return false;
    return !models_.empty();
  }
  // `to` follows `from` from now on (both full names, e.g. "T92.kappa_1", "T92.kappa_2")
  void aliasParameters(const std::string& from, const std::string& to) {
    aliases_[from].push_back(to);
    setParameterValue(to, getParameterValue(from));
  }
  // independent parameters: root frequencies first, then the model parameters that are not aliased to another one
  std::vector<std::string> getParameterNames() const {
    std::vector<std::string> names;
    std::map<std::string, bool> follower;
    for (const auto& kv : aliases_) for (const std::string& t : kv.second) follower[t] = true;
    if (rootFreqs_) for (const std::string& n : rootFreqs_->getParameterNames()) if (!follower.count(n)) names.push_back(n);
    for (size_t k = 0; k < models_.size(); ++k)
      for (const std::string& n : models_[k]->getParameterNames()) {
        const std::string full = n + "_" + std::to_string(k + 1);
        if (!follower.count(full)) names.push_back(full);
      }
    return names;
  }
  double getParameterValue(const std::string& name) const {
    size_t k;
    std::string base;
    if (splitName(name, base, k)) return models_[k]->getParameterValue(base);
    if (rootFreqs_) return rootFreqs_->getParameterValue(name);
    throw ParameterNotFoundException("ParameterNotFoundException: " + name);
  }
  void setParameterValue(const std::string& name, double v) {
    size_t k;
    std::string base;
    if (splitName(name, base, k)) models_[k]->setParameterValue(base, v);
    else if (rootFreqs_) rootFreqs_->setParameterValue(name, v);
    else throw ParameterNotFoundException("ParameterNotFoundException: " + name);
    std::map<std::string, std::vector<std::string> >::const_iterator it = aliases_.find(name);
    if (it != aliases_.end()) for (const std::string& t : it->second) setParameterValue(t, v);
  }

 private:
  bool splitName(const std::string& name, std::string& base, size_t& k) const {
    const size_t u = name.rfind('_');
    if (u == std::string::npos || u + 1 >= name.size()) return false;
    char* end = nullptr;
    const long idx = std::strtol(name.c_str() + u + 1, &end, 10);
    if (*end != 0 || idx < 1 || (size_t)idx > models_.size()) return false;
    base = name.substr(0, u);
    k = (size_t)idx - 1;
    return true;
  }
  const Alphabet* alphabet_;
  std::vector<std::unique_ptr<SubstitutionModel> > models_;
  std::map<int, size_t> nodeToModel_;
  std::unique_ptr<FrequencySet> rootFreqs_;
  std::map<std::string, std::vector<std::string> > aliases_;
};

namespace SubstitutionModelSetTools {
// Model/SubstitutionModelSetTools.cpp:78-183: one copy of `model` per branch (model k + 1 on the k-th node of
// tree.getNodesId() with the root removed), the listed global parameters aliased to the first copy's; takes ownership of
// `model` (deleted, like the reference) and of `rootFreqs`.
inline SubstitutionModelSet* createNonHomogeneousModelSet(SubstitutionModel* model, FrequencySet* rootFreqs, const Tree* tree,
                                                          const std::vector<std::string>& globalParameterNames) {
  std::unique_ptr<SubstitutionModel> tmpl(model);
  const std::vector<std::string> modelParams = model->getParameterNames();
  for (const std::string& g : globalParameterNames)
    if (std::find(modelParams.begin(), modelParams.end(), g) == modelParams.end())
      throw Exception("SubstitutionModelSetTools::createNonHomogeneousModelSet. Parameter '" + g + "' is not valid.");
  SubstitutionModelSet* set = new SubstitutionModelSet(model->getAlphabet());
  if (rootFreqs) set->setRootFrequencies(rootFreqs);
  std::vector<int> ids = tree->getNodesId();
  const int rootId = tree->getRootNode()->getId();
  ids.erase(std::find(ids.begin(), ids.end(), rootId));
  for (int id : ids) set->addModel(model->clone(), std::vector<int>(1, id));
  for (const std::string& g : globalParameterNames)
    for (size_t i = 1; i < ids.size(); ++i) set->aliasParameters(g + "_1", g + "_" + std::to_string(i + 1));
  return set;
}
}  // namespace SubstitutionModelSetTools

}  // namespace bppshim
