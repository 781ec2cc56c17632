// bppgpu_shim.hpp -- C++ host side above the C ABI (include/bppgpu.h), mirroring the reference's class surface for
// the tree-likelihood hot path so that code written against bpp-phyl reads the same:
//
//   reference (src/Bpp/Phyl/...)                                   here (namespace bppshim)
//   Model/SubstitutionModel.h:195-525  TransitionModel / SubstitutionModel   SubstitutionModel (getPij_t ... on the GPU)
//   Model/AbstractSubstitutionModel.cpp:175-421  updateMatrices                AbstractSubstitutionModel::updateMatrices (host)
//   Model/Nucleotide/{JCnuc,K80,HKY85,T92,GTR}.cpp, Model/Protein/LG08.cpp    same names
//   Model/Codon/YN98.cpp (+ AbstractWord/Codon*SubstitutionModel)              YN98
//   Model/ChromosomeSubstitutionModel.cpp:431-802                              ChromosomeSubstitutionModel
//   Model/RateDistribution/{Constant,GammaDiscrete}RateDistribution.h          same names
//   TreeTemplate.h / TreeTemplateTools (parenthesisToTree, unroot, getNodes)   TreeTemplate<Node>, TreeTemplateTools
//   SitePatterns.cpp:52-106                                                    SitePatterns (via bppgpu_site_patterns)
//   Distance/{DistanceMatrix.h,DistanceEstimation,BioNJ}.cpp                   same names (distances on the device, BIONJ on the host)
//   Parsimony/DRTreeParsimonyScore.cpp, OptimizationTools::optimizeTreeNNI     same names (scores and NNI changes on the device)
//   Likelihood/{R,DR}HomogeneousTreeLikelihood, DRNonHomogeneousTreeLikelihood same names; computeTreeLikelihood,
//       fireParameterChanged, getValue, get{First,Second}OrderDerivative ... run on the device through libbppgpu
//
// Only what the hot path needs is here (SURVEY.md section 8); bpp-core / bpp-seq types the signatures mention are
// reduced to minimal stand-ins (RowMatrix, Alphabet, VectorSiteContainer, DiscreteDistribution, ParameterList-like
// name/value access).  There is no CPU fallback: every evaluation goes through the C ABI and throws bppshim::Exception
// with the library's message when no B200 is usable.
#pragma once
// The classes live in shim/: core.hpp (bpp-core stand-ins, host linear algebra) <- seq.hpp (alphabets, containers) <- tree.hpp
// <- io.hpp (Newick, Fasta, Phylip, chrFasta readers) <- models.hpp (rate distributions, substitution models, model sets) <- likelihood.hpp (SitePatterns, tree likelihoods)
// <- ancestral.hpp (reconstruction classes) <- optimizers.hpp (batched Brent, ChromosomeNumberOptimizer, PseudoNewtonOptimizer);
// likelihood.hpp <- distance.hpp (DistanceMatrix, DistanceEstimation, BioNJ); likelihood.hpp <- parsimony.hpp (DRTreeParsimonyScore,
// OptimizationTools::optimizeTreeNNI).
#include "shim/optimizers.hpp"
#include "shim/distance.hpp"
#include "shim/parsimony.hpp"
