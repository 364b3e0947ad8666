// Declarations of the four bootstrap .Call entry points with the SEXP signatures that integration/scde_b200_shim.cpp
// defines, under the name of the reference's header, so that oracle/shim/ref_entry.cpp compiles into the shim build
// (integration/Makefile) without the reference's sources.
#pragma once
#include <RcppArmadillo.h>

RcppExport SEXP logBootPosterior(SEXP Models, SEXP Ucl, SEXP CountsI, SEXP Magnitudes, SEXP Nboot, SEXP Seed,
                                 SEXP ReturnIndividualPosteriors, SEXP LocalThetaFit, SEXP SquareLogitConc,
                                 SEXP EnsembleProbability);
RcppExport SEXP logBootBatchPosterior(SEXP Models, SEXP Ucl, SEXP CountsI, SEXP Magnitudes, SEXP BatchIL, SEXP Composition,
                                      SEXP Nboot, SEXP Seed, SEXP ReturnIndividualPosteriors, SEXP LocalThetaFit,
                                      SEXP SquareLogitConc);
RcppExport SEXP jpmatLogBoot(SEXP Matl, SEXP Nboot, SEXP Seed);
RcppExport SEXP jpmatLogBatchBoot(SEXP Matll, SEXP Comp, SEXP Nboot, SEXP Seed);
