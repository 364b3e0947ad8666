// Declaration of matSlideMult with the SEXP signature that integration/scde_b200_shim.cpp defines (see jpmatLogBoot.h).
#pragma once
#include <RcppArmadillo.h>

RcppExport SEXP matSlideMult(SEXP Mat1, SEXP Mat2);
