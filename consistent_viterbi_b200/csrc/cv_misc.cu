// cv_misc.cu -- training: SURVEY.md 8(f) N3 supervised MLE counts (cv_mle, reference src/hmm/hmm.rs:30-62,192-205) and
// Baum-Welch EM (cv_baum_welch).
#include "cv_internal.cuh"

#include <chrono>

#include "common.cuh"
#include "mle.cuh"
#include "bw.cuh"

using namespace cvb;

#include "mle_host.inl"
#include "bw_host.inl"
