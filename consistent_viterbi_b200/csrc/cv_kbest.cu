// cv_kbest.cu -- exact k-best (list) Viterbi decoding (cv_decode_batch_kbest): the k highest-scoring state paths of every
// sequence under the plain decode's recurrence.
#include "cv_internal.cuh"

#include "kbest.cuh"

using namespace cvb;

#include "kbest_host.inl"
