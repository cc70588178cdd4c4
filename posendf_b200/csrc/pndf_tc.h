// pndf_tc.h -- host interface of the tensor-core DFNet path (pndf_tc.cu), used by pndf_capi.cu.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/pndf.h"

namespace pndf {

struct TcState;
struct KParams;          // pndf_kernel.cuh

int tc_create(TcState** out, const pndf_config* cfg);
void tc_destroy(TcState* s);
// split the flat fp32 parameter vector (reference order, device pointer) into the tf32 hi / lo weight copies; stream-ordered
int tc_set_weights(TcState* s, const float* flat_dev, cudaStream_t st);
// forward (want_grad = 0), forward + gradient, or a.steps projection steps over a.B poses, all in one pass; the weights come from
// this state, the biases, lin6 and the encoder from a, and the previous denoise step's Adam update from a.dn when it is pending
// (prior mode: axis-angle input, one evaluation, no step).  *launches is increased by the kernels launched
int tc_run(TcState* s, const KParams& a, int want_grad, cudaStream_t st, int64_t* launches);
// make sure the activation buffers hold B poses (allocates: call it BEFORE a stream capture that contains tc_run)
int tc_reserve(TcState* s, long long B);
const char* tc_last_error(TcState* s);

}  // namespace pndf
