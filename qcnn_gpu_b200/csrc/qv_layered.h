// Host-visible interface of the per-layer CUDA-core path (qv_layered.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "qv_internal.h"

namespace qv {

// One handle's layered path: its weights in the kernels' word layouts, the activation scratch (min(batch, 8) frames of H x W),
// the row-window buffer, and one event that orders every use of the two: each call below waits for the previous one, on
// whatever stream that ran.  Calls that return int return a QV_* code and set the message.
struct LayeredNet;

cudaError_t layered_create(LayeredNet **out, int batch, int H, int W);   // *out is set even on failure
void layered_free(LayeredNet *ln);
// Packs and uploads the model's weights and biases, freeing the previous ones; the scratch is kept.
int layered_load(LayeredNet *ln, const ModelHost &m, cudaStream_t st);
// n frames of HxW luma in device memory.  With d_ori and d_sse (both or neither), per frame f the SSE of the input and of the
// output against d_ori are ADDED to d_sse[2f] and d_sse[2f + 1].
int layered_forward(LayeredNet *ln, const uint8_t *d_in, uint8_t *d_out, int n, int H, int W, cudaStream_t st,
                    long long *launches, const uint8_t *d_ori, int64_t *d_sse);
// A window of in_rows rows (at most batch x H) run as an image of its own; its rows [out0, out1) are copied to d_out.
int layered_forward_rows(LayeredNet *ln, const uint8_t *d_in, int in_rows, uint8_t *d_out, int out0, int out1, cudaStream_t st,
                         long long *launches);
// Activation 1 / 2 / 3 of the first frame in the scratch as planar int8 [C][H][W]; synchronises st.
int layered_activation(LayeredNet *ln, int which, int8_t *host_out, cudaStream_t st);
cudaError_t sse_accumulate(const uint8_t *a, const uint8_t *b, size_t n, int64_t *d_accum, cudaStream_t st);

}  // namespace qv
