// Host-visible interface of the fused tcgen05 path (qv_fused.cu).  fused_upload, fused_forward and fused_forward_list
// return a QV_* code and set the message.
#pragma once
#include <cstdint>
#include <vector>
#include <cuda_runtime.h>

#include "qv_internal.h"

namespace qv {

struct FusedModel;   // device-resident weights / descriptors in the layout the fused kernel wants

// Builds the device image of the model for the fused kernel into *out (untouched on failure).
int fused_upload(const ModelHost &m, cudaStream_t st, FusedModel **out);
void fused_free(FusedModel *fm);
// A row window of ONE frame (spatial partition over several GPUs): the launch produces image rows [out0, out1) into d_out
// (first row = out0) from d_in, which holds image rows [own0, own1); up to 6 rows above / below come from d_top (first row
// = own0 - top_rows) and d_bot (first row = own1) -- typically the neighbour GPUs' memory, peer-mapped -- once the
// neighbours' publish words have reached `seq`.  pub / done / done_ctr are this GPU's own words (any may be null).
struct FusedRows {
    int own0 = 0, own1 = 0, out0 = 0, out1 = 0, top_rows = 0, bot_rows = 0;
    const uint8_t *d_top = nullptr, *d_bot = nullptr;
    const uint32_t *flag_top = nullptr, *flag_bot = nullptr;
    uint32_t *pub = nullptr, *done = nullptr, *done_ctr = nullptr;
    uint32_t seq = 0;
};
// Whole net on n frames of HxW luma resident in device memory, one launch.  With `rows`: n = 1, H = image height.
// With d_ori and d_sse (both or neither): k_enh_sse instead of k_fused, the same reconstruction, and for every frame f of the
// launch the exact sum (anchor - ori)^2 is ADDED to d_sse[2f] and sum (out - ori)^2 to d_sse[2f + 1] (device int64; the
// integer core of vrcnn_data::psnr_pf, inference/yuv_data.cpp:98-112).  d_ori holds the same pixels as d_out (with `rows`:
// rows [out0, out1)).  There is no SSE form of the profiling build or of the opt-in TMA input ring: with QV_FUSED_TMA=1 an
// SSE launch runs the kernel without TMA.  H > FUSED_SSE_MAX_H is refused (QV_ERR_ARG).
constexpr int FUSED_SSE_MAX_H = 66051;     // per-thread column sums are 32-bit: 255^2 * H < 2^32
int fused_forward(const FusedModel *fm, const uint8_t *d_in, uint8_t *d_out, int n, int H, int W, cudaStream_t st,
                  long long *launches, const FusedRows *rows = nullptr, const uint8_t *d_ori = nullptr, int64_t *d_sse = nullptr);
// Frames of any sizes, one model (qv_forward_frame_list_device): k_enh_list, one launch per QV_FRAME_LIST_LAUNCH_MAX frames,
// each adding 1 to *launches.  With d_sse every frame carries d_ori and height <= FUSED_SSE_MAX_H, and the SSE pair of frame j is
// ADDED to d_sse[2j], d_sse[2j + 1]; without it no frame carries d_ori.  Every launch's row line must fit the planner (at most
// 2^30 row iterations).  A list that breaks a rule is refused (QV_ERR_ARG) before any launch.
int fused_forward_list(const FusedModel *fm, const qv_frame_desc *frames, int n, int64_t *d_sse, cudaStream_t st,
                       long long *launches);
// Stream-ordered helper of the strip protocol: spin (bounded) until *a >= va and *b >= vb (either pointer may be null; the
// words live on OTHER GPUs), reporting a timeout through the model's failure word (code 3).
cudaError_t fused_wait_words(const FusedModel *fm, const uint32_t *a, uint32_t va, const uint32_t *b, uint32_t vb, cudaStream_t st);
// After the stream the kernel ran on has been synchronised: 0, or what a CTA reported (1 = an mbarrier wait timed
// out, 2 = shared-memory / TMEM bases other than the operand table was built for, 3 = a neighbour GPU's rows never
// arrived); the report is cleared.  0 for a null fm (no model uploaded yet).
int fused_take_failure(const FusedModel *fm);

// Test hook (no GPU): weight image, per-phase MMA operand table (bases 0) and constants as the host builds them.
void fused_debug_tables(const ModelHost &m, std::vector<uint8_t> &wimg, std::vector<uint32_t> &ops, std::vector<int32_t> &consts);
// test hook: how a launch is dealt out to the persistent CTAs (5 ints per unit: cta, frame, strip column, y0, y1); no GPU needed
int fused_debug_units(int sm_count, int n_frames, int H, int W, int row0, int row1, bool rows_mode, bool allow_linear, std::vector<int> &units, int &grid);
// test hook: the same for one frame-list launch (the frame of a unit is its index in the list)
int fused_debug_list_units(int sm_count, int n_frames, const int *H, const int *W, std::vector<int> &units, int &grid);

}  // namespace qv
