// Host side of the strip partition (qv_strip.cu): one frame in horizontal strips on several GPUs, each strip reading its
// halo rows from its neighbours' memory.  Calls that return int return a QV_* code and set the message.
#pragma once
#include "qv_fused.h"

namespace qv {

constexpr int STRIP_HALO = 6;   // receptive-field radius of the net: 2 + 2 + 1 + 1 rows

struct StripNet;                               // one strip of this process
struct StripRows { int img_h, row0, row1; };   // rows [row0, row1) of an img_h-row frame

int strip_create(StripNet **out, int dev, int W, int img_h, int row0, int row1);   // dev: the current device
void strip_free(StripNet *s);   // also unlinks it from the strips of this process that have it attached
StripRows strip_rows(const StripNet *s);
uint8_t *strip_slot(const StripNet *s, int slot);
int strip_export(const StripNet *s, qv_strip_desc *out);
int strip_attach(StripNet *s, int side, const qv_strip_desc *neighbour);
// Strips that share a GPU are driven on one stream, all loads of a frame before its forwards; anything else is refused.
int strip_acquire(StripNet *s, int slot, const FusedModel *fm, cudaStream_t st, long long *launches);
int strip_ready(const StripNet *s, const char *who);   // a neighbour on every interior edge
int strip_forward(StripNet *s, int slot, const FusedModel *fm, const uint8_t *d_ori, uint8_t *d_out, int64_t *d_sse,
                  cudaStream_t st, long long *launches, const char *who);
// A call that drives s[0, n) itself: refuses a device of theirs holding another strip; unbind forgets their streams.
int strip_claim(StripNet *const *s, int n, const char *who);
void strip_unbind(StripNet *const *s, int n);

}  // namespace qv
