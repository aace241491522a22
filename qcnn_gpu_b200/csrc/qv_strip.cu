// Spatial strips over several GPUs (SURVEY 8e-ii).  One cudaMalloc'ed block per strip: a 256-byte header (published /
// completed sequence numbers, CTA counter) and two input slots holding this GPU's rows of the frame.  The block is what
// neighbours map (same process: peer access; other process: CUDA IPC) and read their 6 halo rows from, over NVLink.
#include <algorithm>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <random>
#include <unistd.h>

#include "qv_strip.h"

namespace qv {

constexpr size_t STRIP_HDR = 256, STRIP_PUB = 0, STRIP_DONE = 64, STRIP_CTR = 128;
constexpr uint32_t STRIP_MAGIC = 0x51565354u;   // "QVST"
struct StripDescImpl {                          // the content of qv_strip_desc
    uint32_t magic;
    int32_t dev, row0, row1, width, img_h;
    uint64_t nonce;                             // identifies the exporting process
    uint64_t slot_off, slot_stride;
    uint64_t id;                                // the exporting strip (meaningful inside the exporting process only)
    cudaIpcMemHandle_t ipc;
    char pci[16];                               // PCI bus id of the device: device ordinals differ between processes
};
static_assert(sizeof(StripDescImpl) <= sizeof(qv_strip_desc), "qv_strip_desc too small");
static uint64_t process_nonce()   // on first use: a process forked before that gets a nonce of its own
{
    static const uint64_t n = [] { std::random_device rd; return ((uint64_t)rd() << 32) ^ (uint64_t)rd() ^ ((uint64_t)getpid() << 17); }();
    return n;
}
struct StripPeer {
    uint8_t *base = nullptr;                    // the neighbour's block; null: no neighbour attached
    StripNet *net = nullptr;                    // same process only
    bool ipc = false, same_device = false;
    StripDescImpl d{};
};
struct StripNet {
    int dev = 0, W = 0, img_h = 0, row0 = 0, row1 = 0;
    uint64_t id = 0;
    uint8_t *block = nullptr;
    size_t slot_stride = 0;
    uint32_t seq = 0, slot_seq[2] = {0, 0};
    uint32_t fills[2] = {0, 0}, forwards[2] = {0, 0};   // per slot: how often acquired for filling / consumed
    cudaStream_t last_stream = nullptr;         // null: not driven since strip_create / strip_unbind
    StripPeer peer[2];                          // QV_STRIP_ABOVE, QV_STRIP_BELOW
    ~StripNet() { for (StripPeer &p : peer) if (p.ipc) cudaIpcCloseMemHandle(p.base); cudaFree(block); }
};

// The strips of this process, per device.  Kernels that wait for one another must never share a GPU (nothing guarantees that
// two launches on one GPU run at the same time), so strips on the SAME device are ordered by the one stream they are driven
// on instead.  What one strip reads or writes of another (last_stream, fills, forwards, the peer links) is under g_mu.
static std::mutex g_mu;
static std::map<int, std::vector<StripNet *>> g_strips;
static uint64_t g_last_id = 0;
// Both under g_mu.
static int check_stream(const StripNet *s, cudaStream_t st, const char *who)
{
    for (const StripNet *o : g_strips[s->dev])
        if (o != s && o->last_stream && o->last_stream != st) {
            set_error("%s: several strips live on GPU %d: drive all of them on ONE caller-provided stream (kernels of different launches "
                      "must not wait for each other on one GPU, so stream order is what orders them)", who, s->dev);
            return QV_ERR_STATE;
        }
    return QV_OK;
}
static int check_neighbours(const StripNet *s, const char *who)
{
    if ((s->row0 == 0 || s->peer[QV_STRIP_ABOVE].base) && (s->row1 == s->img_h || s->peer[QV_STRIP_BELOW].base)) return QV_OK;
    set_error("%s: rows [%d, %d) of %d have an interior edge with no neighbour attached", who, s->row0, s->row1, s->img_h);
    return QV_ERR_STATE;
}

int strip_create(StripNet **out, int dev, int W, int img_h, int row0, int row1)
{
    std::unique_ptr<StripNet> s(new StripNet);
    s->dev = dev; s->W = W; s->img_h = img_h; s->row0 = row0; s->row1 = row1;
    s->slot_stride = ((size_t)(row1 - row0) * W + 255) / 256 * 256;
    QV_CUDA(cudaMalloc(&s->block, STRIP_HDR + 2 * s->slot_stride));
    QV_CUDA(cudaMemset(s->block, 0, STRIP_HDR));
    QV_CUDA(cudaDeviceSynchronize());
    std::lock_guard<std::mutex> l(g_mu);
    s->id = ++g_last_id;
    g_strips[dev].push_back(*out = s.release());
    return QV_OK;
}

void strip_free(StripNet *s)
{
    std::unique_lock<std::mutex> l(g_mu);
    auto &v = g_strips[s->dev];
    v.erase(std::find(v.begin(), v.end(), s));
    for (auto &dv : g_strips)
        for (StripNet *o : dv.second)
            for (StripPeer &p : o->peer)
                if (p.net == s) p = StripPeer{};
    l.unlock();
    delete s;
}

StripRows strip_rows(const StripNet *s) { return {s->img_h, s->row0, s->row1}; }
uint8_t *strip_slot(const StripNet *s, int slot) { return s->block + STRIP_HDR + (size_t)slot * s->slot_stride; }
int strip_ready(const StripNet *s, const char *who) { std::lock_guard<std::mutex> l(g_mu); return check_neighbours(s, who); }

int strip_export(const StripNet *s, qv_strip_desc *out)
{
    StripDescImpl d{};
    d.magic = STRIP_MAGIC; d.dev = s->dev; d.row0 = s->row0; d.row1 = s->row1; d.width = s->W; d.img_h = s->img_h;
    d.nonce = process_nonce(); d.slot_off = STRIP_HDR; d.slot_stride = s->slot_stride; d.id = s->id;
    QV_CUDA(cudaIpcGetMemHandle(&d.ipc, s->block));
    QV_CUDA(cudaDeviceGetPCIBusId(d.pci, (int)sizeof(d.pci), s->dev));
    memset(out, 0, sizeof(*out));
    memcpy(out, &d, sizeof(d));
    return QV_OK;
}

int strip_attach(StripNet *s, int side, const qv_strip_desc *neighbour)
{
    StripPeer P, old;
    StripDescImpl &d = P.d;
    memcpy(&d, neighbour, sizeof(d));
    if (d.magic != STRIP_MAGIC) { set_error("qv_strip_attach: not a strip descriptor"); return QV_ERR_ARG; }
    if (d.width != s->W || d.img_h != s->img_h) { set_error("qv_strip_attach: the neighbour's frame is %dx%d, this one %dx%d", d.width, d.img_h, s->W, s->img_h); return QV_ERR_ARG; }
    if (side == QV_STRIP_ABOVE ? d.row1 != s->row0 : d.row0 != s->row1) {
        set_error("qv_strip_attach: rows [%d, %d) are not adjacent %s rows [%d, %d)", d.row0, d.row1, side == QV_STRIP_ABOVE ? "above" : "below", s->row0, s->row1);
        return QV_ERR_ARG;
    }
    if (d.row1 - d.row0 < STRIP_HALO) {
        // the halo would reach into the strip after next, which this protocol does not exchange
        set_error("qv_strip_attach: the neighbour holds %d rows, fewer than the %d-row halo (use fewer strips)", d.row1 - d.row0, STRIP_HALO);
        return QV_ERR_ARG;
    }
    // the old neighbour is forgotten whether or not the new one can be attached; the CUDA calls run outside the lock
    { std::lock_guard<std::mutex> l(g_mu); std::swap(old, s->peer[side]); }
    if (old.ipc) cudaIpcCloseMemHandle(old.base);
    char my_pci[16] = {0};
    QV_CUDA(cudaDeviceGetPCIBusId(my_pci, (int)sizeof(my_pci), s->dev));
    P.same_device = strncmp(my_pci, d.pci, sizeof(my_pci)) == 0;
    const bool local = d.nonce == process_nonce();   // same process: plain peer access to the neighbour's block
    if (local && d.dev != s->dev) {
        int can = 0;
        QV_CUDA(cudaDeviceCanAccessPeer(&can, s->dev, d.dev));
        if (!can) { set_error("qv_strip_attach: device %d cannot map memory of device %d (no peer access)", s->dev, d.dev); return QV_ERR_CUDA; }
        const cudaError_t e = cudaDeviceEnablePeerAccess(d.dev, 0);
        if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError(); else QV_CUDA(e);
    } else if (!local) {
        if (P.same_device) {
            // two processes time-slicing one GPU: a kernel of one that waits for a kernel of the other may never see it run
            set_error("qv_strip_attach: the neighbour strip belongs to another process on the SAME GPU; strips of different processes must be on different GPUs");
            return QV_ERR_ARG;
        }
        void *p = nullptr;
        QV_CUDA(cudaIpcOpenMemHandle(&p, d.ipc, cudaIpcMemLazyEnablePeerAccess));
        P.base = (uint8_t *)p;
        P.ipc = true;
    }
    std::lock_guard<std::mutex> l(g_mu);
    if (local)   // linked while it exists: strip_free unlinks it
        for (StripNet *o : g_strips[d.dev])
            if (o->id == d.id) { P.net = o; P.base = o->block; }
    if (!P.base) { set_error("qv_strip_attach: the neighbour strip was released (export it again after its qv_strip_setup)"); return QV_ERR_STATE; }
    s->peer[side] = P;
    return QV_OK;
}

int strip_acquire(StripNet *s, int slot, const FusedModel *fm, cudaStream_t st, long long *launches)
{
    const uint32_t *w[2] = {nullptr, nullptr};
    uint32_t seq;
    {
        std::lock_guard<std::mutex> l(g_mu);
        if (int rc = check_stream(s, st, "qv_strip_acquire")) return rc;
        s->last_stream = st;
        seq = s->slot_seq[slot];
        for (int side = 0; side < 2; ++side) {
            const StripPeer &P = s->peer[side];
            if (!P.base || seq == 0) continue;
            if (!P.same_device) {
                w[side] = reinterpret_cast<const uint32_t *>(P.base + STRIP_DONE);   // another GPU: wait for its "completed step seq"
            } else if (P.net->forwards[slot] < s->forwards[slot]) {
                // the neighbour's forward that read this slot must already be on the (shared) stream
                set_error("qv_strip_acquire: the neighbour strip on the same GPU has not yet consumed slot %d (issue the strips' calls frame by frame)", slot);
                return QV_ERR_STATE;
            }
        }
    }
    if (w[0] || w[1]) {   // seq != 0: forwarded before, so fm is set.  Outside the lock: a launch may block on a full queue
        QV_CUDA(fused_wait_words(fm, w[0], seq, w[1], seq, st));
        *launches += 1;
    }
    std::lock_guard<std::mutex> l(g_mu);   // only an acquired slot counts as filled
    s->fills[slot] += 1;
    return QV_OK;
}

int strip_forward(StripNet *s, int slot, const FusedModel *fm, const uint8_t *d_ori, uint8_t *d_out, int64_t *d_sse,
                  cudaStream_t st, long long *launches, const char *who)
{
    FusedRows fr;
    {
        std::lock_guard<std::mutex> l(g_mu);
        if (int rc = check_neighbours(s, who)) return rc;
        if (d_sse && s->img_h > FUSED_SSE_MAX_H) { set_error("%s: frame height %d exceeds %d", who, s->img_h, FUSED_SSE_MAX_H); return QV_ERR_ARG; }
        if (int rc = check_stream(s, st, who)) return rc;
        fr.own0 = fr.out0 = s->row0; fr.own1 = fr.out1 = s->row1;
        fr.pub = reinterpret_cast<uint32_t *>(s->block + STRIP_PUB);
        fr.done = reinterpret_cast<uint32_t *>(s->block + STRIP_DONE);
        fr.done_ctr = reinterpret_cast<uint32_t *>(s->block + STRIP_CTR);
        for (int side = 0; side < 2; ++side) {
            if (side == QV_STRIP_ABOVE ? s->row0 == 0 : s->row1 == s->img_h) continue;
            const StripPeer &P = s->peer[side];
            const uint8_t *rows = P.base + P.d.slot_off + (size_t)slot * P.d.slot_stride;
            const uint32_t *flag = reinterpret_cast<const uint32_t *>(P.base + STRIP_PUB);
            if (P.same_device) {
                // a neighbour on this very GPU: no kernel may wait for it -- its rows are ordered before this launch by the
                // shared stream, provided its slot was filled for this frame already (checked here, on the host)
                if (P.net->fills[slot] == 0) {
                    set_error("%s: the neighbour strip on the same GPU has not filled slot %d yet (strips that share a GPU: all loads of a frame, then its forwards, on one stream)", who, slot);
                    return QV_ERR_STATE;
                }
                flag = nullptr;
            }
            if (side == QV_STRIP_ABOVE) { fr.top_rows = STRIP_HALO; fr.d_top = rows + (size_t)(P.d.row1 - P.d.row0 - STRIP_HALO) * s->W; fr.flag_top = flag; }
            else { fr.bot_rows = STRIP_HALO; fr.d_bot = rows; fr.flag_bot = flag; }
        }
        fr.seq = s->slot_seq[slot] = ++s->seq;
        s->forwards[slot] += 1;
        s->last_stream = st;
    }
    return fused_forward(fm, strip_slot(s, slot), d_out, 1, s->img_h, s->W, st, launches, &fr, d_ori, d_sse);
}

int strip_claim(StripNet *const *s, int n, const char *who)
{
    std::lock_guard<std::mutex> l(g_mu);
    for (int i = 0; i < n; ++i)
        for (StripNet *o : g_strips[s[i]->dev])
            if (std::find(s, s + n, o) == s + n) {
                set_error("%s: GPU %d also holds a strip handle that is not in this call (strips that share a GPU are driven "
                          "together, on one stream)", who, s[i]->dev);
                return QV_ERR_STATE;
            }
    return QV_OK;
}

void strip_unbind(StripNet *const *s, int n)
{
    std::lock_guard<std::mutex> l(g_mu);
    for (int i = 0; i < n; ++i) s[i]->last_stream = nullptr;
}

}  // namespace qv
