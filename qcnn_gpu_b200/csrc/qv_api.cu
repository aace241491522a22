// C ABI of the network object (include/qvrcnn_b200.h): handle lifetime, model loading,
// the reference's load_data / forward_blu / x_rec read-back, and the batched / pipelined
// variants the multi-GPU driver uses.  Mirrors class qvrcnn (inference/qvrcnn.cuh:25-59,
// inference/qvrcnn.cu:4-68,168-242) and the hot loop of testqvrcnn (inference/kernel.cu:86-97).
#include <algorithm>
#include <atomic>
#include <cerrno>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <random>
#include <thread>
#include <vector>

#include <fcntl.h>
#include <unistd.h>

#include <cuda_runtime.h>

#include "qv_fused.h"
#include "qv_internal.h"
#include "qv_layered.h"

using namespace qv;

// ---- spatial strips over several GPUs (SURVEY 8e-ii) ---------------------------------------------------------
// One cudaMalloc'ed block per handle: a 256-byte header (published / completed sequence numbers, CTA counter) and two
// input slots holding this GPU's rows of the frame.  The block is what neighbours map (same process: peer access;
// other process: CUDA IPC) and read their 6 halo rows from, straight out of this GPU's HBM over NVLink.
namespace {
constexpr int STRIP_HALO = 6;                   // receptive-field radius of the net: 2 + 2 + 1 + 1 rows
constexpr size_t STRIP_HDR = 256, STRIP_PUB = 0, STRIP_DONE = 64, STRIP_CTR = 128;
constexpr uint32_t STRIP_MAGIC = 0x51565354u;   // "QVST"
struct StripDescImpl {                          // the content of qv_strip_desc
    uint32_t magic;
    int32_t dev, row0, row1, width, img_h;
    uint64_t nonce;                             // identifies the exporting process
    uint64_t base, slot_off, slot_stride;
    uint64_t net;                               // the exporting handle (meaningful inside the exporting process only)
    cudaIpcMemHandle_t ipc;
    char pci[16];                               // PCI bus id of the device: device ordinals differ between processes
};
static_assert(sizeof(StripDescImpl) <= sizeof(qv_strip_desc), "qv_strip_desc too small");
struct StripPeer {
    bool attached = false, ipc = false, same_device = false;
    uint8_t *base = nullptr;
    qv_net *net = nullptr;                      // same process only
    StripDescImpl d{};
};
struct StripState {
    bool on = false;
    int img_h = 0, row0 = 0, row1 = 0;
    uint8_t *block = nullptr;
    size_t slot_stride = 0;
    uint32_t seq = 0, slot_seq[2] = {0, 0};
    uint32_t fills[2] = {0, 0}, forwards[2] = {0, 0};   // per slot: how often acquired for filling / consumed (ordering checks between strips that share a GPU)
    cudaStream_t last_stream = nullptr;
    bool used = false;
    StripPeer peer[2];                          // QV_STRIP_ABOVE, QV_STRIP_BELOW
};
// Strip-mode handles of this process, per device.  Kernels that wait for one another must never share a GPU (nothing
// guarantees that two launches on one GPU run at the same time), so strips that live on the SAME device are ordered by
// the stream they are driven on instead: one stream for all of them, all loads of a frame before its forwards (checked).
std::mutex g_strip_mu;
std::vector<qv_net *> g_strip_nets[64];
uint64_t process_nonce()
{
    static const uint64_t n = [] {
        std::random_device rd;
        return ((uint64_t)rd() << 32) ^ (uint64_t)rd() ^ ((uint64_t)getpid() << 17);
    }();
    return n;
}
}  // namespace

struct qv_net {
    StripState strip;
    int dev = 0, batch = 0, H = 0, W = 0;
    cudaStream_t st = nullptr;
    cudaStream_t pst[2] = {nullptr, nullptr};      // pipeline slots of qv_forward_frames_host
    uint8_t *d_x = nullptr, *d_rec = nullptr;      // InputLayer::x / x_rec   (inference/cnn.cu:433-434)
    uint8_t *d_slot_in[2] = {nullptr, nullptr}, *d_slot_out[2] = {nullptr, nullptr};
    uint8_t *h_pin_in[2] = {nullptr, nullptr}, *h_pin_out[2] = {nullptr, nullptr};
    ModelHost model;
    LayeredNet *ln = nullptr;
    FusedModel *fm = nullptr;
    bool uploaded = false;
    int impl = QV_IMPL_AUTO;
    long long launches = 0;
};

static int set_device(const qv_net *net) { QV_CUDA(cudaSetDevice(net->dev)); return QV_OK; }

// Does this handle run the fused kernel?  QV_IMPL_AUTO picks it whenever it is built.
static bool runs_fused(const qv_net *net) { return net->impl == QV_IMPL_FUSED || (net->impl == QV_IMPL_AUTO && net->fm); }

static int validate_qparams(const ModelHost &m)
{
    for (int l = 0; l < QV_NLAYER; ++l) {
        const LayerHost &L = m.L[l];
        if (L.mul <= 0 || L.shift < 1 || L.shift > 30) {
            set_error("layer %d: mul=%d shift=%d outside the supported range (mul>0, 1<=shift<=30)", l, L.mul, L.shift);
            return QV_ERR_RANGE;
        }
        if (l != QV_C4 && (L.blu < 0 || L.blu >= (1 << 24))) {
            set_error("layer %d: blu=%d outside [0, 2^24)", l, L.blu);
            return QV_ERR_RANGE;
        }
    }
    return QV_OK;
}

// Called whenever the host model changed; (re)builds device images once the model is complete.
static int sync_model(qv_net *net)
{
    net->uploaded = false;
    if (!net->model.complete()) return QV_OK;
    int rc = validate_qparams(net->model);
    if (rc) return rc;
    rc = check_fp32_exact_envelope(net->model);
    if (rc) return rc;
    if ((rc = set_device(net))) return rc;
    if ((rc = layered_load(net->ln, net->model, net->st))) return rc;
    if (net->fm) { fused_free(net->fm); net->fm = nullptr; }
    net->fm = fused_upload(net->model, net->st);     // may be null when the fused path is not built
    net->uploaded = true;
    return QV_OK;
}

// With d_ori / d_sse: also adds, per frame f, the SSE of the input and of the output against d_ori to d_sse[2f], d_sse[2f + 1]
// (the integer core of vrcnn_data::psnr_pf, inference/yuv_data.cpp:98-112): the fused path in the kernel's output stage, the
// layered path, the independent cross-check, in separate passes.
static int run_forward(qv_net *net, const uint8_t *d_in, uint8_t *d_out, int n, int H, int W, cudaStream_t st,
                       const uint8_t *d_ori = nullptr, int64_t *d_sse = nullptr)
{
    if (!net->uploaded) {
        set_error("forward called before a complete model (weights + quant params) was loaded");
        return QV_ERR_STATE;
    }
    if (!runs_fused(net)) return layered_forward(net->ln, d_in, d_out, n, H, W, st, &net->launches, d_ori, d_sse);
    if (!net->fm) { set_error("fused tcgen05 path is not available in this build"); return QV_ERR_STATE; }
    if (d_sse && H > FUSED_SSE_MAX_H) { set_error("per-frame SSE: frame height %d exceeds %d", H, FUSED_SSE_MAX_H); return QV_ERR_ARG; }
    QV_CUDA(fused_forward(net->fm, d_in, d_out, n, H, W, st, &net->launches, nullptr, d_ori, d_sse));
    return QV_OK;
}

extern "C" {

int qv_create(int gpu_num, int batch, int channel, int height, int width, qv_net **out)
{
    if (!out) { set_error("qv_create: null output pointer"); return QV_ERR_ARG; }
    *out = nullptr;
    if (channel != 1) { set_error("qv_create: channel must be 1 (luma), got %d", channel); return QV_ERR_ARG; }
    if (batch < 1 || height < 1 || width < 1) { set_error("qv_create: bad geometry %dx%dx%d", batch, height, width); return QV_ERR_ARG; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        set_error("qv_create: no CUDA device (this library has no CPU fallback)");
        return QV_ERR_CUDA;
    }
    if (gpu_num < 0 || gpu_num >= ndev) { set_error("qv_create: gpu_num %d out of range (%d devices)", gpu_num, ndev); return QV_ERR_ARG; }
    QV_CUDA(cudaSetDevice(gpu_num));                                    // inference/qvrcnn.cu:6
    qv_net *net = new qv_net();
    net->dev = gpu_num; net->batch = batch; net->H = height; net->W = width;
    const size_t bytes = (size_t)batch * height * width;
    cudaError_t e = cudaStreamCreateWithFlags(&net->st, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&net->d_x, bytes);             // inference/cnn.cu:433
    if (e == cudaSuccess) e = cudaMalloc(&net->d_rec, bytes);           // inference/cnn.cu:434
    if (e == cudaSuccess) e = layered_create(&net->ln, batch, height, width);
    if (e != cudaSuccess) {
        set_error("qv_create: %s", cudaGetErrorString(e));
        qv_destroy(net);
        return QV_ERR_CUDA;
    }
    *out = net;
    return QV_OK;
}

int qv_destroy(qv_net *net)
{
    if (!net) return QV_OK;
    cudaSetDevice(net->dev);
    if (net->st) cudaStreamSynchronize(net->st);
    qv_strip_release(net);
    layered_free(net->ln);
    if (net->fm) fused_free(net->fm);
    cudaFree(net->d_x); cudaFree(net->d_rec);
    for (int i = 0; i < 2; ++i) {
        cudaFree(net->d_slot_in[i]); cudaFree(net->d_slot_out[i]);
        cudaFreeHost(net->h_pin_in[i]); cudaFreeHost(net->h_pin_out[i]);
        if (net->pst[i]) cudaStreamDestroy(net->pst[i]);
    }
    if (net->st) cudaStreamDestroy(net->st);
    delete net;
    return QV_OK;
}

int qv_load_static_para_mem(qv_net *net, const void *image, size_t len)
{
    if (!net || !image) { set_error("qv_load_static_para_mem: null argument"); return QV_ERR_ARG; }
    ModelHost m;
    int rc = parse_model_vect_c((const uint8_t *)image, len, m);
    if (rc) return rc;
    net->model = m;
    return sync_model(net);
}

int qv_debug_fused_tables(const void *image, size_t len, uint8_t *wimg, uint32_t *ops, int32_t *consts, size_t sizes[3])
{
    if (!image || !sizes) { set_error("qv_debug_fused_tables: null argument"); return QV_ERR_ARG; }
    ModelHost m;
    int rc = parse_model_vect_c((const uint8_t *)image, len, m);
    if (rc) return rc;
    std::vector<uint8_t> w;
    std::vector<uint32_t> o;
    std::vector<int32_t> c;
    fused_debug_tables(m, w, o, c);
    if (wimg && sizes[0] >= w.size()) memcpy(wimg, w.data(), w.size());
    if (ops && sizes[1] >= o.size()) memcpy(ops, o.data(), o.size() * sizeof(uint32_t));
    if (consts && sizes[2] >= c.size()) memcpy(consts, c.data(), c.size() * sizeof(int32_t));
    sizes[0] = w.size(); sizes[1] = o.size(); sizes[2] = c.size();
    return QV_OK;
}

int qv_debug_fused_units(int sm_count, int n_frames, int height, int width, int row0, int row1, int row_window, int allow_line,
                         int32_t *units, size_t *n_units, int *grid)
{
    if (!n_units || !grid) { set_error("qv_debug_fused_units: null argument"); return QV_ERR_ARG; }
    std::vector<int> u;
    int g = 0;
    if (fused_debug_units(sm_count, n_frames, height, width, row0, row1, row_window != 0, allow_line != 0, u, g)) {
        set_error("qv_debug_fused_units: bad geometry");
        return QV_ERR_ARG;
    }
    if (units && *n_units >= u.size() / 5) memcpy(units, u.data(), u.size() * sizeof(int));
    *n_units = u.size() / 5;
    *grid = g;
    return QV_OK;
}

int qv_load_static_para(qv_net *net, const char *filename)
{
    if (!net) { set_error("qv_load_static_para: null handle"); return QV_ERR_ARG; }
    std::vector<uint8_t> buf;
    int rc = read_file(filename, buf);
    if (rc) { set_error("cannot open model file. (%s)", filename ? filename : "(null)"); return rc; }   // qvrcnn.cu:52
    return qv_load_static_para_mem(net, buf.data(), buf.size());
}

int qv_load_static_para_hwcn(qv_net *net, const char *filename)
{
    if (!net) { set_error("qv_load_static_para_hwcn: null handle"); return QV_ERR_ARG; }
    std::vector<uint8_t> buf;
    int rc = read_file(filename, buf);
    if (rc) return rc;
    ModelHost m;
    rc = parse_model_hwcn(buf.data(), buf.size(), m);
    if (rc) return rc;
    net->model = m;
    return sync_model(net);
}

int qv_load_quant_params(qv_net *net, const char *filename)
{
    if (!net) { set_error("qv_load_quant_params: null handle"); return QV_ERR_ARG; }
    int32_t q[18];
    int rc = qv_read_quant_params(filename, q);
    if (rc) return rc;
    for (int l = 0; l < QV_NLAYER; ++l) {
        LayerHost &L = net->model.L[l];
        L.blu = q[3 * l]; L.mul = q[3 * l + 1]; L.shift = q[3 * l + 2];
        L.have_q = true;
    }
    return sync_model(net);
}

int qv_set_weights(qv_net *net, int layer, const int8_t *w_kcrs, const int32_t *bias)
{
    if (!net || !w_kcrs || !bias || layer < 0 || layer >= QV_NLAYER) { set_error("qv_set_weights: bad argument"); return QV_ERR_ARG; }
    const LayerShape &s = kLayers[layer];
    LayerHost &L = net->model.L[layer];
    L.w.assign(w_kcrs, w_kcrs + (size_t)s.cout * s.cin * s.k * s.k);
    L.b.assign(bias, bias + s.cout);
    L.have_w = true;
    return sync_model(net);
}

int qv_get_quant_params(const qv_net *net, int32_t *out18)
{
    if (!net || !out18) { set_error("qv_get_quant_params: null argument"); return QV_ERR_ARG; }
    for (int l = 0; l < QV_NLAYER; ++l) {
        out18[3 * l] = net->model.L[l].blu; out18[3 * l + 1] = net->model.L[l].mul; out18[3 * l + 2] = net->model.L[l].shift;
    }
    return QV_OK;
}

int qv_load_data(qv_net *net, const uint8_t *host_luma)
{
    if (!net || !host_luma) { set_error("qv_load_data: null argument"); return QV_ERR_ARG; }
    int rc = set_device(net);
    if (rc) return rc;
    const size_t bytes = (size_t)net->batch * net->H * net->W;
    QV_CUDA(cudaMemcpyAsync(net->d_x, host_luma, bytes, cudaMemcpyHostToDevice, net->st));   // cnn.cu:441
    QV_CUDA(cudaStreamSynchronize(net->st));
    return QV_OK;
}

// After a synchronisation: did a CTA of the fused kernel report a failure?  (Never a silent wrong answer.)
static int kernel_report(qv_net *net)
{
    const int f = net->fm ? fused_take_failure(net->fm) : 0;
    if (!f) return QV_OK;
    set_error(f == 2 ? "fused kernel: a CTA saw other shared-memory / TMEM bases than the operand table was built for"
              : f == 3 ? "strip mode: a neighbour GPU's rows were never published (the frame data of this call is not valid)"
                       : "fused kernel: an mbarrier wait timed out (the frame data of this call is not valid)");
    return QV_ERR_CUDA;
}

// qv_forward_blu, qv_forward_frames_device and, with d_ori / d_sse, qv_forward_frames_device_sse once their arguments are
// checked.  A null cuda_stream runs on the handle's own stream and synchronises.
static int forward_frames_device(qv_net *net, const uint8_t *d_in, const uint8_t *d_ori, uint8_t *d_out, int n_frames,
                                 int64_t *d_sse, void *cuda_stream)
{
    int rc = set_device(net);
    if (rc) return rc;
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : net->st;
    if (n_frames > 0 && (rc = run_forward(net, d_in, d_out, n_frames, net->H, net->W, st, d_ori, d_sse))) return rc;
    if (!cuda_stream) { QV_CUDA(cudaStreamSynchronize(st)); return kernel_report(net); }
    return QV_OK;
}

int qv_forward_blu(qv_net *net)
{
    if (!net) { set_error("qv_forward_blu: null handle"); return QV_ERR_ARG; }
    return forward_frames_device(net, net->d_x, nullptr, net->d_rec, net->batch, nullptr, nullptr);   // the reference is synchronous (kernel.cu:95)
}

int qv_get_recon(qv_net *net, uint8_t *host_out)
{
    if (!net || !host_out) { set_error("qv_get_recon: null argument"); return QV_ERR_ARG; }
    int rc = set_device(net);
    if (rc) return rc;
    const size_t bytes = (size_t)net->batch * net->H * net->W;
    QV_CUDA(cudaMemcpyAsync(host_out, net->d_rec, bytes, cudaMemcpyDeviceToHost, net->st));   // kernel.cu:96
    QV_CUDA(cudaStreamSynchronize(net->st));
    return kernel_report(net);
}

int qv_forward_frames_device(qv_net *net, const uint8_t *d_in, uint8_t *d_out, int n_frames, void *cuda_stream)
{
    if (!net || !d_in || !d_out || n_frames < 0) { set_error("qv_forward_frames_device: bad argument"); return QV_ERR_ARG; }
    return forward_frames_device(net, d_in, nullptr, d_out, n_frames, nullptr, cuda_stream);
}

int qv_forward_frames_device_sse(qv_net *net, const uint8_t *d_in, const uint8_t *d_ori, uint8_t *d_out, int n_frames,
                                 int64_t *d_sse, void *cuda_stream)
{
    // per-frame form of vrcnn_data::psnr_pf (inference/yuv_data.cpp:98-112): exact integer SSEs, incremented
    if (!net || !d_in || !d_ori || !d_out || !d_sse || n_frames < 0) { set_error("qv_forward_frames_device_sse: bad argument"); return QV_ERR_ARG; }
    return forward_frames_device(net, d_in, d_ori, d_out, n_frames, d_sse, cuda_stream);
}

int qv_forward_rows_device(qv_net *net, const uint8_t *d_in, int img_height, int in_row0, int in_rows, uint8_t *d_out,
                           int out_row0, int out_row1, void *cuda_stream)
{
    if (!net || !d_in || !d_out) { set_error("qv_forward_rows_device: null argument"); return QV_ERR_ARG; }
    // The net's receptive-field radius is 2+2+1+1 = 6 rows: every output row needs the input rows within 6 of it that
    // lie inside the image; outside the image every layer pads its own input with zeros (inference/cnn.cu:44-49).
    const int in_row1 = in_row0 + in_rows;
    if (img_height < 1 || in_row0 < 0 || in_rows < 1 || in_row1 > img_height || out_row0 < in_row0 || out_row1 > in_row1 ||
        out_row0 > out_row1) { set_error("qv_forward_rows_device: inconsistent row ranges"); return QV_ERR_ARG; }
    if ((in_row0 != 0 && out_row0 - in_row0 < STRIP_HALO) || (in_row1 != img_height && in_row1 - out_row1 < STRIP_HALO)) {
        set_error("qv_forward_rows_device: need 6 halo rows on every interior strip edge");
        return QV_ERR_ARG;
    }
    int rc = set_device(net);
    if (rc) return rc;
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : net->st;
    if (!net->uploaded || (runs_fused(net) && !net->fm)) { set_error("forward called before a complete model (weights + quant params) was loaded"); return QV_ERR_STATE; }
    if (runs_fused(net)) {
        // the fused kernel takes the window as what it is: rows [in_row0, in_row1) of an img_height-row image, of which it
        // computes and writes exactly [out_row0, out_row1) -- no scratch frame, no copy
        FusedRows fr;
        fr.own0 = in_row0; fr.own1 = in_row1; fr.out0 = out_row0; fr.out1 = out_row1;
        QV_CUDA(fused_forward(net->fm, d_in, d_out, 1, img_height, net->W, st, &net->launches, &fr));
    } else if ((rc = layered_forward_rows(net->ln, d_in, in_rows, d_out, out_row0 - in_row0, out_row1 - in_row0, st, &net->launches))) {
        return rc;
    }
    if (!cuda_stream) { QV_CUDA(cudaStreamSynchronize(st)); return kernel_report(net); }
    return QV_OK;
}

int qv_synchronize(qv_net *net, void *cuda_stream)
{
    if (!net) { set_error("qv_synchronize: null handle"); return QV_ERR_ARG; }
    int rc = set_device(net);
    if (rc) return rc;
    QV_CUDA(cudaStreamSynchronize(cuda_stream ? (cudaStream_t)cuda_stream : net->st));
    return kernel_report(net);
}

// ---- strips: setup / export / attach / load / forward -------------------------------------------------------------
static void strip_detach(qv_net *net)
{
    for (StripPeer &p : net->strip.peer) {
        if (p.attached && p.ipc && p.base) cudaIpcCloseMemHandle(p.base);
        p = StripPeer{};
    }
}

int qv_strip_release(qv_net *net)
{
    if (!net) { set_error("qv_strip_release: null handle"); return QV_ERR_ARG; }
    if (!net->strip.on) return QV_OK;
    cudaSetDevice(net->dev);
    cudaStreamSynchronize(net->st);
    strip_detach(net);
    cudaFree(net->strip.block);
    net->strip = StripState{};
    if (net->dev >= 0 && net->dev < 64) {
        std::lock_guard<std::mutex> l(g_strip_mu);
        auto &v = g_strip_nets[net->dev];
        v.erase(std::remove(v.begin(), v.end(), net), v.end());
    }
    return QV_OK;
}

int qv_strip_setup(qv_net *net, int img_height, int row0, int row1)
{
    if (!net) { set_error("qv_strip_setup: null handle"); return QV_ERR_ARG; }
    if (img_height < 1 || row0 < 0 || row1 <= row0 || row1 > img_height) { set_error("qv_strip_setup: rows [%d, %d) of %d", row0, row1, img_height); return QV_ERR_ARG; }
    int rc = set_device(net);
    if (rc) return rc;
    qv_strip_release(net);
    StripState &S = net->strip;
    S.img_h = img_height; S.row0 = row0; S.row1 = row1;
    S.slot_stride = ((size_t)(row1 - row0) * net->W + 255) / 256 * 256;
    QV_CUDA(cudaMalloc(&S.block, STRIP_HDR + 2 * S.slot_stride));
    QV_CUDA(cudaMemset(S.block, 0, STRIP_HDR));
    QV_CUDA(cudaDeviceSynchronize());
    S.on = true;
    if (net->dev >= 0 && net->dev < 64) {
        std::lock_guard<std::mutex> l(g_strip_mu);
        g_strip_nets[net->dev].push_back(net);
    }
    return QV_OK;
}

int qv_strip_export(qv_net *net, qv_strip_desc *out)
{
    if (!net || !out) { set_error("qv_strip_export: null argument"); return QV_ERR_ARG; }
    if (!net->strip.on) { set_error("qv_strip_export: qv_strip_setup has not been called"); return QV_ERR_STATE; }
    int rc = set_device(net);
    if (rc) return rc;
    StripDescImpl d{};
    d.magic = STRIP_MAGIC; d.dev = net->dev; d.row0 = net->strip.row0; d.row1 = net->strip.row1; d.width = net->W; d.img_h = net->strip.img_h;
    d.nonce = process_nonce();
    d.base = (uint64_t)(uintptr_t)net->strip.block; d.slot_off = STRIP_HDR; d.slot_stride = net->strip.slot_stride;
    d.net = (uint64_t)(uintptr_t)net;
    QV_CUDA(cudaIpcGetMemHandle(&d.ipc, net->strip.block));
    QV_CUDA(cudaDeviceGetPCIBusId(d.pci, (int)sizeof(d.pci), net->dev));
    memset(out, 0, sizeof(*out));
    memcpy(out, &d, sizeof(d));
    return QV_OK;
}

int qv_strip_attach(qv_net *net, int side, const qv_strip_desc *neighbour)
{
    if (!net || !neighbour || (side != QV_STRIP_ABOVE && side != QV_STRIP_BELOW)) { set_error("qv_strip_attach: bad argument"); return QV_ERR_ARG; }
    StripState &S = net->strip;
    if (!S.on) { set_error("qv_strip_attach: qv_strip_setup has not been called"); return QV_ERR_STATE; }
    StripDescImpl d;
    memcpy(&d, neighbour, sizeof(d));
    if (d.magic != STRIP_MAGIC) { set_error("qv_strip_attach: not a strip descriptor"); return QV_ERR_ARG; }
    if (d.width != net->W || d.img_h != S.img_h) { set_error("qv_strip_attach: the neighbour's frame is %dx%d, this one %dx%d", d.width, d.img_h, net->W, S.img_h); return QV_ERR_ARG; }
    if (side == QV_STRIP_ABOVE ? d.row1 != S.row0 : d.row0 != S.row1) {
        set_error("qv_strip_attach: rows [%d, %d) are not adjacent %s rows [%d, %d)", d.row0, d.row1, side == QV_STRIP_ABOVE ? "above" : "below", S.row0, S.row1);
        return QV_ERR_ARG;
    }
    if (d.row1 - d.row0 < STRIP_HALO) {
        // the halo would reach into the strip after next, which this protocol does not exchange
        set_error("qv_strip_attach: the neighbour holds %d rows, fewer than the %d-row halo (use fewer strips)", d.row1 - d.row0, STRIP_HALO);
        return QV_ERR_ARG;
    }
    int rc = set_device(net);
    if (rc) return rc;
    StripPeer &P = S.peer[side];
    if (P.attached && P.ipc && P.base) cudaIpcCloseMemHandle(P.base);
    P = StripPeer{};
    if (d.nonce == process_nonce()) {
        // same process: plain peer access to the neighbour's allocation
        if (d.dev != net->dev) {
            int can = 0;
            QV_CUDA(cudaDeviceCanAccessPeer(&can, net->dev, d.dev));
            if (!can) { set_error("qv_strip_attach: device %d cannot map memory of device %d (no peer access)", net->dev, d.dev); return QV_ERR_CUDA; }
            cudaError_t e = cudaDeviceEnablePeerAccess(d.dev, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); e = cudaSuccess; }
            QV_CUDA(e);
        }
        P.base = (uint8_t *)(uintptr_t)d.base;
        P.net = (qv_net *)(uintptr_t)d.net;
    } else {
        char my_pci[16] = {0};
        QV_CUDA(cudaDeviceGetPCIBusId(my_pci, (int)sizeof(my_pci), net->dev));
        if (strncmp(my_pci, d.pci, sizeof(my_pci)) == 0) {
            // two processes time-slicing one GPU: a kernel of one that waits for a kernel of the other may never see it run
            set_error("qv_strip_attach: the neighbour strip belongs to another process on the SAME GPU; strips of different processes must be on different GPUs");
            return QV_ERR_ARG;
        }
        void *p = nullptr;
        QV_CUDA(cudaIpcOpenMemHandle(&p, d.ipc, cudaIpcMemLazyEnablePeerAccess));
        P.base = (uint8_t *)p;
        P.ipc = true;
    }
    P.d = d;
    char my_pci[16] = {0};
    QV_CUDA(cudaDeviceGetPCIBusId(my_pci, (int)sizeof(my_pci), net->dev));
    P.same_device = strncmp(my_pci, d.pci, sizeof(my_pci)) == 0;
    P.attached = true;
    return QV_OK;
}

int qv_strip_input(qv_net *net, int slot, void **d_rows)
{
    if (!net || !d_rows || slot < 0 || slot > 1) { set_error("qv_strip_input: bad argument"); return QV_ERR_ARG; }
    if (!net->strip.on) { set_error("qv_strip_input: qv_strip_setup has not been called"); return QV_ERR_STATE; }
    *d_rows = net->strip.block + STRIP_HDR + (size_t)slot * net->strip.slot_stride;
    return QV_OK;
}

// Strips that share this handle's GPU (same process) are ordered by the one stream they must all be driven on.
static int check_shared_device_stream(qv_net *net, cudaStream_t st, const char *who)
{
    std::lock_guard<std::mutex> l(g_strip_mu);
    for (qv_net *o : g_strip_nets[net->dev])
        if (o != net && o->strip.used && o->strip.last_stream != st) {
            set_error("%s: several strips live on GPU %d: drive all of them on ONE caller-provided stream (kernels of different launches "
                      "must not wait for each other on one GPU, so stream order is what orders them)", who, net->dev);
            return QV_ERR_STATE;
        }
    return QV_OK;
}

int qv_strip_acquire(qv_net *net, int slot, void *cuda_stream)
{
    if (!net || slot < 0 || slot > 1) { set_error("qv_strip_acquire: bad argument"); return QV_ERR_ARG; }
    StripState &S = net->strip;
    if (!S.on) { set_error("qv_strip_acquire: qv_strip_setup has not been called"); return QV_ERR_STATE; }
    int rc = set_device(net);
    if (rc) return rc;
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : net->st;
    if ((rc = check_shared_device_stream(net, st, "qv_strip_acquire"))) return rc;
    S.last_stream = st; S.used = true;
    const uint32_t s = S.slot_seq[slot];
    const uint32_t *w[2] = {nullptr, nullptr};
    for (int side = 0; side < 2; ++side) {
        const StripPeer &P = S.peer[side];
        if (!P.attached || s == 0) continue;
        if (P.same_device) {
            // the neighbour's forward that read this slot must already be on the (shared) stream
            if (P.net->strip.forwards[slot] < S.forwards[slot]) {
                set_error("qv_strip_acquire: the neighbour strip on the same GPU has not yet consumed slot %d (issue the strips' calls frame by frame)", slot);
                return QV_ERR_STATE;
            }
        } else {
            w[side] = reinterpret_cast<const uint32_t *>(P.base + STRIP_DONE);      // another GPU: wait for its "completed step s"
        }
    }
    if (net->fm && (w[0] || w[1])) {
        QV_CUDA(fused_wait_words(net->fm, w[0], s, w[1], s, st));
        net->launches += 1;
    }
    S.fills[slot] += 1;
    return QV_OK;
}

int qv_strip_load(qv_net *net, int slot, const uint8_t *host_rows, void *cuda_stream)
{
    if (!host_rows) { set_error("qv_strip_load: null argument"); return QV_ERR_ARG; }
    int rc = qv_strip_acquire(net, slot, cuda_stream);
    if (rc) return rc;
    StripState &S = net->strip;
    QV_CUDA(cudaMemcpyAsync(S.block + STRIP_HDR + (size_t)slot * S.slot_stride, host_rows, (size_t)(S.row1 - S.row0) * net->W,
                            cudaMemcpyHostToDevice, cuda_stream ? (cudaStream_t)cuda_stream : net->st));
    return QV_OK;
}

// What every forward of a strip handle needs: qv_strip_setup, a loaded model on the fused path, a neighbour on every interior edge.
static int strip_ready(const qv_net *net, const char *who)
{
    const StripState &S = net->strip;
    if (!S.on) { set_error("%s: qv_strip_setup has not been called", who); return QV_ERR_STATE; }
    if (!net->uploaded || !net->fm || net->impl == QV_IMPL_LAYERED) {
        set_error("%s: needs a loaded model and the fused path (peer-mapped halo rows are read by the fused kernel)", who);
        return QV_ERR_STATE;
    }
    if ((S.row0 > 0 && !S.peer[QV_STRIP_ABOVE].attached) || (S.row1 < S.img_h && !S.peer[QV_STRIP_BELOW].attached)) {
        set_error("%s: rows [%d, %d) of %d have an interior edge with no neighbour attached", who, S.row0, S.row1, S.img_h);
        return QV_ERR_STATE;
    }
    return QV_OK;
}

static int strip_forward(qv_net *net, int slot, const uint8_t *d_ori, uint8_t *d_out, int64_t *d_sse, void *cuda_stream, const char *who)
{
    StripState &S = net->strip;
    int rc = strip_ready(net, who);
    if (rc) return rc;
    if (d_sse && S.img_h > FUSED_SSE_MAX_H) { set_error("%s: frame height %d exceeds %d", who, S.img_h, FUSED_SSE_MAX_H); return QV_ERR_ARG; }
    rc = set_device(net);
    if (rc) return rc;
    cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : net->st;
    if ((rc = check_shared_device_stream(net, st, who))) return rc;
    const size_t W = net->W;
    FusedRows fr;
    fr.own0 = fr.out0 = S.row0; fr.own1 = fr.out1 = S.row1;
    fr.pub = reinterpret_cast<uint32_t *>(S.block + STRIP_PUB);
    fr.done = reinterpret_cast<uint32_t *>(S.block + STRIP_DONE);
    fr.done_ctr = reinterpret_cast<uint32_t *>(S.block + STRIP_CTR);
    for (int side = 0; side < 2; ++side) {
        if (side == QV_STRIP_ABOVE ? S.row0 == 0 : S.row1 == S.img_h) continue;
        const StripPeer &P = S.peer[side];
        const uint8_t *rows = P.base + P.d.slot_off + (size_t)slot * P.d.slot_stride;
        const uint32_t *flag = reinterpret_cast<const uint32_t *>(P.base + STRIP_PUB);
        if (P.same_device) {
            // a neighbour on this very GPU: no kernel may wait for it -- its rows are ordered before this launch by the shared
            // stream, provided its slot was filled for this frame already (checked here, on the host)
            if (P.net->strip.fills[slot] == 0) {
                set_error("%s: the neighbour strip on the same GPU has not filled slot %d yet (strips that share a GPU: all loads of a frame, then its forwards, on one stream)", who, slot);
                return QV_ERR_STATE;
            }
            flag = nullptr;
        }
        if (side == QV_STRIP_ABOVE) { fr.top_rows = STRIP_HALO; fr.d_top = rows + (size_t)(P.d.row1 - P.d.row0 - STRIP_HALO) * W; fr.flag_top = flag; }
        else { fr.bot_rows = STRIP_HALO; fr.d_bot = rows; fr.flag_bot = flag; }
    }
    const uint32_t seq = ++S.seq;
    S.slot_seq[slot] = seq;
    S.forwards[slot] += 1;
    S.last_stream = st; S.used = true;
    fr.seq = seq;
    const uint8_t *own = S.block + STRIP_HDR + (size_t)slot * S.slot_stride;
    QV_CUDA(fused_forward(net->fm, own, d_out, 1, S.img_h, net->W, st, &net->launches, &fr, d_ori, d_sse));
    if (!cuda_stream) { QV_CUDA(cudaStreamSynchronize(st)); return kernel_report(net); }
    return QV_OK;
}

int qv_strip_forward(qv_net *net, int slot, uint8_t *d_out, void *cuda_stream)
{
    if (!net || !d_out || slot < 0 || slot > 1) { set_error("qv_strip_forward: bad argument"); return QV_ERR_ARG; }
    return strip_forward(net, slot, nullptr, d_out, nullptr, cuda_stream, "qv_strip_forward");
}

int qv_strip_forward_sse(qv_net *net, int slot, const uint8_t *d_ori_rows, uint8_t *d_out, int64_t *d_sse2, void *cuda_stream)
{
    // this GPU's share of vrcnn_data::psnr_pf (inference/yuv_data.cpp:98-112) for one frame; the strips' values add up
    if (!net || !d_ori_rows || !d_out || !d_sse2 || slot < 0 || slot > 1) { set_error("qv_strip_forward_sse: bad argument"); return QV_ERR_ARG; }
    return strip_forward(net, slot, d_ori_rows, d_out, d_sse2, cuda_stream, "qv_strip_forward_sse");
}

int qv_forward_frames_host(qv_net *net, const uint8_t *h_in, uint8_t *h_out, int n_frames)
{
    if (!net || !h_in || !h_out || n_frames < 0) { set_error("qv_forward_frames_host: bad argument"); return QV_ERR_ARG; }
    int rc = set_device(net);
    if (rc) return rc;
    const size_t fpx = (size_t)net->H * net->W;
    // Pipeline granularity: the H2D of chunk k+1 and the D2H of chunk k-1 hide behind the compute of chunk k;
    // only the first upload and the last download are exposed, so the schedule is tapered -- small chunks at
    // both ends (1, 3, 4, 8, 16, 16, 8, 4, 3, 1 sixty-fourths of the frames; measured best of seven schedules at
    // 64 x 1080p, profiles/r1_e2e_chunk_schedules.log), each at most `batch` frames.
    std::vector<int> chunks;
    {
        static const int num[10] = {1, 3, 4, 8, 16, 16, 8, 4, 3, 1};
        int left = n_frames;
        if (n_frames >= 16) {
            for (int k = 0; k < 10 && left > 0; ++k) {
                int want = k == 9 ? left : std::max(1, n_frames * num[k] / 64);
                while (want > 0 && left > 0) {
                    const int c = std::min(std::min(want, left), net->batch);
                    chunks.push_back(c); want -= c; left -= c;
                }
            }
        }
        const int uni = std::max(1, std::min(net->batch, (n_frames + 3) / 4));
        while (left > 0) { const int c = std::min(uni, left); chunks.push_back(c); left -= c; }
    }
    const size_t cbytes = (size_t)net->batch * fpx;
    // Is the caller's memory page-locked already?  Then DMA straight from/to it.
    cudaPointerAttributes ai{}, ao{};
    bool pinned_in = cudaPointerGetAttributes(&ai, h_in) == cudaSuccess && ai.type == cudaMemoryTypeHost;
    bool pinned_out = cudaPointerGetAttributes(&ao, h_out) == cudaSuccess && ao.type == cudaMemoryTypeHost;
    cudaGetLastError();
    for (int i = 0; i < 2; ++i) {
        if (!net->pst[i]) QV_CUDA(cudaStreamCreateWithFlags(&net->pst[i], cudaStreamNonBlocking));
        if (!net->d_slot_in[i]) QV_CUDA(cudaMalloc(&net->d_slot_in[i], cbytes));
        if (!net->d_slot_out[i]) QV_CUDA(cudaMalloc(&net->d_slot_out[i], cbytes));
        if (!pinned_in && !net->h_pin_in[i]) QV_CUDA(cudaMallocHost(&net->h_pin_in[i], cbytes));
        if (!pinned_out && !net->h_pin_out[i]) QV_CUDA(cudaMallocHost(&net->h_pin_out[i], cbytes));
    }
    // Two slots, each an in-order H2D -> forward -> D2H chain on its own stream, so the copies of
    // one chunk overlap the compute of the other (the reference's loop, inference/kernel.cu:91-97,
    // is fully serial: blocking memcpy, forward, sync, blocking memcpy).
    struct Pending { int f0 = -1, c = 0; } pend[2];
    auto drain = [&](int s) -> int {
        if (pend[s].f0 < 0) return QV_OK;
        QV_CUDA(cudaStreamSynchronize(net->pst[s]));
        if (!pinned_out) memcpy(h_out + (size_t)pend[s].f0 * fpx, net->h_pin_out[s], (size_t)pend[s].c * fpx);
        pend[s].f0 = -1;
        return QV_OK;
    };
    int slot = 0;
    int f0 = 0;
    for (size_t ci = 0; ci < chunks.size(); f0 += chunks[ci], ++ci, slot ^= 1) {
        const int c = chunks[ci];
        const size_t bytes = (size_t)c * fpx;
        if ((rc = drain(slot))) return rc;
        const uint8_t *src = h_in + (size_t)f0 * fpx;
        if (!pinned_in) { memcpy(net->h_pin_in[slot], src, bytes); src = net->h_pin_in[slot]; }
        QV_CUDA(cudaMemcpyAsync(net->d_slot_in[slot], src, bytes, cudaMemcpyHostToDevice, net->pst[slot]));
        // The fused kernel has no scratch: its launches of the two slots are left unordered, so the persistent CTAs of the
        // next chunk move onto the SMs the previous chunk's last wave has already left.  The layered path orders its own.
        rc = run_forward(net, net->d_slot_in[slot], net->d_slot_out[slot], c, net->H, net->W, net->pst[slot]);
        if (rc) return rc;
        uint8_t *dst = pinned_out ? h_out + (size_t)f0 * fpx : net->h_pin_out[slot];
        QV_CUDA(cudaMemcpyAsync(dst, net->d_slot_out[slot], bytes, cudaMemcpyDeviceToHost, net->pst[slot]));
        pend[slot].f0 = f0; pend[slot].c = c;
    }
    if ((rc = drain(0))) return rc;
    if ((rc = drain(1))) return rc;
    return kernel_report(net);
}

// ---- streaming file pipeline (SURVEY 8 f2) -------------------------------------------------------------
}  // extern "C"

namespace {
// The files of one streaming call (-1: not given).  The reconstruction is opened without truncation and created if missing:
// several ranks / threads may fill one file, each its own frame range or rows (a caller that lost the race to create it
// must not wipe what another has written).
struct StreamFiles {
    int anchor = -1, ori = -1, recon = -1;
    StreamFiles() = default;
    StreamFiles(const StreamFiles &) = delete;
    StreamFiles &operator=(const StreamFiles &) = delete;
    ~StreamFiles() { for (int fd : {anchor, ori, recon}) if (fd >= 0) close(fd); }
    int open_all(const char *anchor_yuv, const char *ori_yuv, const char *recon_yuv)
    {
        if ((anchor = open(anchor_yuv, O_RDONLY)) < 0) { set_error("open file failed. (%s)", anchor_yuv); return QV_ERR_IO; }   // yuv_data.cpp:19-31
        if (ori_yuv && (ori = open(ori_yuv, O_RDONLY)) < 0) { set_error("open file failed. (%s)", ori_yuv); return QV_ERR_IO; }
        if (recon_yuv && (recon = open(recon_yuv, O_CREAT | O_RDWR, 0644)) < 0) { set_error("open file failed. (%s)", recon_yuv); return QV_ERR_IO; }
        return QV_OK;
    }
};
bool pread_all(int fd, uint8_t *p, size_t n, off_t off)
{
    while (n > 0) {
        const ssize_t r = pread(fd, p, n, off);
        if (r < 0 && errno == EINTR) continue;
        if (r <= 0) return false;
        p += r; n -= (size_t)r; off += r;
    }
    return true;
}
bool pwrite_all(int fd, const uint8_t *p, size_t n, off_t off)
{
    while (n > 0) {
        const ssize_t r = pwrite(fd, p, n, off);
        if (r < 0 && errno == EINTR) continue;
        if (r <= 0) return false;
        p += r; n -= (size_t)r; off += r;
    }
    return true;
}
// Byte offset of luma row `row` of frame `frame` in a YUV 4:2:0 file: frame stride h*w*3/2 (yuv_data.cpp:32-38).
off_t luma_offset(long long frame, int img_h, int w, int row)
{
    const long long fpx = (long long)img_h * w;
    return (off_t)(frame * (fpx + fpx / 2) + (long long)row * w);
}
// Luma rows [row0, row1) of frame `frame`.
bool read_luma(int fd, long long frame, int img_h, int w, int row0, int row1, uint8_t *dst)
{
    return pread_all(fd, dst, (size_t)(row1 - row0) * w, luma_offset(frame, img_h, w, row0));
}
// Luma rows [row0, row1) of frame `frame` in save_recon_as' layout (yuv_data.cpp:119-125); whoever writes the last image row
// also writes the frame's h*w/2 zero bytes of chroma (`zeros`), so the file does not depend on how it was pre-sized.
bool write_recon_rows(int fd, long long frame, int img_h, int w, int row0, int row1, const uint8_t *src, const uint8_t *zeros)
{
    return pwrite_all(fd, src, (size_t)(row1 - row0) * w, luma_offset(frame, img_h, w, row0)) &&
           (row1 < img_h || pwrite_all(fd, zeros, (size_t)img_h * w / 2, luma_offset(frame, img_h, w, img_h)));
}

// What one streaming call holds on one device: streams, events, device and page-locked memory.  The destructor, which also
// runs on every early return, makes the streams idle before it frees anything they may still read or write.
struct DeviceHold {
    int dev = 0;
    std::vector<cudaStream_t> streams;
    std::vector<cudaEvent_t> events;
    std::vector<void *> mem, pinned;
    DeviceHold() = default;
    DeviceHold(const DeviceHold &) = delete;
    DeviceHold &operator=(const DeviceHold &) = delete;
    ~DeviceHold()
    {
        cudaSetDevice(dev);
        idle();
        for (cudaStream_t s : streams) cudaStreamDestroy(s);
        for (cudaEvent_t e : events) cudaEventDestroy(e);
        for (void *p : mem) cudaFree(p);
        for (void *p : pinned) cudaFreeHost(p);
    }
    void idle() { for (cudaStream_t s : streams) cudaStreamSynchronize(s); }
    cudaError_t stream(cudaStream_t *s)
    {
        const cudaError_t e = cudaStreamCreateWithFlags(s, cudaStreamNonBlocking);
        if (e == cudaSuccess) streams.push_back(*s);
        return e;
    }
    cudaError_t event(cudaEvent_t *ev)
    {
        const cudaError_t e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming);
        if (e == cudaSuccess) events.push_back(*ev);
        return e;
    }
    template <class T> cudaError_t alloc(T **p, size_t bytes)
    {
        const cudaError_t e = cudaMalloc(p, bytes);
        if (e == cudaSuccess) mem.push_back(*p);
        return e;
    }
};

constexpr int RING_NS = 3;                       // ring entries: one being read, one on the GPU, one being written
// One handle's band of a streaming call: rows [row0, row1) of every frame, on the device of hold[hold].
struct RingPart {
    int hold = 0, row0 = 0, row1 = 0;
    uint8_t *h_in[RING_NS] = {}, *h_ori[RING_NS] = {}, *h_out[RING_NS] = {};   // page-locked, c_max frames of the band each
    cudaEvent_t done[RING_NS] = {};             // recorded by the GPU stage once the rows of ring entry r are downloaded
};
// The GPU stage of device hold[d] for item k (frames [first_frame + f0, first_frame + f0 + c)) in ring entry r: uploads h_in
// (h_ori) of its parts, runs the forward, downloads h_out and records done[r] of every part.  Returns a QV_ERR_* code.
using RingLaunch = std::function<int(int d, int k, int f0, int c, int r)>;

// The pipeline behind qv_stream_yuv_pf and qv_strip_stream_yuv_pf.  Frames [first_frame, first_frame + n_frames) pass in items
// of up to c_max frames, item k through ring entry k % RING_NS of every part: a reader thread reads the parts' rows of the
// item's frames from the anchor (and original) file, one thread per device of `hold` calls `launch`, and a writer thread
// waits for every part's done event and writes its rows to the reconstruction file.  An entry goes free -> read -> launched
// on every device -> free, so the reader is at most one entry ahead of the GPU stage and the writer one behind.  The first
// failure of any stage wakes them all; its code is returned and its message set on the calling thread.  The ring is
// allocated in `hold`, which frees it once the streams of the GPU stage are idle.
int stream_ring(const char *who, const StreamFiles &F, int img_h, int W, int first_frame, int n_frames, int c_max,
                std::vector<RingPart> &parts, std::vector<DeviceHold> &hold, const RingLaunch &launch)
{
    const bool with_ori = F.ori >= 0;
    for (RingPart &P : parts) {
        DeviceHold &H = hold[P.hold];
        QV_CUDA(cudaSetDevice(H.dev));
        const size_t bytes = (size_t)c_max * (P.row1 - P.row0) * W;
        for (int r = 0; r < RING_NS; ++r) {
            for (uint8_t **p : {&P.h_in[r], &P.h_out[r], with_ori ? &P.h_ori[r] : nullptr})
                if (p) { QV_CUDA(cudaMallocHost(p, bytes)); H.pinned.push_back(*p); }
            QV_CUDA(H.event(&P.done[r]));
        }
    }

    enum { FREE, READ, LAUNCHED };
    struct Entry { int item = -1, state = FREE, launched = 0; } ring[RING_NS];
    std::mutex mu;
    std::condition_variable cv;
    bool failed = false;
    int fail_rc = QV_OK;
    std::string fail_msg;
    auto fail = [&](int code, const std::string &msg) {
        std::lock_guard<std::mutex> l(mu);
        if (!failed) { failed = true; fail_rc = code; fail_msg = msg; }
        cv.notify_all();
    };
    // Waits until entry E holds item k in `state` (a free entry: any item); false once a stage has failed.
    auto wait = [&](const Entry &E, int state, int k) {
        std::unique_lock<std::mutex> l(mu);
        cv.wait(l, [&] { return (E.state == state && (state == FREE || E.item == k)) || failed; });
        return !failed;
    };
    const int items = (n_frames + c_max - 1) / c_max;
    auto frames = [&](int k) { return std::min(c_max, n_frames - k * c_max); };
    auto band = [&](const RingPart &P) { return (size_t)(P.row1 - P.row0) * W; };

    std::thread reader([&] {
        for (int k = 0; k < items; ++k) {
            Entry &E = ring[k % RING_NS];
            if (!wait(E, FREE, k)) return;
            for (RingPart &P : parts)
                for (int j = 0; j < frames(k); ++j) {
                    const long long f = (long long)first_frame + k * c_max + j;
                    if (!read_luma(F.anchor, f, img_h, W, P.row0, P.row1, P.h_in[k % RING_NS] + j * band(P)) ||
                        (with_ori && !read_luma(F.ori, f, img_h, W, P.row0, P.row1, P.h_ori[k % RING_NS] + j * band(P)))) {
                        fail(QV_ERR_IO, std::string(who) + ": short read (file smaller than the requested frame range)");
                        return;
                    }
                }
            { std::lock_guard<std::mutex> l(mu); E.item = k; E.state = READ; }
            cv.notify_all();
        }
    });
    std::thread writer([&] {
        const std::vector<uint8_t> zeros((size_t)img_h * W / 2, 0);
        for (int k = 0; k < items; ++k) {
            Entry &E = ring[k % RING_NS];
            if (!wait(E, LAUNCHED, k)) return;
            for (const RingPart &P : parts) {
                if (cudaSetDevice(hold[P.hold].dev) != cudaSuccess || cudaEventSynchronize(P.done[k % RING_NS]) != cudaSuccess) {
                    fail(QV_ERR_CUDA, std::string(who) + ": the GPU stage failed");
                    return;
                }
                for (int j = 0; F.recon >= 0 && j < frames(k); ++j)
                    if (!write_recon_rows(F.recon, (long long)first_frame + k * c_max + j, img_h, W, P.row0, P.row1,
                                          P.h_out[k % RING_NS] + j * band(P), zeros.data())) {
                        fail(QV_ERR_IO, std::string(who) + ": write to the reconstruction file failed");
                        return;
                    }
            }
            { std::lock_guard<std::mutex> l(mu); E.state = FREE; E.launched = 0; }
            cv.notify_all();
        }
    });
    auto gpu = [&](int d) {
        int rc = QV_OK;
        if (cudaSetDevice(hold[d].dev) != cudaSuccess) { set_error("cudaSetDevice(%d) failed", hold[d].dev); rc = QV_ERR_CUDA; }
        for (int k = 0; k < items && rc == QV_OK; ++k) {
            Entry &E = ring[k % RING_NS];
            if (!wait(E, READ, k)) return;
            if ((rc = launch(d, k, k * c_max, frames(k), k % RING_NS))) break;
            { std::lock_guard<std::mutex> l(mu); if (++E.launched == (int)hold.size()) E.state = LAUNCHED; }
            cv.notify_all();
        }
        if (rc) fail(rc, "GPU " + std::to_string(hold[d].dev) + ": " + get_error());   // the message is thread-local
    };
    std::vector<std::thread> gpus;
    for (size_t d = 0; d < hold.size(); ++d) gpus.emplace_back(gpu, (int)d);
    for (std::thread &t : gpus) t.join();
    reader.join();
    writer.join();
    if (!failed) return QV_OK;
    set_error("%s", fail_msg.c_str());
    return fail_rc;
}
}  // namespace

extern "C" {

// Per-frame SSEs of the anchor and of the reconstruction against the original (vrcnn_data::psnr_pf, inference/yuv_data.cpp:98-112)
// for frames [first_frame, first_frame + n_frames): they are computed with the reconstruction (in the fused kernel, or per frame
// on the layered path) into a device array of n_frames pairs and copied out once at the end.
int qv_stream_yuv_pf(qv_net *net, const char *anchor_yuv, const char *ori_yuv, const char *recon_yuv, int first_frame, int n_frames,
                     int64_t *sse_before_pf, int64_t *sse_after_pf)
{
    if (!net || !anchor_yuv || first_frame < 0 || n_frames < 0) { set_error("qv_stream_yuv_pf: bad argument"); return QV_ERR_ARG; }
    if ((sse_before_pf || sse_after_pf) && !ori_yuv) { set_error("qv_stream_yuv_pf: an SSE was asked for but no original file given"); return QV_ERR_ARG; }
    int rc = set_device(net);
    if (rc) return rc;
    for (int j = 0; j < n_frames; ++j) {
        if (sse_before_pf) sse_before_pf[j] = 0;
        if (sse_after_pf) sse_after_pf[j] = 0;
    }
    if (n_frames == 0) return QV_OK;
    StreamFiles F;
    if ((rc = F.open_all(anchor_yuv, ori_yuv, recon_yuv))) return rc;
    const bool with_ori = F.ori >= 0;
    const size_t fpx = (size_t)net->H * net->W, cbytes = (size_t)net->batch * fpx;
    std::vector<DeviceHold> hold(1);
    DeviceHold &H = hold[0];
    H.dev = net->dev;
    // one whole-frame part; per ring entry, device buffers of a chunk and a stream for its H2D -> forward -> D2H chain
    std::vector<RingPart> parts(1);
    parts[0].row1 = net->H;
    const RingPart &P = parts[0];
    struct { uint8_t *d_in = nullptr, *d_ori = nullptr, *d_out = nullptr; cudaStream_t st = nullptr; } slot[RING_NS];
    for (auto &S : slot) {
        QV_CUDA(H.alloc(&S.d_in, cbytes));
        QV_CUDA(H.alloc(&S.d_out, cbytes));
        if (with_ori) QV_CUDA(H.alloc(&S.d_ori, cbytes));
        QV_CUDA(H.stream(&S.st));
    }
    int64_t *d_sse = nullptr;                                   // [n_frames][2]
    const size_t sse_bytes = (size_t)n_frames * 2 * sizeof(int64_t);
    QV_CUDA(H.alloc(&d_sse, sse_bytes));
    QV_CUDA(cudaMemset(d_sse, 0, sse_bytes));

    rc = stream_ring("qv_stream_yuv_pf", F, net->H, net->W, first_frame, n_frames, net->batch, parts, hold,
                     [&](int, int, int f0, int c, int r) -> int {
        const auto &S = slot[r];
        const size_t bytes = (size_t)c * fpx;
        QV_CUDA(cudaMemcpyAsync(S.d_in, P.h_in[r], bytes, cudaMemcpyHostToDevice, S.st));
        if (with_ori) QV_CUDA(cudaMemcpyAsync(S.d_ori, P.h_ori[r], bytes, cudaMemcpyHostToDevice, S.st));
        const int frc = run_forward(net, S.d_in, S.d_out, c, net->H, net->W, S.st, S.d_ori, with_ori ? d_sse + 2 * (size_t)f0 : nullptr);
        if (frc) return frc;
        QV_CUDA(cudaMemcpyAsync(P.h_out[r], S.d_out, bytes, cudaMemcpyDeviceToHost, S.st));
        QV_CUDA(cudaEventRecord(P.done[r], S.st));
        return QV_OK;
    });
    if (rc) return rc;
    H.idle();
    std::vector<int64_t> h_sse(with_ori ? (size_t)n_frames * 2 : 0);
    if (with_ori && cudaMemcpy(h_sse.data(), d_sse, sse_bytes, cudaMemcpyDeviceToHost) != cudaSuccess) {
        set_error("qv_stream_yuv_pf: copy of the SSEs failed");
        return QV_ERR_CUDA;
    }
    for (int j = 0; with_ori && j < n_frames; ++j) {
        if (sse_before_pf) sse_before_pf[j] = h_sse[2 * (size_t)j];
        if (sse_after_pf) sse_after_pf[j] = h_sse[2 * (size_t)j + 1];
    }
    return kernel_report(net);
}

int qv_stream_yuv(qv_net *net, const char *anchor_yuv, const char *ori_yuv, const char *recon_yuv, int first_frame, int n_frames,
                  int64_t *sse_before, int64_t *sse_after)
{
    // the pooled SSEs of vrcnn_data::psnr (inference/yuv_data.cpp:87-97) are the sums of the per-frame ones
    if (!net || !anchor_yuv || first_frame < 0 || n_frames < 0) { set_error("qv_stream_yuv: bad argument"); return QV_ERR_ARG; }
    if ((sse_before || sse_after) && !ori_yuv) { set_error("qv_stream_yuv: an SSE was asked for but no original file given"); return QV_ERR_ARG; }
    std::vector<int64_t> before(ori_yuv ? n_frames : 0), after(ori_yuv ? n_frames : 0);
    const int rc = qv_stream_yuv_pf(net, anchor_yuv, ori_yuv, recon_yuv, first_frame, n_frames, ori_yuv ? before.data() : nullptr,
                                    ori_yuv ? after.data() : nullptr);
    if (sse_before) *sse_before = 0;
    if (sse_after) *sse_after = 0;
    if (rc != QV_OK) return rc;
    for (size_t j = 0; j < before.size(); ++j) {
        if (sse_before) *sse_before += before[j];
        if (sse_after) *sse_after += after[j];
    }
    return QV_OK;
}

// qv_stream_yuv_pf through the strip partition, on the same ring: one part per strip handle (its own rows of each frame), one
// frame per ring entry, and per frame k the strip's input slot k & 1 on the GPU.  The GPU stage of a device drives its strips
// the way qcnn_gpu --strips does: a device with one strip alternates two streams and an event keeps the forwards in frame
// order; a device with several strips drives them all on one stream, all loads of a frame before its forwards.
int qv_strip_stream_yuv_pf(qv_net *const *nets, int n_nets, const char *anchor_yuv, const char *ori_yuv, const char *recon_yuv,
                           int first_frame, int n_frames, int64_t *sse_before_pf, int64_t *sse_after_pf)
{
    const char *who = "qv_strip_stream_yuv_pf";
    if (!nets || n_nets < 1 || !anchor_yuv || first_frame < 0 || n_frames < 0) { set_error("%s: bad argument", who); return QV_ERR_ARG; }
    if ((sse_before_pf || sse_after_pf) && !ori_yuv) { set_error("%s: an SSE was asked for but no original file given", who); return QV_ERR_ARG; }
    for (int i = 0; i < n_nets; ++i) {
        if (!nets[i]) { set_error("%s: handle %d is null", who, i); return QV_ERR_ARG; }
        for (int j = 0; j < i; ++j)
            if (nets[j] == nets[i]) { set_error("%s: handles %d and %d are the same handle", who, j, i); return QV_ERR_ARG; }
    }
    int rc;
    for (int i = 0; i < n_nets; ++i)
        if ((rc = strip_ready(nets[i], who))) return rc;
    const int img_h = nets[0]->strip.img_h, W = nets[0]->W;
    for (int i = 1; i < n_nets; ++i)
        if (nets[i]->W != W || nets[i]->strip.img_h != img_h) {
            set_error("%s: handle %d holds rows of a %dx%d frame, handle 0 of a %dx%d frame", who, i, nets[i]->W, nets[i]->strip.img_h, W, img_h);
            return QV_ERR_ARG;
        }
    if (ori_yuv && img_h > FUSED_SSE_MAX_H) { set_error("%s: frame height %d exceeds %d", who, img_h, FUSED_SSE_MAX_H); return QV_ERR_ARG; }
    {
        // strips that share a GPU are ordered by the one stream they are driven on, so this call must drive all of them
        std::lock_guard<std::mutex> l(g_strip_mu);
        for (int i = 0; i < n_nets; ++i)
            for (qv_net *o : g_strip_nets[nets[i]->dev])
                if (std::find(nets, nets + n_nets, o) == nets + n_nets) {
                    set_error("%s: GPU %d also holds a strip handle that is not in this call (strips that share a GPU are driven "
                              "together, on one stream)", who, nets[i]->dev);
                    return QV_ERR_STATE;
                }
    }
    for (int j = 0; j < n_frames; ++j) {
        if (sse_before_pf) sse_before_pf[j] = 0;
        if (sse_after_pf) sse_after_pf[j] = 0;
    }
    if (n_frames == 0) return QV_OK;
    StreamFiles F;
    if ((rc = F.open_all(anchor_yuv, ori_yuv, recon_yuv))) return rc;
    const bool with_ori = F.ori >= 0;

    // the devices in order of first use; per device its strips, and per strip its part of the ring
    std::vector<int> devices;
    std::vector<RingPart> parts(n_nets);
    for (int i = 0; i < n_nets; ++i) {
        auto d = std::find(devices.begin(), devices.end(), nets[i]->dev);
        parts[i].hold = (int)(d - devices.begin());
        if (d == devices.end()) devices.push_back(nets[i]->dev);
        parts[i].row0 = nets[i]->strip.row0;
        parts[i].row1 = nets[i]->strip.row1;
    }
    struct StripDevice {
        std::vector<int> strips;
        cudaStream_t st[2] = {};
        cudaEvent_t ev = nullptr;                                   // one strip: orders the forwards of the two streams
    };
    struct StripBuffers {
        uint8_t *d_ori[2] = {}, *d_out[2] = {};                     // per input slot
        int64_t *d_sse = nullptr;                                   // [n_frames][2]
    };
    std::vector<DeviceHold> hold(devices.size());
    std::vector<StripDevice> sd(devices.size());
    std::vector<StripBuffers> buf(n_nets);
    for (int i = 0; i < n_nets; ++i) sd[parts[i].hold].strips.push_back(i);
    const size_t sse_bytes = (size_t)n_frames * 2 * sizeof(int64_t);
    auto bytes = [&](int i) { return (size_t)(parts[i].row1 - parts[i].row0) * W; };
    // the handles' streams are this call's from here on; at the end they are idle and free to be driven on any stream again
    auto unbind = [&]() {
        std::lock_guard<std::mutex> l(g_strip_mu);
        for (int i = 0; i < n_nets; ++i) { nets[i]->strip.used = false; nets[i]->strip.last_stream = nullptr; }
    };
    unbind();
    for (size_t d = 0; d < devices.size(); ++d) {
        hold[d].dev = devices[d];
        // the strips' earlier work, on whatever stream, is complete before this call moves them onto its own streams
        QV_CUDA(cudaSetDevice(devices[d]));
        QV_CUDA(cudaDeviceSynchronize());
        for (int s = 0; s < 2; ++s) QV_CUDA(hold[d].stream(&sd[d].st[s]));
        QV_CUDA(hold[d].event(&sd[d].ev));
        for (int i : sd[d].strips) {
            for (int s = 0; s < 2; ++s) {
                QV_CUDA(hold[d].alloc(&buf[i].d_out[s], bytes(i)));
                if (with_ori) QV_CUDA(hold[d].alloc(&buf[i].d_ori[s], bytes(i)));
            }
            if (with_ori) {
                QV_CUDA(hold[d].alloc(&buf[i].d_sse, sse_bytes));
                QV_CUDA(cudaMemset(buf[i].d_sse, 0, sse_bytes));
            }
        }
    }

    rc = stream_ring(who, F, img_h, W, first_frame, n_frames, 1, parts, hold, [&](int d, int k, int, int, int r) -> int {
        const StripDevice &D = sd[d];
        const bool solo = D.strips.size() == 1;
        const int s = k & 1;
        cudaStream_t q = D.st[solo ? s : 0];
        int lrc;
        for (int i : D.strips)
            if ((lrc = qv_strip_load(nets[i], s, parts[i].h_in[r], q))) return lrc;
        if (solo && k > 0) QV_CUDA(cudaStreamWaitEvent(q, D.ev, 0));
        for (int i : D.strips)
            if (with_ori) QV_CUDA(cudaMemcpyAsync(buf[i].d_ori[s], parts[i].h_ori[r], bytes(i), cudaMemcpyHostToDevice, q));
        for (int i : D.strips) {
            const StripBuffers &B = buf[i];
            lrc = with_ori ? qv_strip_forward_sse(nets[i], s, B.d_ori[s], B.d_out[s], B.d_sse + 2 * (size_t)k, q)
                           : qv_strip_forward(nets[i], s, B.d_out[s], q);
            if (lrc) return lrc;
        }
        if (solo) QV_CUDA(cudaEventRecord(D.ev, q));
        for (int i : D.strips) {
            QV_CUDA(cudaMemcpyAsync(parts[i].h_out[r], buf[i].d_out[s], bytes(i), cudaMemcpyDeviceToHost, q));
            QV_CUDA(cudaEventRecord(parts[i].done[r], q));
        }
        return QV_OK;
    });
    std::vector<int64_t> h_sse(with_ori ? (size_t)n_frames * 2 : 0), sum(h_sse.size(), 0);
    for (size_t d = 0; d < devices.size(); ++d) {
        if (cudaSetDevice(devices[d]) != cudaSuccess && rc == QV_OK) { set_error("%s: cudaSetDevice failed", who); rc = QV_ERR_CUDA; }
        hold[d].idle();
        for (int i : sd[d].strips) {
            if (rc == QV_OK && with_ori && cudaMemcpy(h_sse.data(), buf[i].d_sse, sse_bytes, cudaMemcpyDeviceToHost) != cudaSuccess) {
                set_error("%s: copy of the SSEs failed", who);
                rc = QV_ERR_CUDA;
            }
            for (size_t x = 0; rc == QV_OK && x < sum.size(); ++x) sum[x] += h_sse[x];
        }
    }
    unbind();
    // every handle's fused-kernel report is taken (and cleared) now that its streams are idle; the first failure's message stands
    for (int i = 0; i < n_nets; ++i) {
        if (rc == QV_OK) rc = kernel_report(nets[i]);
        else if (nets[i]->fm) fused_take_failure(nets[i]->fm);
    }
    if (rc != QV_OK) return rc;
    for (int j = 0; with_ori && j < n_frames; ++j) {
        if (sse_before_pf) sse_before_pf[j] = sum[2 * (size_t)j];
        if (sse_after_pf) sse_after_pf[j] = sum[2 * (size_t)j + 1];
    }
    return QV_OK;
}

void *qv_host_alloc(size_t bytes)
{
    if (bytes == 0) bytes = 1;
    void *p = nullptr;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) == cudaSuccess && ndev > 0 && cudaHostAlloc(&p, bytes, cudaHostAllocPortable) == cudaSuccess) return p;
    cudaGetLastError();
    return malloc(bytes);
}

void qv_host_free(void *p)
{
    if (!p) return;
    cudaPointerAttributes a{};
    if (cudaPointerGetAttributes(&a, p) == cudaSuccess && a.type == cudaMemoryTypeHost) { cudaFreeHost(p); return; }
    cudaGetLastError();
    free(p);
}

int qv_device_buffers(qv_net *net, void **d_x, void **d_x_rec)
{
    if (!net) { set_error("qv_device_buffers: null handle"); return QV_ERR_ARG; }
    if (d_x) *d_x = net->d_x;
    if (d_x_rec) *d_x_rec = net->d_rec;
    return QV_OK;
}

int qv_sse_device(const uint8_t *d_a, const uint8_t *d_b, size_t n, int64_t *d_sse_accum, void *cuda_stream)
{
    if (!d_a || !d_b || !d_sse_accum) { set_error("qv_sse_device: null argument"); return QV_ERR_ARG; }
    if (n == 0) return QV_OK;
    QV_CUDA(sse_accumulate(d_a, d_b, n, d_sse_accum, (cudaStream_t)cuda_stream));
    return QV_OK;
}

int qv_set_impl(qv_net *net, int impl)
{
    if (!net || impl < QV_IMPL_AUTO || impl > QV_IMPL_FUSED) { set_error("qv_set_impl: bad argument"); return QV_ERR_ARG; }
    net->impl = impl;
    return QV_OK;
}

int qv_get_impl(const qv_net *net)
{
    if (!net) return QV_ERR_ARG;
    return runs_fused(net) ? QV_IMPL_FUSED : QV_IMPL_LAYERED;
}

long long qv_launch_count(const qv_net *net) { return net ? net->launches : 0; }

int qv_get_activation(qv_net *net, int which, int8_t *host_out)
{
    if (!net || !host_out || which < 1 || which > 3) { set_error("qv_get_activation: bad argument"); return QV_ERR_ARG; }
    int rc = set_device(net);
    if (rc) return rc;
    return layered_activation(net->ln, which, host_out, net->st);
}

}  // extern "C"
