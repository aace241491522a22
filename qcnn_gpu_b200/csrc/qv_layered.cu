// Per-layer CUDA-core path (QV_IMPL_LAYERED): one kernel per conv with the reference's
// surrounding glue folded in -- the -128 preprocess (inference/cnn.cu:445-453) into C1's tile
// load, bias add + BLU requantisation + channel concat (inference/cnn.cu:155, mat.cu:262-303,
// cnn.cu:390-391) into every conv's epilogue, and the output requantisation + residual add +
// clamp (inference/cnn.cu:507-523) into C4.  Activations live in HBM as NHWC int8.
// This path is the simple, independently written second CUDA implementation the fused tcgen05
// kernel is cross-checked against at sizes the CPU oracle cannot reach.
#include <algorithm>
#include <cstdint>
#include <vector>
#include <cuda_runtime.h>

#include "qv_device.cuh"
#include "qv_layered.h"

namespace qv {

constexpr int TX = 32, TY = 8, NT = TX * TY;

__device__ __forceinline__ int pack4(int b0, int b1, int b2, int b3)
{
    return (b0 & 0xff) | ((b1 & 0xff) << 8) | ((b2 & 0xff) << 16) | ((b3 & 0xff) << 24);
}

// ---- C1: 1 -> 64, 5x5, input u8 luma ---------------------------------------------------
// wpk[r][k][2]: word0 = taps s=0..3 of row r, word1 = tap s=4 (upper lanes 0).
__global__ void __launch_bounds__(NT) k_c1(const uint8_t *__restrict__ x, int8_t *__restrict__ a1,
                                           const int32_t *__restrict__ wpk, const int32_t *__restrict__ bias,
                                           QParam q, int H, int W)
{
    constexpr int TH = TY + 4, TW = TX + 4, PITCH = TW + 4;
    __shared__ int8_t s_x[TH * PITCH];
    __shared__ int2 s_w[5 * 64];
    __shared__ int s_b[64];
    const int tid = threadIdx.y * TX + threadIdx.x;
    const int x0 = blockIdx.x * TX, y0 = blockIdx.y * TY;
    const size_t f = blockIdx.z;
    const uint8_t *xf = x + f * (size_t)H * W;
    for (int i = tid; i < 5 * 64; i += NT) s_w[i] = reinterpret_cast<const int2 *>(wpk)[i];
    if (tid < 64) s_b[tid] = bias[tid];
    for (int i = tid; i < TH * TW; i += NT) {
        const int ty = i / TW, tx = i % TW, gy = y0 + ty - 2, gx = x0 + tx - 2;
        int v = 0;                                                  // zero pad in the x-128 domain
        if (gy >= 0 && gy < H && gx >= 0 && gx < W) v = (int)xf[(size_t)gy * W + gx] - 128;   // cnn.cu:450
        s_x[ty * PITCH + tx] = (int8_t)v;
    }
    __syncthreads();
    int acc[64];
#pragma unroll
    for (int k = 0; k < 64; ++k) acc[k] = 0;
#pragma unroll
    for (int r = 0; r < 5; ++r) {
        const int8_t *row = &s_x[(threadIdx.y + r) * PITCH + threadIdx.x];
        const int w0 = pack4(row[0], row[1], row[2], row[3]);
        const int w1 = row[4] & 0xff;
#pragma unroll
        for (int k = 0; k < 64; ++k) {
            const int2 wv = s_w[r * 64 + k];
            acc[k] = __dp4a(w0, wv.x, acc[k]);
            acc[k] = __dp4a(w1, wv.y, acc[k]);
        }
    }
    const int gx = x0 + threadIdx.x, gy = y0 + threadIdx.y;
    if (gx < W && gy < H) {
        int4 *dst = reinterpret_cast<int4 *>(a1 + ((f * H + gy) * (size_t)W + gx) * 64);
#pragma unroll
        for (int v = 0; v < 4; ++v) {
            int o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int k = v * 16 + j * 4;
                o[j] = pack4(blu_requant(acc[k] + s_b[k], q), blu_requant(acc[k + 1] + s_b[k + 1], q),
                             blu_requant(acc[k + 2] + s_b[k + 2], q), blu_requant(acc[k + 3] + s_b[k + 3], q));
            }
            dst[v] = make_int4(o[0], o[1], o[2], o[3]);
        }
    }
}

// ---- dense hidden convs: CIN -> 16 channels per block, KSxKS, NHWC int8 in/out ----------
// wpk[group][tap][c4][16] words (4 input channels per word); output written at channel
// offset out_coff + 16*group of an NHWC tensor with out_ch channels (the concat).
template <int CIN, int KS>
__global__ void __launch_bounds__(NT) k_conv(const int8_t *__restrict__ in, int8_t *__restrict__ out,
                                             const int32_t *__restrict__ wpk, const int32_t *__restrict__ bias,
                                             QParam q, int H, int W, int out_ch, int out_coff, int ngroups)
{
    constexpr int P = (KS - 1) / 2, TH = TY + KS - 1, TW = TX + KS - 1, C4 = CIN / 4;
    extern __shared__ int32_t sm[];
    int32_t *s_in = sm;                       // [C4][TH][TW]
    int32_t *s_w = sm + C4 * TH * TW;         // [KS*KS][C4][16]
    __shared__ int s_b[16];
    const int tid = threadIdx.y * TX + threadIdx.x;
    const int g = blockIdx.z % ngroups;
    const size_t f = blockIdx.z / ngroups;
    const int x0 = blockIdx.x * TX, y0 = blockIdx.y * TY;
    const int32_t *wg = wpk + (size_t)g * KS * KS * C4 * 16;
    for (int i = tid; i < KS * KS * C4 * 16; i += NT) s_w[i] = wg[i];
    if (tid < 16) s_b[tid] = bias[g * 16 + tid];
    const int8_t *inf = in + f * (size_t)H * W * CIN;
    for (int i = tid; i < TH * TW * (CIN / 16); i += NT) {
        const int chunk = i % (CIN / 16), p = i / (CIN / 16);
        const int ty = p / TW, tx = p % TW, gy = y0 + ty - P, gx = x0 + tx - P;
        int4 v = make_int4(0, 0, 0, 0);                              // SAME zero padding, cnn.cu:44-49
        if (gy >= 0 && gy < H && gx >= 0 && gx < W)
            v = *reinterpret_cast<const int4 *>(inf + ((size_t)gy * W + gx) * CIN + chunk * 16);
        int32_t *d = s_in + (chunk * 4) * TH * TW + ty * TW + tx;
        d[0] = v.x; d[TH * TW] = v.y; d[2 * TH * TW] = v.z; d[3 * TH * TW] = v.w;
    }
    __syncthreads();
    int acc[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) acc[k] = 0;
    for (int r = 0; r < KS; ++r)
        for (int s = 0; s < KS; ++s) {
            const int32_t *ap = s_in + (threadIdx.y + r) * TW + threadIdx.x + s;
            const int4 *wp = reinterpret_cast<const int4 *>(s_w + (r * KS + s) * C4 * 16);
#pragma unroll 4
            for (int c4 = 0; c4 < C4; ++c4) {
                const int a = ap[c4 * TH * TW];
#pragma unroll
                for (int v = 0; v < 4; ++v) {
                    const int4 w = wp[c4 * 4 + v];
                    acc[v * 4 + 0] = __dp4a(a, w.x, acc[v * 4 + 0]);
                    acc[v * 4 + 1] = __dp4a(a, w.y, acc[v * 4 + 1]);
                    acc[v * 4 + 2] = __dp4a(a, w.z, acc[v * 4 + 2]);
                    acc[v * 4 + 3] = __dp4a(a, w.w, acc[v * 4 + 3]);
                }
            }
        }
    const int gx = x0 + threadIdx.x, gy = y0 + threadIdx.y;
    if (gx < W && gy < H) {
        int o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
            o[j] = pack4(blu_requant(acc[4 * j] + s_b[4 * j], q), blu_requant(acc[4 * j + 1] + s_b[4 * j + 1], q),
                         blu_requant(acc[4 * j + 2] + s_b[4 * j + 2], q), blu_requant(acc[4 * j + 3] + s_b[4 * j + 3], q));
        *reinterpret_cast<int4 *>(out + ((f * H + gy) * (size_t)W + gx) * out_ch + out_coff + g * 16) =
            make_int4(o[0], o[1], o[2], o[3]);
    }
}

// ---- C4 48 -> 1, 3x3, fused with applyRes_y ----------------------------------------------
__global__ void __launch_bounds__(NT) k_c4_res(const int8_t *__restrict__ a3, const uint8_t *__restrict__ x,
                                               uint8_t *__restrict__ rec, const int32_t *__restrict__ wpk, int bias,
                                               int mul, int shift, int H, int W)
{
    constexpr int TH = TY + 2, TW = TX + 2, C4 = 12;
    __shared__ int32_t s_in[C4 * TH * TW];
    __shared__ int32_t s_w[9 * C4];
    const int tid = threadIdx.y * TX + threadIdx.x;
    const size_t f = blockIdx.z;
    const int x0 = blockIdx.x * TX, y0 = blockIdx.y * TY;
    if (tid < 9 * C4) s_w[tid] = wpk[tid];
    const int8_t *inf = a3 + f * (size_t)H * W * 48;
    for (int i = tid; i < TH * TW * 3; i += NT) {
        const int chunk = i % 3, p = i / 3;
        const int ty = p / TW, tx = p % TW, gy = y0 + ty - 1, gx = x0 + tx - 1;
        int4 v = make_int4(0, 0, 0, 0);
        if (gy >= 0 && gy < H && gx >= 0 && gx < W)
            v = *reinterpret_cast<const int4 *>(inf + ((size_t)gy * W + gx) * 48 + chunk * 16);
        int32_t *d = s_in + (chunk * 4) * TH * TW + ty * TW + tx;
        d[0] = v.x; d[TH * TW] = v.y; d[2 * TH * TW] = v.z; d[3 * TH * TW] = v.w;
    }
    __syncthreads();
    int acc = 0;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        const int32_t *ap = s_in + (threadIdx.y + t / 3) * TW + threadIdx.x + t % 3;
#pragma unroll
        for (int c4 = 0; c4 < C4; ++c4) acc = __dp4a(ap[c4 * TH * TW], s_w[t * C4 + c4], acc);
    }
    const int gx = x0 + threadIdx.x, gy = y0 + threadIdx.y;
    if (gx < W && gy < H) {
        const size_t i = (f * H + gy) * (size_t)W + gx;
        rec[i] = (uint8_t)residual_apply(acc + bias, (int)x[i], mul, shift);
    }
}

// ---- NHWC int8 -> planar [C][H][W] (debug taps only) --------------------------------------
__global__ void k_nhwc_to_planar(const int8_t *__restrict__ in, int8_t *__restrict__ out, int C, int HW)
{
    const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= (size_t)C * HW) return;
    const int c = (int)(i / HW);
    const size_t p = i % HW;
    out[i] = in[p * C + c];
}

// ---- exact int64 SSE (PSNR core, inference/yuv_data.cpp:92-93) -----------------------------
__global__ void __launch_bounds__(256) k_sse(const uint8_t *__restrict__ a, const uint8_t *__restrict__ b, size_t n,
                                             unsigned long long *__restrict__ accum)
{
    unsigned long long s = 0;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const size_t n16 = n / 16;
    const bool aligned = ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b)) & 15) == 0;
    size_t done = 0;
    if (aligned) {
        const uint4 *a4 = reinterpret_cast<const uint4 *>(a), *b4 = reinterpret_cast<const uint4 *>(b);
        for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n16; i += stride) {
            const uint4 va = a4[i], vb = b4[i];
            const unsigned wa[4] = {va.x, va.y, va.z, va.w}, wb[4] = {vb.x, vb.y, vb.z, vb.w};
            unsigned t = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j)
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int d = (int)((wa[j] >> (8 * k)) & 0xff) - (int)((wb[j] >> (8 * k)) & 0xff);
                    t += (unsigned)(d * d);
                }
            s += t;
        }
        done = n16 * 16;
    }
    for (size_t i = done + blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += stride) {
        const int d = (int)a[i] - (int)b[i];
        s += (unsigned)(d * d);
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __shared__ unsigned long long ws[8];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int w = 0; w < 8; ++w) t += ws[w];
        atomicAdd(accum, t);
    }
}

// ---- host side --------------------------------------------------------------------------
struct LayeredLayer {
    int32_t *d_wpk = nullptr;   // packed weights (layout documented at each kernel)
    int32_t *d_bias = nullptr;  // int32 bias[cout]
    QParam q{};
    int cout = 0;
};

struct LayeredNet {
    int batch = 0, H = 0, W = 0;                // the handle's geometry
    LayeredLayer L[QV_NLAYER];
    int c4_bias = 0;
    // C1.v, Conc1.conc, Conc2.conc of the reference (inference/cnn.cu:64,281), NHWC here; the reference also holds 644 B/px
    // of fp32 `u` tensors which this design never materialises.
    int8_t *a1 = nullptr, *a2 = nullptr, *a3 = nullptr;
    int act_frames = 0;
    uint8_t *rows = nullptr;                    // the window of layered_forward_rows, run as an image of its own
    size_t rows_bytes = 0;
    cudaEvent_t ev = nullptr;                   // recorded after the last launch or copy of every call that uses a1..a3 / rows
};

cudaError_t layered_create(LayeredNet **out, int batch, int H, int W)
{
    *out = new LayeredNet{batch, H, W};
    return cudaEventCreateWithFlags(&(*out)->ev, cudaEventDisableTiming);
}

static void free_weights(LayeredNet *ln)
{
    for (LayeredLayer &D : ln->L) { cudaFree(D.d_wpk); cudaFree(D.d_bias); D = LayeredLayer{}; }
}

void layered_free(LayeredNet *ln)
{
    if (!ln) return;
    free_weights(ln);
    cudaFree(ln->a1); cudaFree(ln->a2); cudaFree(ln->a3);
    cudaFree(ln->rows);
    if (ln->ev) cudaEventDestroy(ln->ev);
    delete ln;
}

static int pack_word(const int8_t *p, int stride, int n)
{
    int v = 0;
    for (int j = 0; j < n; ++j) v |= ((int)(uint8_t)p[j * stride]) << (8 * j);
    return v;
}

// Re-pack the plain [K][C][R][S] host weights into the word layouts the kernels above read.
int layered_load(LayeredNet *ln, const ModelHost &m, cudaStream_t st)
{
    free_weights(ln);
    for (int l = 0; l < QV_NLAYER; ++l) {
        const LayerShape &s = kLayers[l];
        const LayerHost &L = m.L[l];
        std::vector<int32_t> wpk;
        const int R = s.k;
        if (l == QV_C1) {                        // [r][k][2]
            wpk.assign(5 * 64 * 2, 0);
            for (int r = 0; r < 5; ++r)
                for (int k = 0; k < 64; ++k) {
                    const int8_t *row = &L.w[((size_t)k * 5 + r) * 5];
                    wpk[(r * 64 + k) * 2 + 0] = pack_word(row, 1, 4);
                    wpk[(r * 64 + k) * 2 + 1] = pack_word(row + 4, 1, 1);
                }
        } else if (l == QV_C4) {                 // [tap][c4]
            wpk.assign(9 * 12, 0);
            for (int t = 0; t < 9; ++t)
                for (int c4 = 0; c4 < 12; ++c4)
                    wpk[t * 12 + c4] = pack_word(&L.w[((size_t)(4 * c4) * 3 + t / 3) * 3 + t % 3], 9, 4);
        } else {                                 // [group][tap][c4][16]
            const int C4 = s.cin / 4, G = s.cout / 16;
            wpk.assign((size_t)G * R * R * C4 * 16, 0);
            for (int g = 0; g < G; ++g)
                for (int t = 0; t < R * R; ++t)
                    for (int c4 = 0; c4 < C4; ++c4)
                        for (int j = 0; j < 16; ++j) {
                            const int k = g * 16 + j;
                            wpk[(((size_t)g * R * R + t) * C4 + c4) * 16 + j] =
                                pack_word(&L.w[(((size_t)k * s.cin + 4 * c4) * R + t / R) * R + t % R], R * R, 4);
                        }
        }
        LayeredLayer &D = ln->L[l];
        D.cout = s.cout;
        D.q.blu = L.blu; D.q.mul = L.mul; D.q.shift = L.shift;
        D.q.rbias = (1 << (L.shift - 1)) / L.mul;                       // inference/mat.cu:268
        QV_CUDA(cudaMalloc(&D.d_wpk, wpk.size() * sizeof(int32_t)));
        QV_CUDA(cudaMalloc(&D.d_bias, L.b.size() * sizeof(int32_t)));
        QV_CUDA(cudaMemcpyAsync(D.d_wpk, wpk.data(), wpk.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        QV_CUDA(cudaMemcpyAsync(D.d_bias, L.b.data(), L.b.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        QV_CUDA(cudaStreamSynchronize(st));   // wpk is a local
    }
    ln->c4_bias = m.L[QV_C4].b[0];
    return QV_OK;
}

template <int CIN, int KS>
static cudaError_t launch_conv(const int8_t *in, int8_t *out, const LayeredLayer &L, int n, int H, int W, int out_ch,
                               int out_coff, cudaStream_t st)
{
    constexpr int TH = TY + KS - 1, TW = TX + KS - 1, C4 = CIN / 4;
    const size_t smem = sizeof(int32_t) * (size_t)(C4 * TH * TW + KS * KS * C4 * 16);
    // function attributes are per device: set it on every launch (a few hundred ns) so that handles on
    // several GPUs of one process all get it
    cudaError_t e = cudaFuncSetAttribute(k_conv<CIN, KS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    const int ngroups = L.cout / 16;
    dim3 grid((W + TX - 1) / TX, (H + TY - 1) / TY, n * ngroups), block(TX, TY);
    k_conv<CIN, KS><<<grid, block, smem, st>>>(in, out, L.d_wpk, L.d_bias, L.q, H, W, out_ch, out_coff, ngroups);
    return cudaGetLastError();
}

// The scratch is allocated at the first forward; n frames run in chunks of as many frames as it holds.
int layered_forward(LayeredNet *ln, const uint8_t *d_in, uint8_t *d_out, int n, int H, int W, cudaStream_t st,
                    long long *launches, const uint8_t *d_ori, int64_t *d_sse)
{
    if (!ln->a1) {
        const int frames = std::min(ln->batch, 8);
        const size_t px = (size_t)frames * ln->H * ln->W;
        QV_CUDA(cudaMalloc(&ln->a1, px * 64));
        QV_CUDA(cudaMalloc(&ln->a2, px * 48));
        QV_CUDA(cudaMalloc(&ln->a3, px * 48));
        ln->act_frames = frames;
    }
    const size_t cap_px = (size_t)ln->act_frames * ln->H * ln->W, fpx = (size_t)H * W;
    if (fpx > cap_px) { set_error("frame of %dx%d exceeds the handle's activation scratch", W, H); return QV_ERR_ARG; }
    QV_CUDA(cudaStreamWaitEvent(st, ln->ev, 0));
    const int chunk = (int)std::max<size_t>(1, cap_px / fpx);
    const LayeredLayer *L = ln->L;
    int8_t *a1 = ln->a1, *a2 = ln->a2, *a3 = ln->a3;
    for (int f0 = 0; f0 < n; f0 += chunk) {
        const int c = std::min(chunk, n - f0);
        const uint8_t *in = d_in + (size_t)f0 * fpx;
        const dim3 block(TX, TY), grid((W + TX - 1) / TX, (H + TY - 1) / TY, c);
        k_c1<<<grid, block, 0, st>>>(in, a1, L[QV_C1].d_wpk, L[QV_C1].d_bias, L[QV_C1].q, H, W);
        QV_CUDA(cudaGetLastError());
        QV_CUDA(launch_conv<64, 3>(a1, a2, L[QV_C2_1], c, H, W, 48, 0, st));
        QV_CUDA(launch_conv<64, 5>(a1, a2, L[QV_C2_2], c, H, W, 48, 32, st));
        QV_CUDA(launch_conv<48, 3>(a2, a3, L[QV_C3_1], c, H, W, 48, 0, st));
        QV_CUDA(launch_conv<48, 1>(a2, a3, L[QV_C3_2], c, H, W, 48, 16, st));
        k_c4_res<<<grid, block, 0, st>>>(a3, in, d_out + (size_t)f0 * fpx, L[QV_C4].d_wpk, ln->c4_bias, L[QV_C4].q.mul,
                                         L[QV_C4].q.shift, H, W);
        QV_CUDA(cudaGetLastError());
        *launches += 6;
    }
    if (d_sse) {
        for (int f = 0; f < n; ++f) {
            const size_t o = (size_t)f * fpx;
            QV_CUDA(sse_accumulate(d_in + o, d_ori + o, fpx, d_sse + 2 * f, st));
            QV_CUDA(sse_accumulate(d_out + o, d_ori + o, fpx, d_sse + 2 * f + 1, st));
        }
        *launches += 2 * n;
    }
    QV_CUDA(cudaEventRecord(ln->ev, st));
    return QV_OK;
}

int layered_forward_rows(LayeredNet *ln, const uint8_t *d_in, int in_rows, uint8_t *d_out, int out0, int out1, cudaStream_t st,
                         long long *launches)
{
    const size_t W = ln->W, need = (size_t)in_rows * W;
    if (need > (size_t)ln->batch * ln->H * ln->W) {
        set_error("qv_forward_rows_device: window larger than the handle's geometry");
        return QV_ERR_ARG;
    }
    if (ln->rows_bytes < need) {
        QV_CUDA(cudaEventSynchronize(ln->ev));     // the buffer's last user, on whatever stream
        cudaFree(ln->rows);
        ln->rows = nullptr; ln->rows_bytes = 0;
        QV_CUDA(cudaMalloc(&ln->rows, need));
        ln->rows_bytes = need;
    }
    const int rc = layered_forward(ln, d_in, ln->rows, 1, in_rows, ln->W, st, launches, nullptr, nullptr);
    if (rc) return rc;
    QV_CUDA(cudaMemcpyAsync(d_out, ln->rows + (size_t)out0 * W, (size_t)(out1 - out0) * W, cudaMemcpyDeviceToDevice, st));
    QV_CUDA(cudaEventRecord(ln->ev, st));       // again: the next user of the buffer waits for the copy too
    return QV_OK;
}

int layered_activation(LayeredNet *ln, int which, int8_t *host_out, cudaStream_t st)
{
    if (!ln->a1) { set_error("qv_get_activation: the layered path has not run on this handle"); return QV_ERR_STATE; }
    const int C = which == 1 ? 64 : 48;
    const int8_t *src = which == 1 ? ln->a1 : (which == 2 ? ln->a2 : ln->a3);
    const size_t HW = (size_t)ln->H * ln->W, n = HW * C;
    int8_t *tmp = nullptr;
    QV_CUDA(cudaStreamWaitEvent(st, ln->ev, 0));
    QV_CUDA(cudaMalloc(&tmp, n));
    k_nhwc_to_planar<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(src, tmp, C, (int)HW);
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess) e = cudaMemcpyAsync(host_out, tmp, n, cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaEventRecord(ln->ev, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(tmp);
    QV_CUDA(e);
    return QV_OK;
}

cudaError_t sse_accumulate(const uint8_t *a, const uint8_t *b, size_t n, int64_t *d_accum, cudaStream_t st)
{
    int blocks = (int)((n / 16 + 255) / 256);
    if (blocks < 1) blocks = 1;
    if (blocks > 148 * 8) blocks = 148 * 8;
    k_sse<<<blocks, 256, 0, st>>>(a, b, n, reinterpret_cast<unsigned long long *>(d_accum));
    return cudaGetLastError();
}

}  // namespace qv
