// Internal host-side types shared by the C-ABI translation units (not installed).
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

#include "../../include/qvrcnn_b200.h"

namespace qv {

// Layer table of inference/qvrcnn.cu:11-18.
struct LayerShape { int cin, cout, k; };
static const LayerShape kLayers[QV_NLAYER] = {
    {1, 64, 5}, {64, 32, 3}, {64, 16, 5}, {48, 16, 3}, {48, 32, 1}, {48, 1, 3}};

struct LayerHost {
    std::vector<int8_t> w;    // plain [K][C][R][S]
    std::vector<int32_t> b;   // [K]
    int32_t blu = 0, mul = 0, shift = 0;
    bool have_w = false, have_q = false;
};

struct ModelHost {
    LayerHost L[QV_NLAYER];
    bool complete() const {
        for (int l = 0; l < QV_NLAYER; ++l)
            if (!L[l].have_w || !L[l].have_q) return false;
        return true;
    }
};

void set_error(const char *fmt, ...);
const char *get_error();

// In a function returning a QV_* code (CUDA translation units): a failed CUDA call sets the message and returns QV_ERR_CUDA.
// Variadic so that template arguments may contain commas.
#define QV_CUDA(...)                                                                        \
    do {                                                                                    \
        cudaError_t e__ = (__VA_ARGS__);                                                    \
        if (e__ != cudaSuccess) {                                                           \
            set_error("%s failed: %s (%s:%d)", #__VA_ARGS__, cudaGetErrorString(e__), __FILE__, __LINE__); \
            return QV_ERR_CUDA;                                                             \
        }                                                                                   \
    } while (0)

// formats (qv_formats.cpp)
size_t model_file_size_vect_c();
size_t model_file_size_hwcn();
int parse_model_vect_c(const uint8_t *buf, size_t len, ModelHost &m);
int parse_model_hwcn(const uint8_t *buf, size_t len, ModelHost &m);
std::vector<uint8_t> serialize_model_vect_c(const ModelHost &m);
int read_file(const char *path, std::vector<uint8_t> &out);
int parse_quant_params(const uint8_t *buf, size_t len, int32_t *out18);
// Exact-integer envelope (SURVEY fact 7): 128*sum|w| + |b| < 2^24 for every output channel.
int check_fp32_exact_envelope(const ModelHost &m);

}  // namespace qv
