// Fused QVRCNN forward for sm_100a: the whole network per column strip, activations resident in
// shared memory, the five dense convolutions as tcgen05.mma kind::i8 implicit GEMMs with int32
// accumulators in TMEM, the 48 -> 1 output layer on CUDA cores; HBM sees one luma byte in and one
// reconstructed byte out per pixel.  Replaces, for one frame batch, the whole of qvrcnn::forward_blu
// (inference/qvrcnn.cu:168-242): ppro, 6 x (cudnnConvolutionForward + cudnnAddTensor),
// quantize_out_blu / concat_blu, applyRes_y.
//
// Geometry.  A CTA owns a work unit = (frame, column strip of WT=120 output pixels, row segment)
// and rolls down the rows.  Every activation row lives in smem as [16-channel plane][pixel][16 B]
// with a pixel pitch of PW=136: the canonical no-swizzle K-major UMMA operand layout (8-pixel x
// 16-byte core matrices, SBO = 128 B, LBO = plane stride), so a horizontal tap s is nothing but a
// different start address in the A descriptor.  Buffer pixel p of a strip whose first output
// column is X0 maps to image column X0 - 8 + p:
//   input  p in [2,134)   a1: p = 4+m   a2: p = 6+m   a3: p = 7+m   out: p = 8+m  (m = MMA row)
//
// Row scatter with accumulator rings.  An M=128 int8 MMA costs >= 44 cycles whatever N is (measured,
// profiles/r1_probe_thr2.log), so per-tap MMAs with N = 16..48 waste the tensor pipe and, worse,
// re-read every activation row from smem once per vertical tap.  Instead each activation row is
// read once per horizontal shift and multiplied by the weights of ALL vertical taps at once:
//   D[pixel, (out_row, k)] += A[in_row, pixel+s][c] * W[r = in_row - out_row + pad][s][c][k]
// The accumulators of the output rows in flight form a ring in TMEM (slot = out_row mod ring
// size); one MMA covers the whole ring, so N = 96 / 128 / 64.  The B operand for a ring of R
// slots is stored as the block sequence [r_max .. r_0, Z] repeated (Z = zero block) and the
// rotation that matches "slot = row mod R" is a start-address offset into it.  The slot of the
// output row completed one step ago sits under the Z block (the MMA adds 0 to it) while the
// workers drain it; the slot of the row that starts now is zeroed by one small MMA with a zero A.
//
// Collector reuse.  60 % of the tensor core's shared-memory traffic is the A operand, re-read by every
// MMA.  MMAs that multiply the SAME activation tile are therefore issued back to back and the second takes
// A from the tensor core's collector (collector::a::fill -> ::lastuse, tools/umma_probe3.cu): C2_2 shift s
// and C2_1 shift s-1 read the same a1 tile, C3_1's centre-tap K-steps and C3_2's two K-steps read the same
// a2 tiles, and the three ring-slot initialisations share the zero tile.
//
// Pipeline.  9 warps, three roles; iteration i, R1 = y0-4+i:
//   warp 4, MMA issue : 27 MMAs per iteration -- C1 for a1 row R1 (im2col operand); the three ring-slot
//                initialisations; C3_1 scatter and C3_2 of a2 row R1-6; C2_2 and C2_1 scatter of a1 row R1-2
//                (the wide MMAs last: they execute slower than they issue, so the tensor pipe still has a
//                backlog during the handshake).  Both descriptors of every MMA come ready-made from a 12-phase table
//                in constant memory (the ring rotations have periods 2, 3, 4, 6), one uniform load per MMA: the issue
//                loop executes no ALU-pipe instruction, which matters because the worker warps of the same SM
//                sub-partition saturate that pipe (profiles/r1_probe3_contention*), and it is this warp's serial
//                work that bounds the kernel.
//   warps 0-3, workers: drain what iteration i-1 completed, TMEM -> requantise -> st.shared: a1 row R1-1; a2 row
//                R1-5 plane 2 (C2_2) and a2 row R1-4 planes 0,1 (C2_1); a3 row R1-8 plane 0 (C3_1) and a3 row
//                R1-7 planes 1,2 (C3_2).  A warp can only read its own TMEM lane quarter, so warp q owns quarter q
//                (pixels 32q .. 32q+31) and drains all ten of its 16-column groups.
//   warps 5-8, C4     : everything that needs no TMEM -- the input ring (global loads one row ahead), the C1
//                operand of a1 row R1+1 (im2col, three stages), C4 on a3 row R1-9 (9 LDS.128 + 108 dp4a per
//                pixel, two running sums carry the partial output rows), applyRes_y and the store of output row
//                R1-10.
// Workers and C4 warps arrive on a named barrier (three ids in rotation) in which the MMA warp blocks before it issues the
// next MMAs, the MMA warp commits to an mbarrier pair that releases the workers, and a second named barrier per iteration
// publishes the a3 rows to the C4 warps.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <type_traits>
#include <vector>

#include <cuda.h>
#include <cuda_runtime.h>

#include "qv_device.cuh"
#include "qv_fused.h"
#include "qv_tcgen05.cuh"


// Code alignment.  The SM's L0 instruction cache works on 128-byte lines (8 instructions) and holds ~6 KB; the three roles' loops
// are ~13 KB per sub-partition, so every warp keeps refetching, and where the loops start relative to a line boundary is worth
// up to 2.4 % (profiles/r2_kernel_ab_code_alignment.log: 5.90 ... 6.04 ms for the eight alignments, period 128 bytes).
// QV_CODE_SHIFT puts that many extra instructions (membar.cta, executed once) in front of the code of all roles; re-run the
// search over its eight values after any edit of the kernel (DESIGN.md section 7).
#ifndef QV_CODE_SHIFT
#define QV_CODE_SHIFT 5          // best of the eight positions for this source (profiles/r2_kernel_ab_row_line_decomposition.log)
#endif

namespace qv {
namespace {
using namespace tc;

constexpr int WT = 120;                    // output columns per strip
constexpr int PW = 136;                    // pixel pitch of every activation row buffer
constexpr int PLANE = PW * 16;             // bytes of one 16-channel plane of one row
constexpr int A_SLOTS = 3, IN_SLOTS = 32, IN_PITCH = 144;
constexpr int A1_ROW = 4 * PLANE, A2_ROW = 3 * PLANE;
constexpr int IM_BYTES = 2 * 128 * 16;     // one im2col A operand for C1: [2 K-planes][128 px][16 B]
constexpr int ZERO_BYTES = 2 * 128 * 16;   // all-zero A operand (ring-slot initialisation)

// ---- B operands (weights) in smem: every block is [2 K-chunks][NR rows][16 B] ---------------------
constexpr int NR22 = 11 * 16, NR21 = 7 * 32, NR31 = 7 * 16, NR32 = 32;
constexpr int W1_BYTES = 2 * 64 * 16;
constexpr int T22 = 2 * NR22 * 16, T21 = 2 * NR21 * 16, T31 = 2 * NR31 * 16, T32 = 2 * NR32 * 16;
constexpr int OFF_W1 = 0;
constexpr int OFF_W22 = OFF_W1 + W1_BYTES;      // 10 tiles (s, h)
constexpr int OFF_W21 = OFF_W22 + 10 * T22;     //  6 tiles (s', h)
constexpr int OFF_W31 = OFF_W21 + 6 * T21;      //  5 K-steps
constexpr int OFF_W32 = OFF_W31 + 5 * T31;      //  2 K-steps
constexpr int OFF_BIAS = OFF_W32 + 2 * T32;
constexpr int BIAS_INTS = 64 + 48 + 48;
constexpr int WIMG_BYTES = OFF_BIAS + BIAS_INTS * 4;         // what lives in global memory per model
constexpr int OFF_A1 = (WIMG_BYTES + 127) / 128 * 128;
constexpr int OFF_A2 = OFF_A1 + A_SLOTS * A1_ROW;
constexpr int OFF_IM = OFF_A2 + A_SLOTS * A2_ROW;
constexpr int OFF_ZERO = OFF_IM + 3 * IM_BYTES;   // three im2col stages: stage (i+1)%3 is written while C1 of iteration i-1 may still read (i-1)%3
constexpr int OFF_IN = OFF_ZERO + ZERO_BYTES;
constexpr int OFF_A3 = (OFF_IN + IN_SLOTS * IN_PITCH + 15) / 16 * 16;   // a3 rows for the C4 warps: 3 slots x [3 planes][pixel][16 B]
constexpr int OFF_CTRL = OFF_A3 + A_SLOTS * A2_ROW;
constexpr int SMEM_BYTES = OFF_CTRL + 64;
static_assert(SMEM_BYTES <= 232448, "exceeds the 227 KB of dynamic shared memory per CTA");
// TMA variant of the input ring (QV_FUSED_TMA): rows land by cp.async.bulk.tensor, whose destination must be 128-byte aligned
constexpr int IN_PITCH_T = 256, IN_BOX = 144;
constexpr int OFF_IN_T = (SMEM_BYTES + 127) / 128 * 128;
constexpr int SMEM_BYTES_T = OFF_IN_T + IN_SLOTS * IN_PITCH_T;
static_assert(SMEM_BYTES_T <= 232448, "exceeds the 227 KB of dynamic shared memory per CTA");

constexpr int NWORKER = 128, NC4 = 128, NTHREADS = NWORKER + 32 + NC4;   // warps 0-3 workers (one per TMEM lane quarter), 4 MMA issue, 5-8 C4
constexpr int MMA_WARP = NWORKER / 32;
constexpr int TR_ITER0 = 300, TR_N = 8;    // profile-mode timeline window
constexpr int PIPE = 14;                   // pipeline depth in rows: output row y0 appears at iteration 14

// ---- TMEM columns (int32 accumulators) -------------------------------------------------------------
constexpr int TM_D1 = 0;        // C1: 2 x 64, double-buffered by iteration parity
constexpr int TM_R22 = 128;     // C2_2 ring: 6 slots x 16
constexpr int TM_R21 = 224;     // C2_1 ring: 4 slots x 32
constexpr int TM_R31 = 352;     // C3_1 ring: 4 slots x 16
constexpr int TM_D32 = 416;     // C3_2: 2 x 32, double-buffered
constexpr int TM_COLS = 512;

// Per 16-column accumulator group: everything the requantiser needs.
struct GroupQ {
    int hi;          // FAST: blu + rbias          (upper clamp of acc + bias')
    unsigned M;      // FAST: mul << (24 - shift)  (q = byte 3 of t * M)
    int blu, mul, shift, rbias;   // generic path: the reference formula verbatim
};

struct alignas(64) FusedParams {
    CUtensorMap tmap_in;               // TMA variant: the input as a 2-D byte tensor {W, n_frames * H}, box {IN_BOX, 1}
    // Row r of frame f is read at in + f*frame_stride + r*W and written at out + f*frame_stride + r*W: `in` / `out` are
    // VIRTUAL bases (buffer pointer minus first-row offset) when the buffers hold only a row window of the image.
    const uint8_t *in;
    uint8_t *out;
    const uint8_t *wimg;
    int n_frames, H, W, nstrips, nseg, seg_rows, n_units, linear, perm_q, perm_s0, perm_r;
    // Spatial partition of one frame over several GPUs (qv_strip_*): this launch produces image rows [ys, ye); `in` holds
    // rows [own0, own1); rows [rlo, own0) are read through in_top and rows [own1, rhi) through in_bot -- virtual bases too,
    // pointing into the NEIGHBOUR GPUs' memory (peer-mapped over NVLink), valid once *flag_top / *flag_bot have reached
    // `seq`.  A whole-frame launch has ys = own0 = rlo = 0, ye = own1 = rhi = H and no flags.
    int ys, ye, own0, own1, rlo, rhi;
    size_t frame_stride;
    const uint8_t *in_top, *in_bot;
    const uint32_t *flag_top, *flag_bot;   // the neighbours' "rows published" words
    uint32_t *pub, *done, *done_ctr;       // this GPU's own words: published sequence number, completed sequence number
    uint32_t seq;
    GroupQ q1, q22, q21, q31, q32;
    int c4_bias, c4_mul, c4_shift;
    int c4_w[108];                     // C4 weights [tap][plane][4 words], 4 channels per word (CUDA-core dp4a)
    long long *dbg;                    // optional per-block phase timers (QV_FUSED_PROFILE=1), else null
    uint32_t sbase16, tmem_base;       // what the operand table was built for (checked by the kernel)
    int *fail_flag;                    // mapped host memory: a CTA that detects a failure reports it here
    int dbg_flags;                     // profiling build only (QV_FUSED_PROFILE + QV_FUSED_EXPERIMENT): 1 = issue no MMAs, 2 = skip the drains
    int bias[BIAS_INTS];               // per accumulator column: layer bias (+ rounding bias on the FAST path)
    // k_enh_sse only: the original luma, addressed like `out` (virtual base, same rows), and the per-frame SSE pairs
    // {sum (anchor - ori)^2, sum (rec - ori)^2} of frame f at sse[2f], sse[2f + 1] (incremented).  Kept behind every
    // other field so that k_fused's parameter offsets, and with them its code, do not move.
    const uint8_t *ori;
    unsigned long long *sse;
};

// Frame lists (k_enh_list): the frame table of one launch, passed by value behind FusedParams in the kernel parameters, so
// that it needs no device copy and no lifetime rule.  The units are cut from one row line over every (frame, strip column)
// column, column c of frame f being H_f rows long: line0 / col0 are the line position and the index of the frame's first
// column, and the entry behind the last frame holds the line length and the column count.
struct ListFrame {
    const uint8_t *in;
    uint8_t *out;
    const uint8_t *ori;
    int H, W, line0, col0;
};
struct alignas(64) FusedListParams {
    FusedParams p;                     // first member: the body's P is this, at the offsets every other kernel uses
    ListFrame fr[QV_FRAME_LIST_LAUNCH_MAX + 1];
};
static_assert(sizeof(FusedListParams) <= 32764, "exceeds the kernel-parameter limit: lower QV_FRAME_LIST_LAUNCH_MAX");
static_assert(std::is_standard_layout<FusedListParams>::value, "list_of() reads the table through a FusedParams reference");

// Operands of the 27 MMAs of one row iteration, for each of the 12 phases R1 mod 12 (the ring rotations have periods 2,
// 3, 4 and 6).  PhaseBases / FixedBases are the host-side description (what rotates, what does not); PhaseOps is its
// expansion into ready-made descriptors in constant memory, so that the MMA warp needs uniform-datapath loads only:
// measured (profiles/r1_probe3_contention*.log), integer ALU work of the worker warps that share the MMA warp's SM
// sub-partition starves exactly the ALU-pipe instructions (address arithmetic, R2UR) an issue loop would otherwise
// need, and the tensor pipe's queue is only a handful of instructions deep.
struct PhaseBases {                    // low descriptor words (16-byte units | LBO << 16) and TMEM addresses that rotate with R1
    uint32_t im, a1_r2, a2_r6, b22;    // C1 operand stage ; a1 row R1-2 ; a2 row R1-6 ; C2_2 ring window start
    uint32_t b21, b31, d1, d32;        // C2_1 / C3_1 ring window starts ; C1 / C3_2 accumulator stages
    uint32_t z22, z21, z31, pad;       // ring slots of the rows that start in this iteration
};
struct FixedBases { uint32_t zeroA, w1, w32, r22, r21, r31, pad0, pad1; };   // what does not rotate
constexpr int N_PHASE = 12;
constexpr int N_MMA = 27;
struct PhaseOps {
    uint4 ab[N_MMA];                   // {A lo, A hi, B lo, B hi} in issue order
    uint32_t d1, d32, z22, z21, z31, pad[3];
};
__constant__ PhaseOps c_ops[N_PHASE];

__host__ __device__ __forceinline__ int mod_pos(int a, int m) { int r = a % m; return r < 0 ? r + m : r; }

// Ring indices without divisions: c3 / c6 track R1 mod 3 / mod 6 incrementally; (c - k) mod n for a
// compile-time k is one compare-and-add.  Powers of two use masks on R1 + 4096 (R1 may be negative).
__host__ __device__ __forceinline__ int wrap_sub(int c, int k, int n) { const int v = c - (k % n); return v < 0 ? v + n : v; }
__host__ __device__ __forceinline__ int wrap_inc(int c, int n) { return c + 1 == n ? 0 : c + 1; }

// One lane polls the mbarrier (every try_wait is a shared-memory access that competes with the tensor
// core's operand fetches: 256 pollers measurably slow the MMAs down), the rest of the warp parks at
// __syncwarp, which also carries the acquired memory ordering to them.
__device__ __forceinline__ void warp_wait(uint64_t *bar, uint32_t parity, int lane, int *fail)
{
    if (lane == 0 && !tc::mbar_wait(bar, parity)) *fail = 1;
    __syncwarp();
}

// Strip mode: spin (bounded, ~2 s) until a neighbour GPU's "rows published" word has reached `seq`.  The acquire at system
// scope orders the halo-row loads that follow behind the neighbour's release (k_fused publishes at its start: the rows
// were complete before the launch by stream order).
__device__ __forceinline__ bool peer_wait(const uint32_t *flag, uint32_t seq)
{
    for (int n = 0; n < 4000000; ++n) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if ((int)(v - seq) >= 0) return true;
        __nanosleep(200);
    }
    return false;
}

// Row-window launches deal the work out by ROWS, not by whole segments: the nstrips x (ye - ys) row-iterations of the
// launch form one line, CTA b takes [b * chunk, (b + 1) * chunk) of it, and that range is cut where it crosses into the next
// strip column: unit = b + j * gridDim.x is the j-th piece.  (One 8K frame over 8 GPUs leaves 64 columns of 540 rows for 148
// SMs: equal segments use 128 of them for 284 iterations, the line gives every SM 234 rows + the pipeline fill.)
// ok = false for a piece that does not exist.
struct UnitGeo { int strip, f, y0, y1; bool ok; };
template <bool ROWS>
__host__ __device__ __forceinline__ UnitGeo unit_geo(const FusedParams &P, int unit, int H, int grid)
{
    UnitGeo g;
    if (!ROWS && P.linear) {           // whole frames, dealt out by rows: the line runs over all (frame, strip) columns
        const int b = unit % grid, j = unit / grid;
        const int lo = b * P.seg_rows, hi = min(P.n_frames * P.nstrips * H, lo + P.seg_rows), c = lo / H + j;
        const int start = j == 0 ? lo : c * H, end = min(hi, (c + 1) * H);
        // position c on the line -> column q + s * perm_q: CTAs b and b + 1 are ~perm_s positions apart, so they work on
        // neighbouring strip columns of one frame at the same time and the shared halo columns and output sectors meet in L2
        const int full = P.perm_r * (P.perm_s0 + 1);
        const int q = c < full ? c / (P.perm_s0 + 1) : P.perm_r + (c - full) / P.perm_s0;
        const int sl = c < full ? c - q * (P.perm_s0 + 1) : (c - full) - (q - P.perm_r) * P.perm_s0;
        const int col = q + sl * P.perm_q;
        g.f = col / P.nstrips;
        g.strip = col - g.f * P.nstrips;
        g.y0 = start - c * H;
        g.y1 = g.y0 + (end - start);
        g.ok = start < end;
    } else if (!ROWS) {                // whole frames: (frame, strip column, equal row segment)
        const int seg = unit % P.nseg;
        g.strip = (unit / P.nseg) % P.nstrips;
        g.f = unit / (P.nseg * P.nstrips);
        g.y0 = seg * P.seg_rows;
        g.y1 = min(H, g.y0 + P.seg_rows);
        g.ok = true;
    } else {
        const int R = P.ye - P.ys, b = unit % grid, j = unit / grid;
        const int lo = b * P.seg_rows, hi = min(P.nstrips * R, lo + P.seg_rows), c0 = lo / R;
        const int start = j == 0 ? lo : (c0 + j) * R, end = min(hi, (c0 + j + 1) * R);
        g.strip = c0 + j;
        g.f = 0;
        g.y0 = P.ys + (start - g.strip * R);
        g.y1 = g.y0 + (end - start);
        g.ok = start < end;
    }
    return g;
}

// The frame table of a k_enh_list launch, from the FusedParams at its start.
__host__ __device__ __forceinline__ const FusedListParams &list_of(const FusedParams &P)
{
    return reinterpret_cast<const FusedListParams &>(P);
}

// The last frame of the list whose first column starts at or before line position (by_col: column index) v.  A binary
// search over the table's prefix sums, once per unit.
__host__ __device__ __forceinline__ int list_find(const FusedListParams &L, int v, bool by_col)
{
    int lo = 0, hi = L.p.n_frames - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if ((by_col ? L.fr[mid].col0 : L.fr[mid].line0) <= v) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// Frame lists: CTA b takes [b * chunk, (b + 1) * chunk) of the row line, and unit b + j * grid is the part of it in the j-th
// column it touches, as in the whole-frame line but without the column permutation (unit_geo): g.f is the frame's index in
// the launch.
__host__ __device__ __forceinline__ UnitGeo list_unit_geo(const FusedListParams &L, int unit, int grid)
{
    const int n = L.p.n_frames, b = unit % grid, j = unit / grid;
    const int lo = b * L.p.seg_rows, hi = min(L.fr[n].line0, lo + L.p.seg_rows);
    UnitGeo g{0, 0, 0, 0, false};
    if (lo >= hi) return g;
    int f = list_find(L, lo, false);
    const int col = L.fr[f].col0 + (lo - L.fr[f].line0) / L.fr[f].H + j;
    if (col >= L.fr[n].col0) return g;
    if (j > 0) f = list_find(L, col, true);
    const ListFrame &F = L.fr[f];
    g.f = f;
    g.strip = col - F.col0;
    const int c0 = F.line0 + g.strip * F.H;          // line position of the column's first row
    const int start = max(lo, c0), end = min(hi, c0 + F.H);
    g.y0 = start - c0;
    g.y1 = end - c0;
    g.ok = start < end;
    return g;
}

// What the kernel body calls: the unit's geometry, and H / W of the frame it belongs to.  The if constexpr keeps the frame
// table out of every other kernel's code, and H / W of those stay the values the body read from P once at its start
// (reading P.H again per unit, behind the loops' asm volatile memory clobbers, changes their instruction streams).
template <bool ROWS, bool LIST>
__device__ __forceinline__ UnitGeo unit_at(const FusedParams &P, int unit, int H, int grid)
{
    if constexpr (LIST) return list_unit_geo(list_of(P), unit, grid);
    else return unit_geo<ROWS>(P, unit, H, grid);
}
template <bool LIST> __device__ __forceinline__ int frame_h(const FusedParams &P, int f, int H)
{
    if constexpr (LIST) return list_of(P).fr[f].H;
    else return H;
}
template <bool LIST> __device__ __forceinline__ int frame_w(const FusedParams &P, int f, int W)
{
    if constexpr (LIST) return list_of(P).fr[f].W;
    else return W;
}

// workers / C4 warps -> MMA warp, event ev: every lane arrives on named barrier 2 + ev mod 3, the MMA warp blocks in
// bar.sync on the same id.  A warp blocked there issues nothing (a warp polling an mbarrier does, and on the MMA warp's SM
// sub-partition that is measurable: DESIGN.md section 7) and is released ~40 cycles after the last arrival.  Three ids are
// enough: a C4 warp arrives for event k after the named barrier that ended iteration k-2, which the workers reach only after
// the commit of iteration k-3, which the MMA warp issues after it has passed event k-3; the workers arrive later still.  So
// the arrivals for event k cannot begin before the MMA warp has left the barrier of event k-3, the previous user of that id.
__device__ __forceinline__ void work_arrive(uint32_t ev)
{
    asm volatile("bar.arrive %0, %1;" ::"r"(2u + ev % 3u), "n"(NWORKER + NC4 + 32) : "memory");
}

// ---- requantise 16 accumulator columns of this thread's pixel and store them as one 16-byte
// ---- channel group of an activation row (mat.cu:262-303 folded into the TMEM epilogue)
template <bool FAST, int BOFF>
__device__ __forceinline__ void requant(const uint32_t (&r)[16], const FusedParams &P, const GroupQ &g, bool valid,
                                        uint32_t (&o)[4])
{
    const unsigned Mz = valid ? g.M : 0u;           // FAST: an out-of-image pixel multiplies by 0
#pragma unroll
    for (int v = 0; v < 4; ++v) {
        // biases sit in the kernel-parameter constant bank at compile-time offsets: no smem traffic
        const int bb[4] = {P.bias[BOFF + 4 * v], P.bias[BOFF + 4 * v + 1], P.bias[BOFF + 4 * v + 2], P.bias[BOFF + 4 * v + 3]};
        uint32_t q[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (FAST) {
                // t = clamp(acc + b + rbias, 0, blu + rbias);  t * (mul << (24-shift)) < 2^31 and its top
                // byte is (t * mul) >> shift  -- see DESIGN.md "epilogue arithmetic"
                const unsigned t = (unsigned)__viaddmin_s32_relu((int)r[4 * v + j], bb[j], g.hi);
                q[j] = t * Mz;
            } else {
                QParam qp{g.blu, g.mul, g.shift, g.rbias};
                q[j] = valid ? ((unsigned)blu_requant((int)r[4 * v + j] + bb[j], qp) << 24) : 0u;
            }
        }
        // gather the four top bytes into one word
        o[v] = __byte_perm(__byte_perm(q[0], q[1], 0x0073), __byte_perm(q[2], q[3], 0x0073), 0x5410);
    }
}
template <bool FAST, int BOFF>
__device__ __forceinline__ void requant_store(const uint32_t (&r)[16], const FusedParams &P, const GroupQ &g, bool valid,
                                              uint8_t *dst)
{
    uint32_t o[4];
    requant<FAST, BOFF>(r, P, g, valid, o);
    *reinterpret_cast<uint4 *>(dst) = make_uint4(o[0], o[1], o[2], o[3]);
}
// C4 (48 -> 1, 3x3): the products of one a3 pixel (three 16-channel planes v[pl]) at horizontal tap DX with the three
// vertical taps, added to acc[dy]
template <int DX>
__device__ __forceinline__ void c4_taps(const uint4 (&v)[3], const FusedParams &P, int (&acc)[3])
{
#pragma unroll
    for (int dy = 0; dy < 3; ++dy)
#pragma unroll
        for (int pl = 0; pl < 3; ++pl) {
            const int *w = &P.c4_w[((dy * 3 + DX) * 3 + pl) * 4];
            acc[dy] = __dp4a((int)v[pl].x, w[0], acc[dy]);
            acc[dy] = __dp4a((int)v[pl].y, w[1], acc[dy]);
            acc[dy] = __dp4a((int)v[pl].z, w[2], acc[dy]);
            acc[dy] = __dp4a((int)v[pl].w, w[3], acc[dy]);
        }
}

// ROWS: the launch covers a row window of one frame (strips over several GPUs).  The whole-frame instantiation keeps
// the plain addressing: every instruction the C4 warps spend on the input ring is taken from the MMA warp's issue slots
// (same SM sub-partition), and the window arithmetic cost 2.5 % at 64 x 1080p (profiles/r2_kernel_ab_rowwindow.log).
// TMA: the input ring is filled by cp.async.bulk.tensor.2d (one elected thread, one 144-byte box per row, completion on an
// mbarrier) instead of per-thread byte loads and stores.  TMA pads out-of-image columns with 0 where the net needs 128 (0 in
// the x - 128 domain), so edge strips patch those bytes after the row has landed, and out-of-image rows are filled by hand.
template <bool FAST, bool PROF, bool ROWS, bool TMA = false>
__global__ void __launch_bounds__(NTHREADS, 1) k_fused(const __grid_constant__ FusedParams P)
{
    constexpr bool SSE = false, LIST = false;
#include "qv_fused_body.inc"
}

// The same network, and per frame the exact SSE of the anchor and of the reconstruction against the original (the integer
// core of vrcnn_data::psnr_pf, inference/yuv_data.cpp:98-112).  Its own name: the k_fused builds are counted and the hot one
// is found by its mangled name.  The body is k_fused's, included textually: moved into a __forceinline__ device function it
// compiled k_fused into a different instruction stream that measured 1.2 % slower at 64 x 1080p
// (profiles/frame_sse_kernel_ab_forceinline.log).
template <bool FAST, bool ROWS>
__global__ void __launch_bounds__(NTHREADS, 1) k_enh_sse(const __grid_constant__ FusedParams P)
{
    constexpr bool SSE = true, PROF = false, TMA = false, LIST = false;
#include "qv_fused_body.inc"
}

// Frames of different sizes in one launch (qv_forward_frame_list_device), with (SSE) or without the per-frame SSEs: every
// unit reads its frame's pointers and geometry from the frame table behind P.  Its own name, so that the k_fused /
// k_enh_sse builds stay what they are.
template <bool FAST, bool SSE>
__global__ void __launch_bounds__(NTHREADS, 1) k_enh_list(const __grid_constant__ FusedListParams PL)
{
    constexpr bool PROF = false, ROWS = false, TMA = false, LIST = true;
    const FusedParams &P = PL.p;
#include "qv_fused_body.inc"
}

// ---- strip protocol helper (stream-ordered): wait for words that ANOTHER GPU writes -----------------------------------------------------
__global__ void k_wait_words(const uint32_t *a, uint32_t va, const uint32_t *b, uint32_t vb, int *fail_flag)
{
    const uint32_t *w = threadIdx.x == 0 ? a : b;
    const uint32_t v = threadIdx.x == 0 ? va : vb;
    if (w && !peer_wait(w, v)) { *reinterpret_cast<volatile int *>(fail_flag) = 3; __threadfence_system(); }
}

// Shared-memory window base and TMEM base a CTA of k_fused sees (same launch shape: dynamic smem only, all 512 columns).
__global__ void k_bases(uint32_t *out)
{
    extern __shared__ __align__(1024) uint8_t sm[];
    uint32_t *slot = reinterpret_cast<uint32_t *>(sm);
    tmem_alloc(slot, TM_COLS);
    tmem_relinquish();
    fence_before_sync();
    __syncwarp();
    fence_after_sync();
    const uint32_t tm = *slot;
    if (threadIdx.x == 0) { out[0] = smem_u32(sm); out[1] = tm; }
    __syncwarp();
    tmem_dealloc(tm, TM_COLS);
}

// The operand bases of one iteration for every phase R1 mod 12, and the ones that never change.
void build_mma_bases(uint32_t sb, uint32_t tm, PhaseBases *pb, FixedBases &fb)
{
    constexpr uint32_t LP = (uint32_t)(PLANE >> 4) << 16;                  // LBO = one plane: K-halves are planes p, p+1
    const uint32_t w22 = sb + (OFF_W22 >> 4) + ((uint32_t)NR22 << 16), w21 = sb + (OFF_W21 >> 4) + ((uint32_t)NR21 << 16);
    const uint32_t w31 = sb + (OFF_W31 >> 4) + ((uint32_t)NR31 << 16);
    fb = FixedBases{};
    fb.zeroA = sb + (OFF_ZERO >> 4) + ((128u * 16 >> 4) << 16);
    fb.w1 = sb + (OFF_W1 >> 4) + (64u << 16);
    fb.w32 = sb + (OFF_W32 >> 4) + ((uint32_t)NR32 << 16);
    fb.r22 = tm + TM_R22; fb.r21 = tm + TM_R21; fb.r31 = tm + TM_R31;
    for (int ph = 0; ph < N_PHASE; ++ph) {
        const int R1p = ph + 4096 / N_PHASE * N_PHASE + N_PHASE, c3 = ph % 3, c6 = ph % 6;     // R1p = R1 (mod 12), large enough for R1p - k > 0
        const uint32_t par = ph & 1;
        const int qa = wrap_sub(c6, 2, 6);                                            // (R1-2) mod 6
        PhaseBases &e = pb[ph];
        e = PhaseBases{};
        e.im = sb + ((OFF_IM + c3 * IM_BYTES) >> 4) + ((128u * 16 >> 4) << 16);            // stage R1 mod 3
        e.a1_r2 = sb + (OFF_A1 >> 4) + wrap_sub(c3, 2, 3) * (A1_ROW >> 4) + LP;       // a1 row R1-2 (C2_2, C2_1)
        e.a2_r6 = sb + (OFF_A2 >> 4) + c3 * (A2_ROW >> 4);                            // a2 row R1-6 (C3_1, C3_2)
        e.b22 = w22 + (qa <= 2 ? 2 - qa : 8 - qa) * 16;                               // window start (8 - qa) mod 6 blocks of 16 rows
        e.b21 = w21 + ((1 - (R1p - 2)) & 3) * 32;                                     // (1 - (R1-2) mod 4) mod 4 blocks of 32 rows
        e.b31 = w31 + ((1 - (R1p - 6)) & 3) * 16;
        e.d1 = tm + TM_D1 + par * 64; e.d32 = tm + TM_D32 + par * 32;
        e.z22 = tm + TM_R22 + c6 * 16;                                                // C2_2 row R1   starts: zero its slot
        e.z21 = tm + TM_R21 + ((R1p - 1) & 3) * 32;                                   // C2_1 row R1-1 starts
        e.z31 = tm + TM_R31 + ((R1p - 5) & 3) * 16;                                   // C3_1 row R1-5 starts
    }
}

// The per-MMA expansion of the two tables above, in the kernel's issue order.
void build_mma_ops(const PhaseBases *pb, const FixedBases &fb, PhaseOps *ops)
{
    constexpr uint32_t HI = (128u >> 4) | (1u << 14);                       // SBO = 128 B, descriptor version 1
    constexpr uint32_t LP = (uint32_t)(PLANE >> 4) << 16, LX = 1u << 16;
    for (int ph = 0; ph < N_PHASE; ++ph) {
        const PhaseBases &e = pb[ph];
        PhaseOps &o = ops[ph];
        o = PhaseOps{};
        int k = 0;
        auto put = [&](uint32_t a, uint32_t b) { o.ab[k++] = make_uint4(a, HI, b, HI); };
        put(e.im, fb.w1);
        put(fb.zeroA, fb.w1); put(fb.zeroA, fb.w1); put(fb.zeroA, fb.w1);
        put(e.a2_r6 + 6 + LP, e.b31);
        put(e.a2_r6 + 7 + LP, e.b31 + (T31 >> 4));
        put(e.a2_r6 + 7 + LP, fb.w32);
        put(e.a2_r6 + 8 + LP, e.b31 + 2 * (T31 >> 4));
        put(e.a2_r6 + ((2 * PLANE) >> 4) + 6 + LX, e.b31 + 3 * (T31 >> 4));
        put(e.a2_r6 + ((2 * PLANE) >> 4) + 6 + LX, fb.w32 + (T32 >> 4));
        put(e.a2_r6 + ((2 * PLANE) >> 4) + 8 + LX, e.b31 + 4 * (T31 >> 4));
        for (int t = 0; t < 10; ++t) {
            const int sft = t / 2, h = t & 1;
            const uint32_t a = e.a1_r2 + ((h * 2 * PLANE + (4 + sft) * 16) >> 4);
            put(a, e.b22 + t * (T22 >> 4));
            if (sft >= 1 && sft <= 3) put(a, e.b21 + ((sft - 1) * 2 + h) * (T21 >> 4));
        }
        o.d1 = e.d1; o.d32 = e.d32; o.z22 = e.z22; o.z21 = e.z21; o.z31 = e.z31;
    }
}

}  // namespace

// =================================== host side ==========================================
struct FusedModel {
    int *h_fail = nullptr;             // cudaHostAlloc'ed, mapped: kernel failure report
    uint8_t *d_wimg = nullptr;
    FusedParams proto{};               // the model's constants; every per-launch field stays zero (launch_params)
    bool fast = true;
    int sm_count = 148;
    // environment switches, read once at upload (never on the per-launch path)
    bool env_profile = false, env_test_fail = false, env_tma = false;
    int env_experiment = 0;
    void *encode_tiled = nullptr;      // cuTensorMapEncodeTiled (driver entry point; the library does not link libcuda)
};

// Every kernel build the host launches, with the dynamic shared memory it runs with: fused_upload raises each one's limit,
// build_of picks the one a launch runs.  The first twelve come in pairs, generic requantiser first, so that entry + fast
// is the build for a model.
struct KernelBuild { const void *fn; int smem; };
const KernelBuild k_builds[] = {
    {(const void *)k_fused<false, false, false>, SMEM_BYTES}, {(const void *)k_fused<true, false, false>, SMEM_BYTES},
    {(const void *)k_fused<false, false, true>, SMEM_BYTES},  {(const void *)k_fused<true, false, true>, SMEM_BYTES},
    {(const void *)k_enh_sse<false, false>, SMEM_BYTES},      {(const void *)k_enh_sse<true, false>, SMEM_BYTES},
    {(const void *)k_enh_sse<false, true>, SMEM_BYTES},       {(const void *)k_enh_sse<true, true>, SMEM_BYTES},
    {(const void *)k_enh_list<false, false>, SMEM_BYTES},     {(const void *)k_enh_list<true, false>, SMEM_BYTES},
    {(const void *)k_enh_list<false, true>, SMEM_BYTES},      {(const void *)k_enh_list<true, true>, SMEM_BYTES},
    {(const void *)k_fused<true, true, false>, SMEM_BYTES},
    {(const void *)k_fused<true, false, false, true>, SMEM_BYTES_T},
    {(const void *)k_bases, SMEM_BYTES},
};
enum { B_WHOLE = 0, B_ROWS = 2, B_SSE = 4, B_SSE_ROWS = 6, B_LIST = 8, B_LIST_SSE = 10, B_PROFILE = 12, B_TMA = 13, B_BASES = 14 };
static_assert(sizeof(k_builds) / sizeof(k_builds[0]) == B_BASES + 1, "one entry per build");

// The build a launch runs: a frame list, the SSE form and a row window have their own; whole frames of a fast model run the
// profiling build with QV_FUSED_PROFILE, else the TMA input ring with `tma` (QV_FUSED_TMA and an input a tensor map can
// describe), else the plain kernel.
static int build_of(bool fast, bool list, bool sse, bool rows, bool profile, bool tma)
{
    if (list) return (sse ? B_LIST_SSE : B_LIST) + fast;
    if (sse) return (rows ? B_SSE_ROWS : B_SSE) + fast;
    if (rows) return B_ROWS + fast;
    if (fast && profile) return B_PROFILE;
    if (fast && tma) return B_TMA;
    return B_WHOLE + fast;
}

// One launch of build b (not k_bases) on `grid` CTAs; params points at its FusedParams (FusedListParams for a frame list).
static int launch(int b, int grid, void *params, cudaStream_t st, long long *launches)
{
    if (launches) *launches += 1;
    QV_CUDA(cudaLaunchKernel(k_builds[b].fn, grid, NTHREADS, &params, k_builds[b].smem, st));   // &params: the one argument
    return QV_OK;
}

// The parameters every launch starts from: the model's constants, with QV_FUSED_TEST_FAIL applied.
static FusedParams launch_params(const FusedModel *fm)
{
    FusedParams P = fm->proto;
    if (fm->env_test_fail) P.sbase16 ^= 1u;
    return P;
}

// The operand table lives in constant memory: one copy per device, and its content depends only on the shared-memory
// window / TMEM bases a CTA of this launch shape gets -- the same for every model.  It is written once per device, under
// a lock, so that distinct handles can load models from distinct threads (include/qvrcnn_b200.h).
struct OpsBases { uint32_t sbase16, tmem_base; };
static std::mutex g_ops_mu;
static std::map<int, OpsBases> g_ops;   // device -> the bases its table was built for

// Writes 16 K-bytes of row n, K-chunk j, of a B block laid out [2][NR][16].
static void put_chunk(uint8_t *blk, int NR, int j, int n, const int8_t *src16) { memcpy(blk + ((size_t)j * NR + n) * 16, src16, 16); }

// Everything of the model that is built on the host: the weight image (the B operands in their ring block sequences, the
// biases) and the kernel-parameter constants (requantiser rows, C4 weights).  Returns whether the fast requantiser applies.
static bool build_host_image(const ModelHost &m, std::vector<uint8_t> &img, FusedParams &P)
{
    img.assign(WIMG_BYTES, 0);
    auto Wt = [&](int l, int k, int c, int r, int s) -> int8_t {
        const LayerShape &sh = kLayers[l];
        return m.L[l].w[(((size_t)k * sh.cin + c) * sh.k + r) * sh.k + s];
    };
    // ---- W1: B[n][k], k = 4r+s (s<4) | 20+r (s=4) | zero --------------------------------------
    for (int n = 0; n < 64; ++n) {
        int8_t k32[32] = {0};
        for (int r = 0; r < 5; ++r) {
            for (int s = 0; s < 4; ++s) k32[4 * r + s] = Wt(QV_C1, n, 0, r, s);
            k32[20 + r] = Wt(QV_C1, n, 0, r, 4);
        }
        put_chunk(img.data() + OFF_W1, 64, 0, n, k32);
        put_chunk(img.data() + OFF_W1, 64, 1, n, k32 + 16);
    }
    // Ring block sequences: vertical tap r per block (-1 = zero block); a window of R consecutive blocks,
    // starting at the offset the kernel computes from (row mod R), lines the taps up with the ring slots.
    const int S22[11] = {4, 3, 2, 1, 0, -1, 4, 3, 2, 1, 0};
    const int S3[7] = {2, 1, 0, -1, 2, 1, 0};
    int8_t c16[16];
    // ---- W22: tile (s, h): rows blk*16 + ch ; channels 32h + 16j + b ------------------------------
    for (int s = 0; s < 5; ++s)
        for (int h = 0; h < 2; ++h) {
            uint8_t *blk = img.data() + OFF_W22 + (s * 2 + h) * T22;
            for (int bi = 0; bi < 11; ++bi)
                if (S22[bi] >= 0)
                    for (int j = 0; j < 2; ++j)
                        for (int ch = 0; ch < 16; ++ch) {
                            for (int b = 0; b < 16; ++b) c16[b] = Wt(QV_C2_2, ch, 32 * h + 16 * j + b, S22[bi], s);
                            put_chunk(blk, NR22, j, bi * 16 + ch, c16);
                        }
        }
    // ---- W21: tile (s', h): rows blk*32 + ch --------------------------------------------------------
    for (int s = 0; s < 3; ++s)
        for (int h = 0; h < 2; ++h) {
            uint8_t *blk = img.data() + OFF_W21 + (s * 2 + h) * T21;
            for (int bi = 0; bi < 7; ++bi)
                if (S3[bi] >= 0)
                    for (int j = 0; j < 2; ++j)
                        for (int ch = 0; ch < 32; ++ch) {
                            for (int b = 0; b < 16; ++b) c16[b] = Wt(QV_C2_1, ch, 32 * h + 16 * j + b, S3[bi], s);
                            put_chunk(blk, NR21, j, bi * 32 + ch, c16);
                        }
        }
    // ---- K-step -> (s, plane) units of a 48-channel activation row -----------------------------------
    //   k = 0,1,2: (s=k, plane 0) | (s=k, plane 1) ;  k = 3: (s=0, plane 2) | (s=1, plane 2) ;  k = 4: (s=2, plane 2) | zero
    auto unit = [](int k, int j, int &s, int &pl) -> bool {
        if (k < 3) { s = k; pl = j; return true; }
        if (k == 3) { s = j; pl = 2; return true; }
        s = 2; pl = 2;
        return j == 0;
    };
    // ---- W31 (rows blk*16 + ch) ----------------------------------------------------------------------
    for (int k = 0; k < 5; ++k)
        for (int bi = 0; bi < 7; ++bi)
            if (S3[bi] >= 0)
                for (int j = 0; j < 2; ++j) {
                    int s, pl;
                    if (!unit(k, j, s, pl)) continue;
                    for (int ch = 0; ch < 16; ++ch) {
                        for (int b = 0; b < 16; ++b) c16[b] = Wt(QV_C3_1, ch, 16 * pl + b, S3[bi], s);
                        put_chunk(img.data() + OFF_W31 + k * T31, NR31, j, bi * 16 + ch, c16);
                    }
                }
    // ---- W32 (1x1): K-step 0 = planes 0,1 of the centre pixel (the tile of C3_1's K-step 1) ; K-step 1 = zero | plane 2
    //      (the tile of C3_1's K-step 3: plane 2 of the pixel to the left | plane 2 of the centre pixel) ------------------
    for (int ch = 0; ch < 32; ++ch)
        for (int pl = 0; pl < 3; ++pl) {
            for (int b = 0; b < 16; ++b) c16[b] = Wt(QV_C3_2, ch, 16 * pl + b, 0, 0);
            put_chunk(img.data() + OFF_W32 + (pl / 2) * T32, NR32, pl == 2 ? 1 : pl, ch, c16);
        }
    // ---- requantiser constants ---------------------------------------------------------------------
    auto mkq = [&](int l, GroupQ &g) -> bool {
        const LayerHost &L = m.L[l];
        g.blu = L.blu; g.mul = L.mul; g.shift = L.shift; g.rbias = (1 << (L.shift - 1)) / L.mul;
        g.hi = L.blu + g.rbias;
        const long long top = ((long long)L.blu + g.rbias) * L.mul;
        const bool ok = L.shift <= 24 && L.mul < (1ll << L.shift) && top < (1ll << 31) && (top >> L.shift) == 127 && g.hi < (1 << 30);
        g.M = ok ? (unsigned)((unsigned long long)L.mul << (24 - L.shift)) : 0u;
        return ok;
    };
    bool fast = true;
    fast &= mkq(QV_C1, P.q1); fast &= mkq(QV_C2_2, P.q22); fast &= mkq(QV_C2_1, P.q21);
    fast &= mkq(QV_C3_1, P.q31); fast &= mkq(QV_C3_2, P.q32);
    int *bias = reinterpret_cast<int *>(img.data() + OFF_BIAS);
    auto addb = [&](int l, int dst0, const GroupQ &g) {
        for (int k = 0; k < kLayers[l].cout; ++k) bias[dst0 + k] = m.L[l].b[k] + (fast ? g.rbias : 0);
    };
    addb(QV_C1, 0, P.q1);
    addb(QV_C2_2, 64, P.q22); addb(QV_C2_1, 64 + 16, P.q21);
    addb(QV_C3_1, 112, P.q31); addb(QV_C3_2, 112 + 16, P.q32);
    memcpy(P.bias, bias, sizeof(P.bias));
    P.c4_bias = m.L[QV_C4].b[0]; P.c4_mul = m.L[QV_C4].mul; P.c4_shift = m.L[QV_C4].shift;
    for (int t = 0; t < 9; ++t)
        for (int pl = 0; pl < 3; ++pl)
            for (int j = 0; j < 4; ++j) {
                unsigned v = 0;
                for (int b = 0; b < 4; ++b) v |= (unsigned)(uint8_t)Wt(QV_C4, 0, 16 * pl + 4 * j + b, t / 3, t % 3) << (8 * b);
                P.c4_w[(t * 3 + pl) * 4 + j] = (int)v;
            }
    return fast;
}

// Test hook, no GPU involved: the structures the host builds for the kernel -- weight image, the per-phase MMA operand
// table (for shared-memory window base 0 and TMEM base 0) and the constants -- so that a CPU emulation of the kernel's
// dataflow can be checked against the oracle (tests/test_fused_tables.py).
void fused_debug_tables(const ModelHost &m, std::vector<uint8_t> &wimg, std::vector<uint32_t> &ops, std::vector<int32_t> &consts)
{
    FusedParams P{};
    const bool fast = build_host_image(m, wimg, P);
    PhaseBases pb[N_PHASE];
    FixedBases fb;
    build_mma_bases(0, 0, pb, fb);
    std::vector<PhaseOps> po(N_PHASE);
    build_mma_ops(pb, fb, po.data());
    ops.assign(reinterpret_cast<const uint32_t *>(po.data()), reinterpret_cast<const uint32_t *>(po.data() + N_PHASE));
    consts = {WIMG_BYTES, SMEM_BYTES, OFF_A1, OFF_A2, OFF_IM, OFF_ZERO, OFF_IN, OFF_A3, PW, PLANE, A1_ROW, A2_ROW, IM_BYTES, IN_SLOTS,
              IN_PITCH, WT, PIPE, TM_D1, TM_R22, TM_R21, TM_R31, TM_D32, N_PHASE, N_MMA, fast ? 1 : 0, P.c4_bias, P.c4_mul, P.c4_shift};
    for (const GroupQ *g : {&P.q1, &P.q22, &P.q21, &P.q31, &P.q32})
        for (int v : {g->hi, (int)g->M, g->blu, g->mul, g->shift, g->rbias}) consts.push_back(v);
    consts.insert(consts.end(), P.bias, P.bias + BIAS_INTS);
    consts.insert(consts.end(), P.c4_w, P.c4_w + 108);
}

// Writes the operand table of device dev (the current one) on its first model; P takes the bases it was built for.  Under g_ops_mu.
static int operand_table(int dev, cudaStream_t st, FusedParams &P)
{
    auto it = g_ops.find(dev);
    if (it == g_ops.end()) {
        uint32_t *d_b = nullptr, h_b[2] = {0, 0};
        QV_CUDA(cudaMalloc(&d_b, 8));
        k_bases<<<1, 32, k_builds[B_BASES].smem, st>>>(d_b);
        cudaError_t e = cudaMemcpyAsync(h_b, d_b, 8, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        cudaFree(d_b);
        QV_CUDA(e);
        PhaseBases pb[N_PHASE];
        FixedBases fb;
        build_mma_bases(h_b[0] >> 4, h_b[1], pb, fb);
        std::vector<PhaseOps> ops(N_PHASE);      // outlives the copy: synchronised below
        build_mma_ops(pb, fb, ops.data());
        QV_CUDA(cudaMemcpyToSymbolAsync(c_ops, ops.data(), sizeof(PhaseOps) * N_PHASE, 0, cudaMemcpyHostToDevice, st));
        QV_CUDA(cudaStreamSynchronize(st));
        it = g_ops.emplace(dev, OpsBases{h_b[0] >> 4, h_b[1]}).first;
    }
    P.sbase16 = it->second.sbase16; P.tmem_base = it->second.tmem_base;
    return QV_OK;
}

int fused_upload(const ModelHost &m, cudaStream_t st, FusedModel **out)
{
    std::unique_ptr<FusedModel, void (*)(FusedModel *)> fm(new FusedModel(), fused_free);   // freed on every failure
    FusedParams &P = fm->proto;
    std::vector<uint8_t> img;
    fm->fast = build_host_image(m, img, P);
    QV_CUDA(cudaMalloc(&fm->d_wimg, WIMG_BYTES));
    QV_CUDA(cudaMemcpyAsync(fm->d_wimg, img.data(), WIMG_BYTES, cudaMemcpyHostToDevice, st));
    QV_CUDA(cudaStreamSynchronize(st));
    for (const KernelBuild &k : k_builds) QV_CUDA(cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, k.smem));
    int dev = 0;
    QV_CUDA(cudaGetDevice(&dev));
    {
        std::lock_guard<std::mutex> lock(g_ops_mu);
        if (int rc = operand_table(dev, st, P)) return rc;
    }
    QV_CUDA(cudaDeviceGetAttribute(&fm->sm_count, cudaDevAttrMultiProcessorCount, dev));
    fm->env_profile = getenv("QV_FUSED_PROFILE") != nullptr;
    fm->env_experiment = getenv("QV_FUSED_EXPERIMENT") ? atoi(getenv("QV_FUSED_EXPERIMENT")) : 0;
    fm->env_test_fail = getenv("QV_FUSED_TEST_FAIL") != nullptr;     // tests only: make every CTA report a base mismatch
    fm->env_tma = getenv("QV_FUSED_TMA") != nullptr && atoi(getenv("QV_FUSED_TMA")) != 0;
    if (fm->env_tma) {
        cudaDriverEntryPointQueryResult qr;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fm->encode_tiled, cudaEnableDefault, &qr) != cudaSuccess || qr != cudaDriverEntryPointSuccess)
            fm->encode_tiled = nullptr;
        cudaGetLastError();
    }
    P.wimg = fm->d_wimg;
    QV_CUDA(cudaHostAlloc(&fm->h_fail, sizeof(int), cudaHostAllocMapped));
    *fm->h_fail = 0;
    QV_CUDA(cudaHostGetDevicePointer(&P.fail_flag, fm->h_fail, 0));
    *out = fm.release();
    return QV_OK;
}

cudaError_t fused_wait_words(const FusedModel *fm, const uint32_t *a, uint32_t va, const uint32_t *b, uint32_t vb, cudaStream_t st)
{
    if (!a && !b) return cudaSuccess;
    k_wait_words<<<1, 2, 0, st>>>(a, va, b, vb, fm->proto.fail_flag);
    return cudaGetLastError();
}

void fused_free(FusedModel *fm)
{
    if (!fm) return;
    if (fm->h_fail) cudaFreeHost(fm->h_fail);
    cudaFree(fm->d_wimg);
    delete fm;
}

int fused_take_failure(const FusedModel *fm)
{
    if (!fm) return 0;
    const int f = *reinterpret_cast<volatile int *>(fm->h_fail);
    if (f) *fm->h_fail = 0;
    return f;
}

// How a launch is dealt out to the persistent CTAs: fills the geometry fields of P (nstrips, nseg, seg_rows, n_units, linear,
// perm_*) from n_frames, W and the output rows [ys, ye), and returns the grid.  Host-only arithmetic; unit_geo() is its reader.
static cudaError_t plan_units(FusedParams &P, int sm_count, bool allow_linear, bool rows_mode, int &grid)
{
    const int rows_out = P.ye - P.ys;
    P.nstrips = (P.W + WT - 1) / WT;
    grid = 1;
    P.linear = 0;
    if (rows_mode) {
        // one line of nstrips * rows_out row-iterations, cut into equal chunks (rows_unit): every SM gets the same number
        // of rows; a chunk pays the PIPE iterations of pipeline fill once per strip column it touches (never below 32 rows
        // per CTA)
        const long long total = (long long)P.nstrips * rows_out;
        if (total > 0x3fffffffll) return cudaErrorInvalidValue;
        grid = (int)std::max<long long>(1, std::min<long long>(sm_count, total / 32));
        P.seg_rows = (int)((total + grid - 1) / grid);                 // the chunk
        grid = (int)((total + P.seg_rows - 1) / P.seg_rows);
        const int pieces = (P.seg_rows + rows_out - 1) / rows_out + 1;  // strip columns a chunk can touch
        P.nseg = 1;
        P.n_units = grid * pieces;
    } else {
        // Row segments.  Units are dealt to the persistent CTAs round-robin, so the makespan is
        // ceil(units / SMs) * (rows per segment + PIPE) row-iterations; pick the cut that minimises it
        // (never below 16 rows per segment: every segment pays PIPE iterations of pipeline fill).
        const long long cols = (long long)P.n_frames * P.nstrips;
        int nseg = 1;
        {
            long long best = -1;
            const int max_seg = std::max(1, std::min(rows_out / 16, 256));
            for (int c = 1; c <= max_seg; ++c) {
                const int rws = (rows_out + c - 1) / c, real = (rows_out + rws - 1) / rws;
                const long long waves = (cols * real + sm_count - 1) / sm_count;
                const long long cost = waves * (rws + PIPE);
                if (best < 0 || cost < best) { best = cost; nseg = c; }
            }
        }
        P.seg_rows = (rows_out + nseg - 1) / nseg;
        P.nseg = (rows_out + P.seg_rows - 1) / P.seg_rows;
        const long long units = cols * P.nseg;
        if (units > 0x7fffffffll) return cudaErrorInvalidValue;
        P.n_units = (int)units;
        grid = (int)std::min<long long>(units, sm_count);
        // ... or the line of cols * H row-iterations cut into one equal chunk per SM (see unit_geo): no idle SMs in the last
        // wave, one pipeline fill per strip column a chunk touches.  64 x 1080p: 7585 iterations per SM against 7658.
        const long long total = cols * rows_out, g2 = std::max<long long>(1, std::min<long long>(sm_count, total / 32));
        const long long chunk = (total + g2 - 1) / g2, pieces = (chunk + rows_out - 1) / rows_out + 1;
        const long long cost_equal = (units + grid - 1) / grid * (P.seg_rows + PIPE);
        if (allow_linear && total <= 0x3fffffffll && chunk + pieces * PIPE < cost_equal) {
            P.linear = 1;
            P.seg_rows = (int)chunk;
            grid = (int)((total + chunk - 1) / chunk);
            P.nseg = 1;
            P.n_units = grid * (int)pieces;
            const long long per = (cols + grid - 1) / grid;               // columns per chunk, rounded up
            P.perm_q = (int)((cols + per - 1) / per);
            P.perm_s0 = (int)(cols / P.perm_q);
            P.perm_r = (int)(cols % P.perm_q);
        }
    }
    return cudaSuccess;
}

// Test hook (qv_debug_fused_units): the units of a launch as the kernel's CTAs will see them, 5 ints each (cta, frame, strip column, y0, y1)
int fused_debug_units(int sm_count, int n_frames, int H, int W, int row0, int row1, bool rows_mode, bool allow_linear, std::vector<int> &units, int &grid)
{
    FusedParams P{};
    P.n_frames = n_frames; P.H = H; P.W = W; P.ys = row0; P.ye = row1;
    if (sm_count < 1 || n_frames < 1 || W < 1 || row0 < 0 || row1 > H || row0 >= row1 || (rows_mode && n_frames != 1)) return -1;
    if (plan_units(P, sm_count, allow_linear, rows_mode, grid) != cudaSuccess) return -1;
    units.clear();
    for (int u = 0; u < P.n_units; ++u) {
        const UnitGeo g = rows_mode ? unit_geo<true>(P, u, H, grid) : unit_geo<false>(P, u, H, grid);
        if (!g.ok) continue;
        const int v[5] = {u % grid, g.f, g.strip, g.y0, g.y1};
        units.insert(units.end(), v, v + 5);
    }
    return 0;
}

// The plan of one frame-list launch: fills the frame table and the geometry fields of L.p that list_unit_geo reads and returns
// the grid.  The row line over all (frame, strip column) columns is cut into one equal chunk per SM, as plan_units' line;
// a chunk pays PIPE iterations of pipeline fill per column it touches.
static cudaError_t plan_list(FusedListParams &L, const qv_frame_desc *frames, int n, int sm_count, int &grid)
{
    if (n < 1 || n > QV_FRAME_LIST_LAUNCH_MAX || sm_count < 1) return cudaErrorInvalidValue;
    long long line = 0, cols = 0;
    for (int f = 0; f < n; ++f) {
        const qv_frame_desc &fr = frames[f];
        if (fr.height < 1 || fr.width < 1) return cudaErrorInvalidValue;
        L.fr[f] = ListFrame{fr.d_in, fr.d_out, fr.d_ori, fr.height, fr.width, (int)line, (int)cols};
        const long long nstrips = (fr.width + WT - 1) / WT;
        line += nstrips * fr.height;
        cols += nstrips;
        if (line > 0x3fffffffll) return cudaErrorInvalidValue;
    }
    L.fr[n] = ListFrame{nullptr, nullptr, nullptr, 0, 0, (int)line, (int)cols};
    FusedParams &P = L.p;
    P.n_frames = n;
    grid = (int)std::max<long long>(1, std::min<long long>(sm_count, line / 32));
    const int chunk = (int)((line + grid - 1) / grid);
    grid = (int)((line + chunk - 1) / chunk);
    // units per CTA: the columns its chunk touches, at most
    int pieces = 1;
    for (int b = 0; b < grid; ++b) {
        const int lo = b * chunk, last = (int)std::min<long long>(line, (long long)lo + chunk) - 1;
        auto col_at = [&](int v) { const int f = list_find(L, v, false); return L.fr[f].col0 + (v - L.fr[f].line0) / L.fr[f].H; };
        pieces = std::max(pieces, col_at(last) - col_at(lo) + 1);
    }
    if ((long long)grid * pieces > 0x7fffffffll) return cudaErrorInvalidValue;
    P.seg_rows = chunk;
    P.n_units = grid * pieces;
    P.nseg = 1;
    P.linear = 1;
    return cudaSuccess;
}

int fused_debug_list_units(int sm_count, int n_frames, const int *H, const int *W, std::vector<int> &units, int &grid)
{
    if (n_frames < 1 || n_frames > QV_FRAME_LIST_LAUNCH_MAX) return -1;
    std::vector<qv_frame_desc> fr(n_frames);
    for (int f = 0; f < n_frames; ++f) fr[f] = qv_frame_desc{nullptr, nullptr, nullptr, H[f], W[f]};
    std::unique_ptr<FusedListParams> L(new FusedListParams{});
    if (plan_list(*L, fr.data(), n_frames, sm_count, grid) != cudaSuccess) return -1;
    units.clear();
    for (int u = 0; u < L->p.n_units; ++u) {
        const UnitGeo g = list_unit_geo(*L, u, grid);
        if (!g.ok) continue;
        const int v[5] = {u % grid, g.f, g.strip, g.y0, g.y1};
        units.insert(units.end(), v, v + 5);
    }
    return 0;
}

int fused_forward_list(const FusedModel *fm, const qv_frame_desc *frames, int n, int64_t *d_sse, cudaStream_t st, long long *launches)
{
    for (int f = 0; f < n; ++f) {
        if (!frames[f].d_ori != !d_sse) { set_error("fused_forward_list: frame %d: d_ori and d_sse go together", f); return QV_ERR_ARG; }
        if (d_sse && frames[f].height > FUSED_SSE_MAX_H) {      // the C4 threads' 32-bit column sums
            set_error("fused_forward_list: per-frame SSE: frame %d height %d exceeds %d", f, frames[f].height, FUSED_SSE_MAX_H);
            return QV_ERR_ARG;
        }
    }
    std::unique_ptr<FusedListParams> L(new FusedListParams{});      // 12 KB: not on the stack
    int grid = 1;
    auto plan = [&](int f0) {
        L->p = launch_params(fm);
        return plan_list(*L, frames + f0, std::min(QV_FRAME_LIST_LAUNCH_MAX, n - f0), fm->sm_count, grid) == cudaSuccess;
    };
    for (int f0 = 0; f0 < n; f0 += QV_FRAME_LIST_LAUNCH_MAX)        // every launch's plan, before the first launch
        if (!plan(f0)) {
            set_error("fused_forward_list: the frames of one launch exceed 2^30 strip-column rows");
            return QV_ERR_ARG;
        }
    for (int f0 = 0; f0 < n; f0 += QV_FRAME_LIST_LAUNCH_MAX) {
        plan(f0);
        L->p.sse = d_sse ? reinterpret_cast<unsigned long long *>(d_sse + 2 * (size_t)f0) : nullptr;
        if (int rc = launch(build_of(fm->fast, true, d_sse != nullptr, false, false, false), grid, L.get(), st, launches)) return rc;
    }
    return QV_OK;
}

// The profiling build (QV_FUSED_PROFILE=1): one launch with per-block phase timers; once it has finished, their averages
// and the timeline of block 0 go to stderr.
static int launch_profiled(const FusedModel *fm, FusedParams &P, int grid, cudaStream_t st, long long *launches)
{
    std::vector<long long> h((size_t)grid * 16 + TR_N * 48);
    const size_t bytes = h.size() * sizeof(long long);
    QV_CUDA(cudaMalloc(&P.dbg, bytes));
    const std::unique_ptr<long long, cudaError_t (*)(void *)> hold(P.dbg, cudaFree);
    P.dbg_flags = fm->env_experiment;
    QV_CUDA(cudaMemsetAsync(P.dbg, 0, bytes, st));
    if (int rc = launch(B_PROFILE, grid, &P, st, launches)) return rc;
    QV_CUDA(cudaStreamSynchronize(st));
    QV_CUDA(cudaMemcpy(h.data(), P.dbg, bytes, cudaMemcpyDeviceToHost));
    double a[16] = {0};
    for (int b = 0; b < grid; ++b) for (int k = 0; k < 16; ++k) a[k] += (double)h[(size_t)b * 16 + k] / grid;
    const double iters = P.linear ? (double)P.seg_rows + PIPE * (P.n_units / grid - 1) : (double)P.n_units / grid * (P.seg_rows + PIPE);
    fprintf(stderr, "[qv fused profile] units=%d grid=%d iters/block~%.0f | cycles per iteration: MMA warp wait=%.0f issue=%.0f | "
            "worker w0: wait_mma=%.0f drain=%.0f (of which tcgen05.ld+wait %.0f) fence+arrive=%.0f bar=%.0f | "
            "second traced worker (thread NWORKER/2): wait_mma=%.0f drain=%.0f (tcgen05.ld+wait %.0f) fence+arrive=%.0f bar=%.0f\n",
            P.n_units, grid, iters, a[0] / iters, a[1] / iters, a[2] / iters, a[3] / iters, a[14] / iters, a[4] / iters, a[5] / iters,
            a[8] / iters, a[9] / iters, a[15] / iters, a[10] / iters, a[11] / iters);
    // timeline of block 0: per traced iteration, cycles relative to the first issue start
    const long long *tr = h.data() + (size_t)grid * 16, t0 = tr[0];
    if (t0)
        for (int k = 0; k < TR_N; ++k, tr += 16)
            fprintf(stderr, "[qv fused trace] it %d | mma: start %lld end %lld | w0: commit %lld drained %lld arrived %lld bar %lld | "
                    "w2: commit %lld drained %lld arrived %lld bar %lld\n", TR_ITER0 + k, tr[0] - t0, tr[1] - t0, tr[2] - t0, tr[3] - t0,
                    tr[4] - t0, tr[5] - t0, tr[6] - t0, tr[7] - t0, tr[8] - t0, tr[9] - t0);
    tr = h.data() + (size_t)grid * 16;
    if (t0)
        for (int k = 0; k < TR_N; ++k, tr += 16)
            fprintf(stderr, "[qv fused mma-side] it %d | loop top %lld  wait done %lld  fence done %lld  (issue start %lld)  commit issued %lld  end %lld\n",
                    TR_ITER0 + k, tr[10] - t0, tr[11] - t0, tr[12] - t0, tr[0] - t0, tr[13] - t0, tr[1] - t0);
    if (t0)
        for (int k = 0; k < TR_N; ++k) {
            const long long *sp = h.data() + (size_t)grid * 16 + TR_N * 16 + k * 32, s0 = h[(size_t)grid * 16 + k * 16];
            fprintf(stderr, "[qv fused stamps] it %d:", TR_ITER0 + k);
            for (int j = 0; j < 27; ++j) fprintf(stderr, " %lld", sp[j] - (j ? sp[j - 1] : s0));
            fprintf(stderr, "\n");
        }
    return QV_OK;
}

int fused_forward(const FusedModel *fm, const uint8_t *d_in, uint8_t *d_out, int n, int H, int W, cudaStream_t st,
                  long long *launches, const FusedRows *rows, const uint8_t *d_ori, int64_t *d_sse)
{
    if (n <= 0) return QV_OK;
    const bool sse = d_ori && d_sse;
    if ((d_ori || d_sse) && !sse) { set_error("fused_forward: d_ori and d_sse go together"); return QV_ERR_ARG; }
    if (sse && H > FUSED_SSE_MAX_H) {      // the C4 threads' 32-bit column sums
        set_error("fused_forward: per-frame SSE: frame height %d exceeds %d", H, FUSED_SSE_MAX_H);
        return QV_ERR_ARG;
    }
    FusedParams P = launch_params(fm);
    P.ori = d_ori;
    P.sse = reinterpret_cast<unsigned long long *>(d_sse);
    P.n_frames = n; P.H = H; P.W = W;
    P.frame_stride = (size_t)H * W;
    P.in = d_in; P.out = d_out;
    P.ye = P.own1 = P.rhi = H;
    if (rows) {
        // one frame, a row window of it: H is the height of the IMAGE (each layer's zero padding applies at the image
        // edges only, inference/cnn.cu:44-49), the buffers hold the rows the launch description names
        const char *bad = "fused_forward: inconsistent row window";
        if (n != 1 || rows->own0 < 0 || rows->own1 > H || rows->own0 >= rows->own1 || rows->out0 < rows->own0 || rows->out1 > rows->own1 ||
            rows->out0 > rows->out1 || rows->top_rows < 0 || rows->bot_rows < 0) { set_error("%s", bad); return QV_ERR_ARG; }
        if (rows->out0 == rows->out1) return QV_OK;
        P.own0 = rows->own0; P.own1 = rows->own1; P.ys = rows->out0; P.ye = rows->out1;
        P.rlo = rows->d_top ? rows->own0 - rows->top_rows : rows->own0;
        P.rhi = rows->d_bot ? rows->own1 + rows->bot_rows : rows->own1;
        if (P.rlo < 0 || P.rhi > H) { set_error("%s", bad); return QV_ERR_ARG; }
        P.in = d_in - (ptrdiff_t)rows->own0 * W;
        P.out = d_out - (ptrdiff_t)rows->out0 * W;
        if (sse) P.ori = d_ori - (ptrdiff_t)rows->out0 * W;
        P.in_top = rows->d_top ? rows->d_top - (ptrdiff_t)P.rlo * W : nullptr;
        P.in_bot = rows->d_bot ? rows->d_bot - (ptrdiff_t)rows->own1 * W : nullptr;
        P.flag_top = rows->d_top ? rows->flag_top : nullptr;
        P.flag_bot = rows->d_bot ? rows->flag_bot : nullptr;
        P.pub = rows->pub; P.done = rows->done; P.done_ctr = rows->done_ctr; P.seq = rows->seq;
    }
    int grid = 1;
    if (plan_units(P, fm->sm_count, true, rows != nullptr, grid) != cudaSuccess) {
        set_error("fused_forward: %d frames of %dx%d are more work units than one launch takes", n, W, H);
        return QV_ERR_ARG;
    }
    // TMA input ring (opt-in, QV_FUSED_TMA=1): input a tensor map can describe (16-byte aligned base and row pitch)
    const bool tma = fm->env_tma && fm->encode_tiled && W % 16 == 0 && W >= IN_BOX && ((uintptr_t)d_in & 15) == 0;
    int b = build_of(fm->fast, false, sse, rows != nullptr, fm->env_profile, tma);
    if (b == B_PROFILE) return launch_profiled(fm, P, grid, st, launches);
    if (b == B_TMA) {
        using EncodeFn = CUresult (*)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                      const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
        const cuuint64_t dims[2] = {(cuuint64_t)W, (cuuint64_t)n * (cuuint64_t)H}, strides[1] = {(cuuint64_t)W};
        const cuuint32_t box[2] = {(cuuint32_t)IN_BOX, 1}, estr[2] = {1, 1};
        if (reinterpret_cast<EncodeFn>(fm->encode_tiled)(&P.tmap_in, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<uint8_t *>(d_in), dims, strides, box, estr,
                                                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                                                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
            b = B_WHOLE + fm->fast;                                     // no tensor map: the plain input ring
    }
    return launch(b, grid, &P, st, launches);
}

}  // namespace qv
