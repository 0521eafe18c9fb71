// qnet.cu — forward pass of the reference's Q-network (structs.jl:127-139) on the 5th-gen tensor cores.
//
//   Conv((3,3), 2=>16, relu; pad=1) -> Conv((3,3), 16=>32, relu; pad=1) -> Conv((6,6), 32=>64, relu) ->
//   Flux.flatten -> Dense(1600, 64, relu) -> Dense(64, 3)          call sites: utils.jl:165 (acting), 448 (targets)
//
// Flux's Conv is a true convolution over WHCN arrays: with the kernel flipped once on the host,
//   out(x, y, o) = b[o] + sum_{k1,k2,c} Wf[k1,k2,c,o] * in_pad(x + k1, y + k2, c),   x = Julia dim 1, y = dim 2.
//
// Kernel A: the three convolutions for 16 sample slots per CTA iteration, activations never leave shared memory.
// Every conv is an implicit GEMM on tcgen05 WITHOUT im2col: activations are stored "chunk-planar"
// ([8-channel chunk][pixel][sample slot][8 x 16-bit], the no-swizzle K-major canonical layout, one 16-byte row per
// pixel-sample), so the operand of kernel offset (k1,k2) is the same plane read at a start address shifted by a
// constant number of pixels — a different shared-memory descriptor, no data movement:
//   conv1: 2 input channels, 1 % of the FLOPs: CUDA cores, straight from the Float32 observations, run by otherwise idle
//          warps while the tensor core works through conv3 of the previous iteration;
//   conv2: rows (M) = 128 consecutive (pixel, slot) positions of the zero-padded 12x12 grids, shift = (12 k2 + k1) * 16;
//   conv3: the WEIGHTS are the M operand (two kernel rows stacked: lanes 0..63 = 64 output channels of k2 = 2j, lanes
//          64..127 = those of k2 = 2j+1), N = 80 = 5 output columns x 16 slots of one input row.
// Kernel B (k_qnet_head): Dense(1600,64,relu) as a TMA/tcgen05 GEMM over the conv3 activations with Dense(64,3) fused
// into its epilogue.
//
// Two precisions (snk_qnet_create's `precision` argument):
//   SNK_QNET_BF16 (engine 17, k_qnet_convs17): bf16 operands, FP32 accumulation, conv3 weights stationary in tensor
//          memory; the fast mode (1.5e-2 of max|Q| against Float64 — NOT the reference's Float32 fidelity).
//   SNK_QNET_F32  (k_qnet_convs_split): Float32-faithful.  Every weight and every activation is split into two fp16 numbers
//          (x = hi + lo, 22 significant bits) and all four partial products go through the tensor cores with FP32
//          accumulation:  the two halves of an ACTIVATION live in two different sample slots (slot s = hi of sample s,
//          slot s + 8 = 2^11 * lo of sample s; the layers are linear up to the epilogue, so the slots are simply two
//          independent "virtual samples" whose accumulators the epilogue adds: real = acc[s] + 2^-11 acc[s + 8]), the two
//          halves of a WEIGHT are two MMAs into the same accumulator (lo first, so that the tensor core's truncating
//          FP32 accumulation hits the small terms while the accumulator is small).  8 real samples per iteration, 4x the
//          MMAs of the bf16 mode per sample; conv1 and Dense(64,3) are plain FP32 FMAs.  Tolerance: tests/test_qnet_gpu.py.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <new>

#include "common.h"
#include "peer.h"
#include "qnet_theta.h"
#include "sm100.h"

namespace snk {
namespace qgrad {       // qnet_grads.cu
int preload_sample_grads();
int launch_sample_grads(const float *theta_dev, const float *states, const uint8_t *actions, const double *targets, long long B,
                        void *hi, void *lo, long long pitch, float *J, long long ldJ, float *loss, int sms, cudaStream_t st);
}
namespace qnet {

constexpr int THREADS = 512;                  // split engine: warps 0,1 MMA issuers, warp 2 weight producer, warps 4..15 = 3 epilogue groups
constexpr int PIX12 = 144;                    // padded 12x12 grid
constexpr int NISSUE = 2;                     // MMA-issuing warps (two schedulers): with small MMAs one thread cannot issue fast enough
constexpr int NGRP = 3;                       // epilogue groups of 4 warps (one per TMEM lane quarter)

// packed parameter blob (device): byte offsets
constexpr size_t P_W1 = 0;                                   // conv1 weights fp32 [tap = k2*3+k1][c][o] (flipped), host-side source of the kernel params
constexpr size_t P_W2 = P_W1 + 18 * 16 * 4;                  // bf16 [k2][k1][chunk (2)][o (32)][8]
constexpr size_t P_BIAS = P_W2 + 9 * 1024;                   // b1 (16) b2 (32) b3 (64) f32
constexpr size_t P_W4 = P_BIAS + 112 * 4;                    // [64][1600] bf16, columns in kernel-A order
constexpr size_t P_B4 = P_W4 + 64 * 1600 * 2, P_W5 = P_B4 + 64 * 4, P_B5 = P_W5 + 3 * 64 * 4;
constexpr size_t P_W3B = P_B5 + 16;                          // bf16 conv3 weights as 36 stacked-tap M operands of 4 KB
// Float32-faithful mode: fp16 (lo, hi) pairs of the same layouts
constexpr size_t P_S_W2 = P_W3B + 36 * 4096;                 // [k2][k1][chunk][n = (hi | lo) x 32 channels][8] fp16
constexpr size_t P_S_W3 = P_S_W2 + 2 * 9 * 1024;             // 72 blocks (k2, k1, m) of 4 KB: 128 rows = (hi | lo) x 64 channels
constexpr size_t P_S_W4 = P_S_W3 + 72 * 4096;                // [128][1600] fp16: rows [0,64) = hi, [64,128) = lo (one N = 128 operand)
constexpr size_t P_END = P_S_W4 + 128 * 1600 * 2;

__device__ __forceinline__ uint32_t pack_relu_bf16(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(fmaxf(a, 0.f), fmaxf(b, 0.f));
    return *reinterpret_cast<uint32_t *>(&h);
}

struct ConvArgs {
    const float *obs;            // (10,10,2,N) f32
    long long n;
    const uint8_t *params;       // packed blob
    __nv_bfloat16 *out3;         // [N][1600] bf16: k' = (oy*5 + ox)*64 + c
    long long *timing;           // optional (debug): clock64 stamps of block 0
    // conv1 weights [tap = k2*3+k1][c][o] (flipped) and bias, by value: kernel parameters sit in the constant bank, so
    // the FMAs of the CUDA-core conv1 take them as constant operands — no shared-memory traffic to fight the tensor
    // core's operand fetch with
    __half2 w1h[144];            // [tap*2 + c][o/2]: fp16 pairs for the packed HFMA2 path (inputs are -1..2 exactly; fp16
    __half2 b1h[8];              // accumulation over 18 taps errs ~1e-3, below the bf16 rounding of the result)
};
// Float32-faithful mode
struct SplitArgs {
    const float *obs;            // (10,10,2,N) f32
    long long n;
    const uint8_t *params;
    __half *out3;                // [2 N][1600] fp16: row 2 s = hi, row 2 s + 1 = 2^11 * lo of sample s; k' = (oy*5 + ox)*64 + c
    int *overflow;               // set to 1 when an activation left the fp16 range (|x| > 65504): the result is not valid
    long long *timing;           // optional (debug): clock64 stamps of block 0, 8 per iteration, first 16 iterations
    float w1f[288];              // conv1 weights [tap*2 + c][o] fp32 (constant-bank FFMA operands)
    float b1f[16];
};

// ---- shared layout of the 16-slot engines ----------------------------------------------------------------------
// 16 sample slots go through one iteration.  conv2's rows are [pixel of the padded 12x12 grid][slot] so that its epilogue
// writes conv3's layout ([input row r][x][slot]) with consecutive lanes on consecutive 16-byte units.  conv3 is turned around:
//   M = 128 = the 64 output channels of kernel row k2 = 2j (lanes 0..63) stacked on those of k2 = 2j+1 (lanes 64..127),
//   N = 80  = the 5 output columns x 16 slots of ONE input row r (the 5 consecutive pixels starting at tap column k1 are
//             10 contiguous 8-slot core matrices),
//   accumulator tile t (80 TMEM columns, t = 0..5) takes input rows r = t + 2j: its lower lanes hold the even-k2 part of
//   output row t, its upper lanes the odd-k2 part of output row t-1;  out[y] = lower(T_y) + upper(T_{y+1}).
namespace e16 {
constexpr int S = 16;
constexpr int ROWS12 = S * PIX12;             // 2304 flat positions [pixel][slot] = 18 tiles exactly
constexpr int A1_PLANE = ROWS12 * 16;         // bytes per 8-channel plane; shifted reads of the last tile run into the
                                              // following plane / region (their rows are discarded outputs)
constexpr int A2_PLANE = 100 * S * 16;        // [r][x][slot]
// conv2 output rows are [pixel p = 12 y + x of the padded grid][slot]: the real outputs (y < 10) are p < 120, i.e. the first
// 1920 rows = 15 tiles exactly; the last three tiles of the 12x12 grid (y = 10, 11) hold nothing and are not computed
constexpr int TILES2 = 120 * S / 128;
static_assert(TILES2 * 128 == 120 * S, "conv2 tiles must end on the last real output row");

// conv1 on the CUDA cores, one thread per (sample, image row y, half row): the 3 x 7 x 2 input patch is loaded once (42
// loads in flight together) and the five pixels are accumulated weight-major, so every conv1 weight is fetched from the
// constant bank once per five pixels.  (A pixel-at-a-time loop spent its time on 72 LDC.64 per 144 HFMA2.)
// Writes conv2's operand plane A1 ([pixel of the padded 12x12 grid][sample], chunk-planar bf16).
// SPREAD = false: a warp's lanes are consecutive half rows of one sample (coalesced loads, but every 16-byte store of the
// warp lands in the same bank group: 20-way conflicts).  SPREAD = true: a warp is 8 samples x 4 half rows, so each quarter
// warp stores 8 consecutive samples of one pixel = one conflict-free 128-byte wavefront (loads touch ~10 lines instead of ~7).
template <bool SPREAD = false>
__device__ __forceinline__ void conv1_pixmajor(const ConvArgs &a, long long s0, uint8_t *A1, int t, int nt) {
#pragma unroll 1
    for (int item = t; item < S * 20; item += nt) {
        const int s = SPREAD ? 8 * ((item >> 5) & 1) + (item & 7) : item / 20;
        const int r = SPREAD ? 4 * (item >> 6) + ((item >> 3) & 3) : item - 20 * s;
        const int y = r >> 1, x0 = (r & 1) * 5;
        const bool live = (s0 + s) < a.n;
        const float *ob = a.obs + (live ? (s0 + s) : 0) * 200;
        __half2 in[3][7][2];                                     // [k2][column x0 - 1 + j][c], value broadcast to both halves
#pragma unroll
        for (int k2 = 0; k2 < 3; k2++) {
            const int yy = y + k2 - 1;
            const bool rok = live && yy >= 0 && yy <= 9;
            const float *row = ob + (rok ? yy * 10 : 0);
#pragma unroll
            for (int j = 0; j < 7; j++) {
                const int xx = x0 - 1 + j;
                const bool ok = rok && xx >= 0 && xx <= 9;
#pragma unroll
                for (int c = 0; c < 2; c++) {
                    const float f = __ldg(row + c * 100 + (ok ? xx : 0));
                    in[k2][j][c] = __float2half2_rn(ok ? f : 0.f);
                }
            }
        }
        __half2 acc[5][8];
#pragma unroll
        for (int px = 0; px < 5; px++)
#pragma unroll
            for (int o = 0; o < 8; o++) acc[px][o] = a.b1h[o];
#pragma unroll
        for (int k2 = 0; k2 < 3; k2++)
#pragma unroll
            for (int k1 = 0; k1 < 3; k1++)
#pragma unroll
                for (int c = 0; c < 2; c++)
#pragma unroll
                    for (int o = 0; o < 8; o++) {
                        const __half2 w = a.w1h[((k2 * 3 + k1) * 2 + c) * 8 + o];
#pragma unroll
                        for (int px = 0; px < 5; px++) acc[px][o] = __hfma2(in[k2][px + k1][c], w, acc[px][o]);
                    }
        uint8_t *dst = A1 + (((y + 1) * 12 + (x0 + 1)) * S + s) * 16;
#pragma unroll
        for (int px = 0; px < 5; px++) {
            uint32_t w[8];
#pragma unroll
            for (int j = 0; j < 8; j++) { const float2 f = __half22float2(acc[px][j]); w[j] = pack_relu_bf16(f.x, f.y); }
            *reinterpret_cast<uint4 *>(dst + px * S * 16) = make_uint4(w[0], w[1], w[2], w[3]);
            *reinterpret_cast<uint4 *>(dst + px * S * 16 + A1_PLANE) = make_uint4(w[4], w[5], w[6], w[7]);
        }
    }
}
}  // namespace e16

// ---- kernel A, Float32-faithful mode: fp16 (hi, lo) split operands, weights streamed through shared memory ---------
// 8 real samples per iteration occupy the 16 slots: slot s = fp16(x), slot s + 8 = fp16(2^11 (x - fp16(x))) of sample s's
// activations x.  Both halves run through the same MMAs as two independent "virtual samples" (every layer is linear up to
// its epilogue); the epilogue adds the two accumulators (real = acc[s] + 2^-11 acc[s+8]), applies bias and relu in FP32
// and splits the result again for the next layer.  Each weight is two fp16 numbers as well (w = hi + lo, lo unscaled);
// the two halves sit side by side in ONE operand, so that they cost one MMA instead of two and land in separate
// accumulators (the small lo products are added to the large hi sums in FP32 registers, not by the tensor core's
// truncating accumulator):
//   conv2: B (N operand) = [W2 hi (32 channels) | W2 lo (32 channels)], N = 64: 9 MMAs of 128x64x16 per tile; the epilogue
//          adds accumulator columns j and j + 32;
//   conv3: A (M operand) = [W3 hi (64 channels) ; W3 lo (64 channels)] of ONE kernel tap, 128 rows; tile y (80 TMEM columns)
//          = output row y: 72 MMAs (6 x 6 taps x 2 channel halves) of 128x80x16 over input rows y .. y+5; the epilogue adds
//          TMEM lanes l and l + 64 (through shared memory: they belong to different warps).
// Both halves of the conv3 weights (2 x 147 KB) cannot stay in tensor memory, so they stream through a ring of 4 KB blocks
// (cp.async.bulk + mbarrier), 72 blocks per iteration, each used by all five tiles; the five 80-column conv3 accumulators
// fill 400 of the 512 TMEM columns and conv2 (8 buffers x 64 columns) time-shares them:  conv2 -> barrier -> conv3 (+ next
// conv1 on the CUDA cores) -> conv3 epilogue -> barrier.  Measured (tools/phase_probe.py): the kernel is bound by the tensor
// pipe's operand fetch (6.5 KB of shared memory per conv3 MMA).
// Error budget against Float64 (tests/test_qnet_gpu.py): operands carry 22 bits (2^-22 relative each), products of fp16
// numbers are exact in FP32, the accumulator adds with truncation (measured in round 1: ~3e-8 relative per MMA step;
// 9 / 72 / 25 steps per layer).  |activation| must stay below 65504 (fp16 range); the kernel raises a flag otherwise
// (snk_qnet_overflow_host).
namespace split {
#define SPLIT_STAMP(k) do { if (a.timing != nullptr && blockIdx.x == 0 && it_local >= 0 && it_local < 16 && lane == 0) a.timing[it_local * 8 + (k)] = clock64(); } while (0)
constexpr int S = e16::S, SR = 8;             // 16 slots = 8 real samples x (hi, lo)
constexpr int A2_PLANE = e16::A2_PLANE;
// conv2's input A1: rows = [pixel of the padded 12x12 grid][8 real samples] (NOT slots): the two fp16 halves of an activation sit
// along K — four planes of 8 channels: hi 0..7, hi 8..15, lo 0..7, lo 8..15 (lo UNSCALED here: both halves add into one
// accumulator; below 2^-14 it is an fp16 subnormal, 3e-8 absolute, far inside the error budget) — so a conv2 row is a real
// sample: half the rows of the slot layout and no cross-lane combine in the epilogue.
constexpr int A1_PLANE = PIX12 * SR * 16;     // 18,432 bytes per 8-channel plane
constexpr int TILES2 = 8;                     // real outputs are pixels p < 120: 960 rows = 7.5 tiles
static_assert(4 * A1_PLANE == 2 * e16::A1_PLANE, "A1 keeps its size");
constexpr int NSLOT = 8;                      // ring of 4 KB conv3 weight blocks
constexpr int NBLK = 72;                      // (k2, k1, m) weight blocks per iteration, each 128 rows = [hi | lo] x 64 channels
constexpr int NACC = 8;                       // conv2 accumulator buffers of 64 columns (all 512 columns)
constexpr int OFF_A1 = 0;
constexpr int OFF_A2 = OFF_A1 + 4 * A1_PLANE;
constexpr int OFF_W2 = OFF_A2 + 4 * A2_PLANE;
constexpr int OFF_W3 = OFF_W2 + 2 * 9 * 1024;
constexpr int OFF_BIAS = OFF_W3 + NSLOT * 4096;
constexpr int OFF_BAR = OFF_BIAS + 112 * 4;
constexpr int SMEM = OFF_BAR + 512 + 128;
static_assert(SMEM <= 232448, "split engine shared memory over the 227 KB limit");
static_assert(5 * 40 * 64 * 4 <= 4 * A2_PLANE, "epilogue scratch must fit in the conv3 input planes");
static_assert(NBLK % NSLOT == 0 && NSLOT % 2 == 0, "the issuer waits for ring slots in aligned pairs");
#ifndef SPLIT_C3_ISSUERS
#define SPLIT_C3_ISSUERS 1   /* warps issuing the conv3 MMAs */
#endif
#ifndef SPLIT_RELEASE
#define SPLIT_RELEASE 2      /* ring slots released by one commit; measured conv3 phase: 1 -> 27.2 k cycles, 2 -> 25.7 k, 4 -> 26.5 k (ring stalls) */
#endif
#ifndef SPLIT_EXP
#define SPLIT_EXP 0          /* timing experiments (garbage results): 1 = every conv3 MMA reads the same A block, 2 = the same B offset */
#endif
#ifndef SPLIT_NOCONV1
#define SPLIT_NOCONV1 0  /* timing experiment: skip conv1 (results are garbage) */
#endif
#ifndef SPLIT_NOLOAD
#define SPLIT_NOLOAD 0   /* timing experiment: skip the conv3 weight loads (results are garbage) */
#endif
constexpr float LO_SCALE = 2048.0f, LO_UNSCALE = 1.0f / 2048.0f;      // 2^11: keeps the low halves in fp16's normal range
// B-descriptor offset (16-byte units) of weight block be = (k2*6 + k1)*2 + m for tile 0 (output row 0): (k2*10 + k1)*S + 2m*(A2_PLANE/16)
__constant__ uint32_t c_boff[NBLK] = {0, 3200, 16, 3216, 32, 3232, 48, 3248, 64, 3264, 80, 3280, 160, 3360, 176, 3376, 192, 3392, 208, 3408, 224, 3424, 240, 3440, 320, 3520, 336, 3536, 352, 3552, 368, 3568, 384, 3584, 400, 3600, 480, 3680, 496, 3696, 512, 3712, 528, 3728, 544, 3744, 560, 3760, 640, 3840, 656, 3856, 672, 3872, 688, 3888, 704, 3904, 720, 3920, 800, 4000, 816, 4016, 832, 4032, 848, 4048, 864, 4064, 880, 4080};

// two values >= 0 (after relu) -> {fp16 bits of r0, r1} of their high halves, or of 2^11 x their low halves; packed
// conversions (cvt.rn.f16x2.f32): 9 instructions per pair
__device__ __forceinline__ uint32_t split_pair(float r0, float r1, bool want_lo) {
    const __half2 h = __floats2half2_rn(r0, r1);
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn((r0 - hf.x) * LO_SCALE, (r1 - hf.y) * LO_SCALE);
    const __half2 o = want_lo ? l : h;
    return *reinterpret_cast<const uint32_t *>(&o);
}
// both halves of a pair at once; SCALED: lo = 2^11 (r - hi) (slot layout), else lo = r - hi
template <bool SCALED>
__device__ __forceinline__ void split_pair2(float r0, float r1, uint32_t &hi, uint32_t &lo) {
    const __half2 h = __floats2half2_rn(r0, r1);
    const float2 hf = __half22float2(h);
    const __half2 l = SCALED ? __floats2half2_rn((r0 - hf.x) * LO_SCALE, (r1 - hf.y) * LO_SCALE) : __floats2half2_rn(r0 - hf.x, r1 - hf.y);
    hi = *reinterpret_cast<const uint32_t *>(&h);
    lo = *reinterpret_cast<const uint32_t *>(&l);
}
// x >= 0 (after relu) -> the fp16 bits of its high half, or of 2^11 x its low half
__device__ __forceinline__ unsigned short split_half(float r, bool want_lo) {
    const __half h = __float2half_rn(r);
    const __half l = __float2half_rn((r - __half2float(h)) * LO_SCALE);
    return __half_as_ushort(want_lo ? l : h);
}

// conv1 (2 -> 16 channels, 3x3, pad 1, relu) of the 8 real samples starting at s0 in plain FP32 on the CUDA cores, one
// thread per (sample, image row y, half row) as in e16::conv1_pixmajor, the 16 output channels in two passes of 8 (one
// 16-byte unit of a chunk plane each) to stay inside the register budget.  A quarter warp = 8 samples of one half row, so
// its 16-byte stores form conflict-free 128-byte wavefronts.  Writes the hi and the (unscaled) lo planes of conv2's operand A1.
__device__ __forceinline__ void conv1_f32_split(const SplitArgs &a, long long s0, uint8_t *A1, int t, int nt, float &amax) {
#pragma unroll 1
    for (int item = t; item < SR * 20; item += nt) {
        const int s = item & 7, r = item >> 3;
        const int y = r >> 1, x0 = (r & 1) * 5;
        const bool live = (s0 + s) < a.n;
        const float *ob = a.obs + (live ? (s0 + s) : 0) * 200;
        float in[3][7][2];                                       // [k2][column x0 - 1 + j][c]
#pragma unroll
        for (int k2 = 0; k2 < 3; k2++) {
            const int yy = y + k2 - 1;
            const bool rok = live && yy >= 0 && yy <= 9;
            const float *row = ob + (rok ? yy * 10 : 0);
#pragma unroll
            for (int j = 0; j < 7; j++) {
                const int xx = x0 - 1 + j;
                const bool ok = rok && xx >= 0 && xx <= 9;
#pragma unroll
                for (int c = 0; c < 2; c++) {
                    const float f = __ldg(row + c * 100 + (ok ? xx : 0));
                    in[k2][j][c] = ok ? f : 0.f;
                }
            }
        }
        uint8_t *dst = A1 + (((y + 1) * 12 + (x0 + 1)) * SR + s) * 16;
#pragma unroll
        for (int o8 = 0; o8 < 2; o8++) {
            float acc[5][8];
#pragma unroll
            for (int px = 0; px < 5; px++)
#pragma unroll
                for (int o = 0; o < 8; o++) acc[px][o] = a.b1f[o8 * 8 + o];
#pragma unroll
            for (int k2 = 0; k2 < 3; k2++)
#pragma unroll
                for (int k1 = 0; k1 < 3; k1++)
#pragma unroll
                    for (int c = 0; c < 2; c++)
#pragma unroll
                        for (int o = 0; o < 8; o++) {
                            const float w = a.w1f[((k2 * 3 + k1) * 2 + c) * 16 + o8 * 8 + o];
#pragma unroll
                            for (int px = 0; px < 5; px++) acc[px][o] = fmaf(in[k2][px + k1][c], w, acc[px][o]);
                        }
#pragma unroll
            for (int px = 0; px < 5; px++) {
                uint32_t wh[4], wl[4];
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const float r0 = fmaxf(acc[px][2 * j], 0.f), r1 = fmaxf(acc[px][2 * j + 1], 0.f);
                    amax = fmaxf(amax, fmaxf(r0, r1));
                    split_pair2<false>(r0, r1, wh[j], wl[j]);
                }
                uint8_t *d = dst + px * SR * 16 + o8 * A1_PLANE;
                *reinterpret_cast<uint4 *>(d) = make_uint4(wh[0], wh[1], wh[2], wh[3]);                      // plane o8: high halves
                *reinterpret_cast<uint4 *>(d + 2 * A1_PLANE) = make_uint4(wl[0], wl[1], wl[2], wl[3]);       // plane 2 + o8: low halves
            }
        }
    }
}

__global__ void __launch_bounds__(THREADS, 1) k_qnet_convs_split(const __grid_constant__ SplitArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
    uint8_t *A1 = smem + OFF_A1, *A2 = smem + OFF_A2;
    const float *bias = (const float *)(smem + OFF_BIAS);
    uint64_t *bars = (uint64_t *)(smem + OFF_BAR);
    uint64_t *acc_full = bars, *acc_empty = bars + NACC, *w3_full = bars + 2 * NACC, *w3_empty = w3_full + NSLOT, *c3_full = w3_empty + NSLOT;
    uint32_t *tmem_slot = (uint32_t *)(c3_full + 1);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int uwarp = __shfl_sync(0xffffffffu, warp, 0);      // the same value, provably warp-uniform for the compiler
    float amax = 0.f;                                         // largest activation this thread has produced (fp16 range check)

    for (int i = tid; i < OFF_A2 / 16; i += THREADS) reinterpret_cast<uint4 *>(smem)[i] = make_uint4(0, 0, 0, 0);   // A1 borders stay zero
    for (int i = tid; i < 2 * 9 * 1024 / 16; i += THREADS)
        reinterpret_cast<uint4 *>(smem + OFF_W2)[i] = reinterpret_cast<const uint4 *>(a.params + P_S_W2)[i];
    for (int i = tid; i < 112; i += THREADS) reinterpret_cast<float *>(smem + OFF_BIAS)[i] = reinterpret_cast<const float *>(a.params + P_BIAS)[i];
    if (tid == 0) {
        for (int i = 0; i < NACC; i++) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 4); }
        for (int i = 0; i < NSLOT; i++) { mbar_init(&w3_full[i], 1); mbar_init(&w3_empty[i], SPLIT_C3_ISSUERS); }
        mbar_init(c3_full, SPLIT_C3_ISSUERS);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    __syncthreads();
    const long long n_iter = (a.n + SR - 1) / SR;
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    const uint64_t dA1 = desc_nosw(smem_u32(A1), A1_PLANE, 128);             // conv2 A: 8-sample core matrices; + 2 planes = the lo half
    const uint64_t dA2 = desc_nosw(smem_u32(A2), A2_PLANE, 128);             // conv3 B (N operand): likewise
    const uint64_t dW2 = desc_nosw(smem_u32(smem + OFF_W2), 1024, 128);      // conv2 B: 64 rows ([hi | lo] x 32 channels), 2 KB per tap
    const uint64_t dW3 = desc_nosw(smem_u32(smem + OFF_W3), 2048, 128);      // conv3 A: 128 stacked rows, K chunks 2 KB apart

    uint32_t acc_it = 0, w3_it = 0, c3_it = 0;
    // The loop starts one pass early: pass -1 only runs the conv1 of the first real iteration, through the same (single)
    // call site as the overlapped conv1 of every later pass.
    long long it_local = -1;
    for (long long it = (long long)blockIdx.x - gridDim.x; it < n_iter; it += gridDim.x, it_local++) {
        const bool real = it_local >= 0;
        const long long s0 = it * SR;
        if (real && warp == 4) SPLIT_STAMP(0);
        if (real && warp == 2 && lane == 0) {
            // weight producer, part 1: fill the ring while conv2 runs
            for (int bi = 0; bi < NSLOT; bi++) {
                const uint32_t u = w3_it + bi;
                const int b = u % NSLOT;
                if ((b % SPLIT_RELEASE) == 0) mbar_wait(&w3_empty[b], ((u / NSLOT) & 1) ^ 1);     // one release per SPLIT_RELEASE slots
                if (SPLIT_NOLOAD) { mbar_arrive(&w3_full[b]); continue; }
                mbar_expect_tx(&w3_full[b], 4096);
                bulk_load(smem + OFF_W3 + b * 4096, a.params + P_S_W3 + (size_t)bi * 4096, 4096, &w3_full[b]);
            }
        }

        // ================= conv2: 16 -> 32, 3x3, pad 1; rows = [pixel][sample]; K = [hi ; lo] activation halves, N = [hi | lo] weight halves =================
        if (!real) {
        } else if (warp < NISSUE) {
            tc_fence_after();
            for (int t = 0; t < TILES2; t++) {
                const uint32_t u = acc_it + t;
                if ((int)(u % NISSUE) != uwarp) continue;                   // issuer w owns the tiles of its parity
                const int b = u % NACC;
                mbar_wait(&acc_empty[b], ((u / NACC) & 1) ^ 1);
                tc_fence_after();
                const uint32_t d = tmem + b * 64;
                const uint64_t at = dA1 + (uint64_t)(t * 128);
                if (elect_one()) {
#pragma unroll
                    for (int half = 1; half >= 0; half--)                   // the low activation halves first (small terms first)
#pragma unroll
                        for (int k2 = 0; k2 < 3; k2++)
#pragma unroll
                            for (int k1 = 0; k1 < 3; k1++)
                                umma_bf16(d, at + (uint64_t)(half * 2 * (A1_PLANE / 16) + (k2 * 12 + k1) * SR),
                                          dW2 + (uint64_t)((k2 * 3 + k1) * 128), idesc_f16(128, 64), (half == 1 && (k2 | k1) == 0) ? 0u : 1u);
                    umma_commit(&acc_full[b]);
                }
                __syncwarp();
            }
        } else if (warp >= 4) {
            const int grp = (warp - 4) >> 2, q = warp & 3;
            for (int t = 0; t < TILES2; t++) {
                const uint32_t u = acc_it + t;
                if ((int)(u % NGRP) != grp) continue;
                const int b = u % NACC;
                mbar_wait(&acc_full[b], (u / NACC) & 1);
                tc_fence_after();
                const int P = t * 128 + q * 32 + lane;                      // row = [pixel][sample]
                const int pix = P / SR, y = pix / 12, x = pix - 12 * y;
                const bool valid = x < 10 && y < 10;                        // other rows are discarded garbage
                uint8_t *dst = A2 + ((y * 10 + x) * S + (lane & 7)) * 16;   // [r][x][slot]: slot s = hi, slot s + 8 = 2^11 lo
                const uint32_t src = tmem + ((uint32_t)(q * 32) << 16) + b * 64;
#pragma unroll
                for (int hh = 0; hh < 2; hh++) {                            // output channels 16 hh .. 16 hh + 15
                    uint32_t vh[16], vl[16];
                    tmem_ld16(src + hh * 16, vh);                           // hi-weight products
                    tmem_ld16(src + 32 + hh * 16, vl);                      // lo-weight products
                    tmem_ld_wait();
                    if (hh == 1) {                                          // accumulator drained
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(&acc_empty[b]);
                    }
                    uint32_t wh[8], wl[8];
#pragma unroll
                    for (int j = 0; j < 16; j += 2) {
                        const float r0 = fmaxf(__uint_as_float(vh[j]) + __uint_as_float(vl[j]) + bias[16 + hh * 16 + j], 0.f);
                        const float r1 = fmaxf(__uint_as_float(vh[j + 1]) + __uint_as_float(vl[j + 1]) + bias[16 + hh * 16 + j + 1], 0.f);
                        if (valid) amax = fmaxf(amax, fmaxf(r0, r1));
                        split_pair2<true>(r0, r1, wh[j >> 1], wl[j >> 1]);
                    }
                    if (valid) {
#pragma unroll
                        for (int c8 = 0; c8 < 2; c8++) {
                            uint8_t *d8 = dst + (2 * hh + c8) * A2_PLANE;
                            *reinterpret_cast<uint4 *>(d8) = make_uint4(wh[4 * c8], wh[4 * c8 + 1], wh[4 * c8 + 2], wh[4 * c8 + 3]);
                            *reinterpret_cast<uint4 *>(d8 + SR * 16) = make_uint4(wl[4 * c8], wl[4 * c8 + 1], wl[4 * c8 + 2], wl[4 * c8 + 3]);
                        }
                    }
                }
            }
        }
        if (real) acc_it += TILES2;
        if (real && warp == 4) SPLIT_STAMP(1);
        fence_proxy_async();
        tc_fence_before();
        __syncthreads();
        if (real && warp == 4) SPLIT_STAMP(2);

        // ================= conv3: 32 -> 64, 6x6, valid; M = [hi ; lo] weight halves of one tap, tile y = output row y =================
        if (warp < NISSUE) {
            if (real && (SPLIT_C3_ISSUERS == 2 || warp == 0)) {
                // The whole issuer warp runs this loop with warp-uniform values and one elected lane issues: descriptors
                // then live in uniform registers.  The B-descriptor offset of a block comes from a constant table; blocks
                // are waited for in pairs.  With two issuers, issuer 0 owns output rows 0, 2, 4 and issuer 1 rows 1, 3.
                tc_fence_after();
                const int first = SPLIT_C3_ISSUERS == 2 ? uwarp : 0, stride = SPLIT_C3_ISSUERS;
                const uint64_t bbase = dA2 + (uint64_t)(first * 10 * S);
                const uint32_t dbase = tmem + first * 80;
                const int my_tiles = (5 - first + stride - 1) / stride;
#pragma unroll 2
                for (int bi = 0; bi < NBLK; bi += 2) {
                    const uint32_t b0 = (w3_it + bi) % NSLOT, b1 = b0 + 1;  // w3_it and bi are even
                    const uint32_t par = ((w3_it + bi) / NSLOT) & 1;       // both blocks share the ring pass
                    const uint64_t o0 = bbase + (SPLIT_EXP & 2 ? 0 : c_boff[bi]), o1 = bbase + (SPLIT_EXP & 2 ? 0 : c_boff[bi + 1]);   // SPLIT_EXP: timing experiments
                    const uint64_t w0 = dW3 + (uint64_t)((SPLIT_EXP & 1 ? 0 : b0) * 256), w1 = w0 + (SPLIT_EXP & 1 ? 0 : 256);
                    mbar_wait(&w3_full[b0], par);
                    mbar_wait(&w3_full[b1], par);
                    tc_fence_after();
                    if (elect_one()) {
                        // one weight block against all tiles, then the next: consecutive MMAs share their A operand
#pragma unroll
                        for (int i = 0; i < 5; i++)
                            if (i < my_tiles) umma_bf16(dbase + i * stride * 80, w0, o0 + (uint64_t)(i * stride * 10 * S), idesc_f16(128, 80), bi ? 1u : 0u);
#pragma unroll
                        for (int i = 0; i < 5; i++)
                            if (i < my_tiles) umma_bf16(dbase + i * stride * 80, w1, o1 + (uint64_t)(i * stride * 10 * S), idesc_f16(128, 80), 1u);
                        // one tcgen05.commit per SPLIT_RELEASE slots (each costs the MMA stream ~40 cycles): it tracks all
                        // earlier MMAs, i.e. every slot of the group
                        if ((b1 + 1) % SPLIT_RELEASE == 0) umma_commit(&w3_empty[b1 + 1 - SPLIT_RELEASE]);
                    }
                    __syncwarp();
                }
                if (elect_one()) umma_commit(c3_full);
                __syncwarp();
            }
        } else {
            if (real && warp == 2 && lane == 0) {
                for (int bi = NSLOT; bi < NBLK; bi++) {
                    const uint32_t u = w3_it + bi;
                    const int b = u % NSLOT;
                    if ((b % SPLIT_RELEASE) == 0) mbar_wait(&w3_empty[b], ((u / NSLOT) & 1) ^ 1);
                    if (SPLIT_NOLOAD) { mbar_arrive(&w3_full[b]); continue; }
                    mbar_expect_tx(&w3_full[b], 4096);
                    bulk_load(smem + OFF_W3 + b * 4096, a.params + P_S_W3 + (size_t)bi * 4096, 4096, &w3_full[b]);
                }
            }
            // next iteration's conv1 on the CUDA cores, by warps of the two schedulers without an MMA issuer
            if ((warp & 3) >= 2 && warp != 2 && it + gridDim.x < n_iter) {
                const int w7 = warp == 3 ? 0 : 2 * ((warp - 4) >> 2) + (warp & 1) + 1;      // 3,6,7,10,11,14,15 -> 0..6
                if (!SPLIT_NOCONV1) conv1_f32_split(a, (it + gridDim.x) * SR, A1, w7 * 32 + lane, 224, amax);
                if (real && warp == 15) SPLIT_STAMP(6);
            }
            if (real && warp >= 4) {
                const int grp = (warp - 4) >> 2, q = warp & 3;
                mbar_wait_relaxed(c3_full, c3_it & 1);
                tc_fence_after();
                if (warp == 4) SPLIT_STAMP(3);
                float *scratch = reinterpret_cast<float *>(A2);             // [y][column = x*8 + sample][oc]: conv3 no longer reads A2
                // Tile y = output row y.  Warp quarter q owns TMEM lanes 32q..32q+31: output channels (q & 1)*32 + lane of the
                // hi-weight half (q < 2) or of the lo-weight half (q >= 2) of the same outputs.  The lo-half warps reduce their
                // part over its two slots (column x*16 + s = high-half slot of sample s, + 8 the low one) and park it in shared
                // memory; the hi-half warps add it to theirs, bias, relu, split, store.  Group g takes rows g and g + 3.
                const int oc = (q & 1) * 32 + lane;
                const uint32_t my = tmem + ((uint32_t)(q * 32) << 16);       // + y*80: my lanes of output row y
                // even rows: the lo-half warps park, the hi-half warps finish; odd rows the other way round (all twelve warps work
                // in both phases)
                for (int y = grp; y < 5; y += NGRP) {
                    if (((y & 1) == 0) != (q >= 2)) continue;
#pragma unroll 1
                    for (int h = 0; h < 5; h++) {
                        uint32_t v[16];
                        tmem_ld16(my + y * 80 + h * 16, v);
                        tmem_ld_wait();
#pragma unroll
                        for (int i = 0; i < 8; i++)
                            scratch[(y * 40 + h * 8 + i) * 64 + oc] = fmaf(__uint_as_float(v[i + 8]), LO_UNSCALE, __uint_as_float(v[i]));
                    }
                }
                nbar_sync(1, 384);
                const float bo = bias[48 + oc];
                const int live = (int)(a.n - s0 < SR ? a.n - s0 : SR);
                for (int y = grp; y < 5; y += NGRP) {
                    if (((y & 1) == 0) == (q >= 2)) continue;
#pragma unroll 1
                    for (int h = 0; h < 5; h++) {                            // h = output column x
                        uint32_t v[16];
                        tmem_ld16(my + y * 80 + h * 16, v);
                        float other[8];                                      // all loads first: the stores below may alias as far
#pragma unroll                                                               // as the compiler knows, and would serialise them
                        for (int i = 0; i < 8; i++) other[i] = scratch[(y * 40 + h * 8 + i) * 64 + oc];
                        tmem_ld_wait();
                        unsigned short *dst = reinterpret_cast<unsigned short *>(a.out3) + 2 * s0 * 1600 + (y * 5 + h) * 64 + oc;
#pragma unroll
                        for (int i = 0; i < 8; i += 2) {                     // i = sample
                            const float r0 = fmaxf(fmaf(__uint_as_float(v[i + 8]), LO_UNSCALE, __uint_as_float(v[i])) + other[i] + bo, 0.f);
                            const float r1 = fmaxf(fmaf(__uint_as_float(v[i + 9]), LO_UNSCALE, __uint_as_float(v[i + 1])) + other[i + 1] + bo, 0.f);
                            const uint32_t ph = split_pair(r0, r1, false), pl = split_pair(r0, r1, true);
                            if (i < live) {
                                amax = fmaxf(amax, r0);
                                dst[(2 * i) * 1600] = (unsigned short)ph;
                                dst[(2 * i + 1) * 1600] = (unsigned short)pl;
                            }
                            if (i + 1 < live) {
                                amax = fmaxf(amax, r1);
                                dst[(2 * i + 2) * 1600] = (unsigned short)(ph >> 16);
                                dst[(2 * i + 3) * 1600] = (unsigned short)(pl >> 16);
                            }
                        }
                    }
                }
                tc_fence_before();
                if (warp == 4) SPLIT_STAMP(4);
            }
        }
        if (real) { w3_it += NBLK; c3_it++; }
        fence_proxy_async();
        __syncthreads();                            // conv3 accumulators drained (conv2 reuses the columns), A1/A2 handed over
        if (real && warp == 4) SPLIT_STAMP(5);
    }

    if (amax > 65504.f) *a.overflow = 1;
    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem, 512);
    }
}
}  // namespace split

// ---- kernel A, engine 17: conv3 weights stationary in tensor memory -------------------------------------------
// Engine 16's conv3 is still bound by the tensor core's shared-memory operand fetch (6.5 KB per 40-cycle MMA) and keeps
// all six accumulator tiles live, so its epilogue cannot overlap anything.  Here the 36 stacked-tap weight blocks
// (128 rows x 16 channels = 8 TMEM columns each, 288 columns in all) are written into tensor memory ONCE per CTA with
// tcgen05.st and every conv3 MMA takes its A operand from there (tcgen05.mma [d], [a_tmem], b_desc: lane = row, 32-bit
// column j = K elements 2j, 2j+1 — tools/probes/probe_ts_mma.cu).  Per MMA only the 2.5 KB of B (80 pixel-samples) come
// from shared memory: conv3 becomes math-bound, needs no weight ring, and because the weights no longer stream the six
// output tiles are computed ONE AFTER THE OTHER into two 80-column accumulators, tile t+1's MMAs under tile t's epilogue.
//   TMEM: [0,288) conv3 weights | [288,448) 2 conv3 accumulators | [448,512) 2 conv2 accumulators (conv2 also borrows the
//   first 32 columns of each conv3 accumulator while conv3 is not running: 4 conv2 buffers).
//   tile t (input rows t, t+2, t+4): lanes 0..63 = even-k2 part of output row t, lanes 64..127 = odd-k2 part of row t-1.
//   Epilogue of tile t: the lower-lane warps park their half in shared memory (two 20 KB buffers), the upper-lane warps add
//   the half parked one tile earlier, bias, relu, and write output row t-1.
// Warp roles: 0 = MMA issuer (conv2 even tiles, all of conv3), 1 = conv2 odd tiles, 4..11 = conv2 epilogue (group g drains
// buffer g) and conv3 tile epilogues (columns 0..47 | 48..79), 2, 3 and 12.. = the next iteration's conv1 on the CUDA cores (ten warps: its 320 items in one pass).
// One block barrier per iteration (conv2 -> conv3); everything else is handed over through mbarriers, so conv2 of the next
// iteration starts under the last conv3 epilogue.
namespace e17 {
constexpr int S = e16::S, A1_PLANE = e16::A1_PLANE, A2_PLANE = e16::A2_PLANE;
// conv2 output rows are [pixel p = 12 y + x of the padded grid][sample]: the real outputs (y < 10) are p < 120, i.e. the first
// 1920 rows = 15 tiles exactly; the last three tiles of the 12x12 grid (y = 10, 11) hold nothing and are not computed
constexpr int TILES2 = 120 * S / 128;
static_assert(TILES2 * 128 == 120 * S, "conv2 tiles must end on the last real output row");
constexpr int TM_W3 = 0, TM_C3 = 288, TM_C2 = 448;
constexpr int SCR = 80 * 64 * 4;              // one parked half tile: [column = x*16 + sample][oc] fp32
#ifndef E17_WARPS
#define E17_WARPS 20
#endif
#ifndef E17_SPREAD
#define E17_SPREAD 1   /* conv1 lane mapping, see conv1_pixmajor */
#endif
constexpr int NWARPS = E17_WARPS, NTHREADS = NWARPS * 32;
constexpr int NC1W = NWARPS - 10;             // warps running conv1: 2, 3 and 12.. (320 items = 10 warps: one pass)
constexpr int OFF_A1 = 0;
constexpr int OFF_A2 = OFF_A1 + 2 * A1_PLANE;
constexpr int OFF_W2 = OFF_A2 + 4 * A2_PLANE;
constexpr int OFF_SCR = OFF_W2 + 9 * 1024;
constexpr int OFF_BIAS = OFF_SCR + 2 * SCR;
constexpr int OFF_BAR = OFF_BIAS + 112 * 4;
constexpr int SMEM = OFF_BAR + 256 + 128;
static_assert(SMEM <= 232448, "engine 17 shared memory over the 227 KB limit");

// debug stamps of CTA 0 (snk_qnet_debug_timing): 64 slots per iteration, first 8 iterations; the buffer holds 512 int64
#define E17_STAMP(slot) do { if (a.timing != nullptr && blockIdx.x == 0 && lane == 0 && it_local >= 0 && it_local < 8) a.timing[it_local * 64 + (slot)] = clock64(); } while (0)
#ifndef E17_NOSTORE
#define E17_NOSTORE 0   /* timing experiment: conv3 epilogue without its global stores */
#endif
// 16 parked values of one thread (one per sample, 256 B apart) in one statement: the loads issue back to back
__device__ __forceinline__ void lds16_stride256(uint32_t saddr, float (&o)[16]) {
    asm volatile(
        "ld.shared.f32 %0, [%16];\n\tld.shared.f32 %1, [%16+256];\n\tld.shared.f32 %2, [%16+512];\n\tld.shared.f32 %3, [%16+768];\n\t"
        "ld.shared.f32 %4, [%16+1024];\n\tld.shared.f32 %5, [%16+1280];\n\tld.shared.f32 %6, [%16+1536];\n\tld.shared.f32 %7, [%16+1792];\n\t"
        "ld.shared.f32 %8, [%16+2048];\n\tld.shared.f32 %9, [%16+2304];\n\tld.shared.f32 %10, [%16+2560];\n\tld.shared.f32 %11, [%16+2816];\n\t"
        "ld.shared.f32 %12, [%16+3072];\n\tld.shared.f32 %13, [%16+3328];\n\tld.shared.f32 %14, [%16+3584];\n\tld.shared.f32 %15, [%16+3840];"
        : "=f"(o[0]), "=f"(o[1]), "=f"(o[2]), "=f"(o[3]), "=f"(o[4]), "=f"(o[5]), "=f"(o[6]), "=f"(o[7]), "=f"(o[8]), "=f"(o[9]),
          "=f"(o[10]), "=f"(o[11]), "=f"(o[12]), "=f"(o[13]), "=f"(o[14]), "=f"(o[15])
        : "r"(saddr) : "memory");
}
__device__ __forceinline__ void sts_f32(uint32_t saddr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(saddr), "f"(v) : "memory"); }
__device__ __forceinline__ uint32_t cvt_relu_bf16x2(float hi, float lo) {      // {bf16(max(hi,0)), bf16(max(lo,0))}
    uint32_t d;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
    return d;
}
__global__ void __launch_bounds__(NTHREADS, 1) k_qnet_convs17(const __grid_constant__ ConvArgs a) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 127) & ~(uintptr_t)127);
    uint8_t *A1 = smem + OFF_A1, *A2 = smem + OFF_A2;
    const float *bias = (const float *)(smem + OFF_BIAS);
    uint64_t *bars = (uint64_t *)(smem + OFF_BAR);
    uint64_t *acc_full = bars, *acc_empty = bars + 4, *c3_full = bars + 8, *c3_empty = bars + 10, *a1_full = bars + 12, *c3_done = bars + 13;
    uint64_t *c3_drained = bars + 14;                         // [2]: the last two conv3 tiles of an iteration have left their accumulators
    uint32_t *tmem_slot = (uint32_t *)(bars + 16);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int uwarp = __shfl_sync(0xffffffffu, warp, 0);      // the same value, provably warp-uniform for the compiler

    for (int i = tid; i < OFF_A2 / 16; i += NTHREADS) reinterpret_cast<uint4 *>(smem)[i] = make_uint4(0, 0, 0, 0);   // A1 borders stay zero
    for (int i = tid; i < 9 * 1024 / 16; i += NTHREADS)
        reinterpret_cast<uint4 *>(smem + OFF_W2)[i] = reinterpret_cast<const uint4 *>(a.params + P_W2)[i];
    for (int i = tid; i < 112; i += NTHREADS) reinterpret_cast<float *>(smem + OFF_BIAS)[i] = reinterpret_cast<const float *>(a.params + P_BIAS)[i];
    if (tid == 0) {
        for (int i = 0; i < 4; i++) { mbar_init(&acc_full[i], 1); mbar_init(&acc_empty[i], 4); }
        for (int i = 0; i < 2; i++) { mbar_init(&c3_full[i], 1); mbar_init(&c3_empty[i], 8); mbar_init(&c3_drained[i], 8); }
        mbar_init(a1_full, NC1W);
        mbar_init(c3_done, 1);
        fence_barrier_init();
    }
    if (warp == 0) tmem_alloc(tmem_slot, 512);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    {
        // conv3 weights -> tensor memory: block be = (j*6 + k1)*2 + m at columns 8 be; a thread writes the 16 channels of
        // the stacked row (= TMEM lane) 32 q + lane of its warp's lane quarter q
        const int q = warp & 3;
        for (int be = warp >> 2; be < 36; be += NTHREADS / 128) {
            const uint8_t *src = a.params + P_W3B + (size_t)be * 4096 + (q * 32 + lane) * 16;
            const uint4 lo = *reinterpret_cast<const uint4 *>(src), hi = *reinterpret_cast<const uint4 *>(src + 2048);
            tmem_st8(tmem + ((uint32_t)(q * 32) << 16) + TM_W3 + be * 8, lo, hi);
        }
        tmem_st_wait();
    }
    const long long n_iter = (a.n + S - 1) / S;
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    const uint64_t dA1 = desc_nosw(smem_u32(A1), A1_PLANE, 128);             // conv2 A: 8-sample core matrices, contiguous
    const uint64_t dA2 = desc_nosw(smem_u32(A2), A2_PLANE, 128);             // conv3 B (N operand): likewise
    const uint64_t dW2 = desc_nosw(smem_u32(smem + OFF_W2), 512, 128);
    const bool conv1_warp = warp == 2 || warp == 3 || warp >= 12;
    const int w7 = warp <= 3 ? warp - 2 : warp - 10;                          // 2, 3, 12, 13, ... -> 0, 1, 2, 3, ...

    uint32_t acc_it = 0, c3_it = 0;
    // The loop starts one pass early: pass -1 only runs the conv1 of the first real iteration, through the same (single)
    // call site as the overlapped conv1 of every later pass.
    long long it_local = -1;
    for (long long it = (long long)blockIdx.x - gridDim.x; it < n_iter; it += gridDim.x, it_local++) {
        const bool real = it_local >= 0;
        const long long s0 = it * S;
        if (real) {
            if (warp == 4) E17_STAMP(0);
            // ================= conv2: 16 -> 32, 3x3, pad 1; rows = [pixel][sample] =================
            if (warp < 2) {
                mbar_wait(a1_full, (uint32_t)it_local & 1);                   // conv1 of this iteration has written A1
                tc_fence_after();
                // Four accumulators: 0, 1 are conv2's own columns, 2, 3 borrow the first 32 columns of the two conv3 accumulators
                // (idle during conv2 once the last two conv3 tiles of the previous iteration have been drained).  Running tile
                // index u -> buffer u & 3, issuer u & 1 (so an issuer alternates between two buffers and is always one tile ahead
                // of the epilogue), epilogue group u & 1.
                for (int t = (uwarp - acc_it) & 1; t < TILES2; t += 2) {
                    const uint32_t u = acc_it + t, bsel = u & 3;
                    if (bsel >= 2 && it_local > 0 && t < 4) mbar_wait(&c3_drained[bsel - 2], ((uint32_t)it_local - 1) & 1);
                    mbar_wait(&acc_empty[bsel], ((u >> 2) & 1) ^ 1);
                    tc_fence_after();
                    const uint32_t d = tmem + (bsel < 2 ? TM_C2 + bsel * 32 : TM_C3 + (bsel - 2) * 80);
                    const uint64_t at = dA1 + (uint64_t)(t * 128);
                    if (elect_one()) {
#pragma unroll
                        for (int k2 = 0; k2 < 3; k2++)
#pragma unroll
                            for (int k1 = 0; k1 < 3; k1++)
                                umma_bf16(d, at + (uint64_t)((k2 * 12 + k1) * S), dW2 + (uint64_t)((k2 * 3 + k1) * 64),
                                          idesc_bf16(128, 32), (k2 | k1) ? 1u : 0u);
                        umma_commit(&acc_full[bsel]);
                    }
                    __syncwarp();
                }
            } else if (warp >= 4 && warp < 12) {
                // a waiter has to see EVERY phase of its mbarrier (parity waits only tell adjacent phases apart): group g drains
                // buffers g and g + 2 in strict alternation, nobody else waits on their barriers
                const int grp = (warp - 4) >> 2, q = warp & 3;
                if (it_local > 0) mbar_wait(c3_done, ((uint32_t)it_local - 1) & 1);   // the previous conv3 has read A2
                for (int t = (grp - acc_it) & 1; t < TILES2; t += 2) {
                    const uint32_t u = acc_it + t;
                    const int b = u & 3;                                        // group g sees every phase of buffers g and g + 2
                    mbar_wait(&acc_full[b], (u >> 2) & 1);
                    tc_fence_after();
                    uint32_t v[32];
                    const uint32_t src = tmem + ((uint32_t)(q * 32) << 16) + (b < 2 ? TM_C2 + b * 32 : TM_C3 + (b - 2) * 80);
                    tmem_ld16(src, *reinterpret_cast<uint32_t(*)[16]>(&v[0]));
                    tmem_ld16(src + 16, *reinterpret_cast<uint32_t(*)[16]>(&v[16]));
                    tmem_ld_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&acc_empty[b]);
                    const int P = t * 128 + q * 32 + lane;
                    const int pix = P / S, s = P - pix * S, y = pix / 12, x = pix - 12 * y;
                    if (x < 10 && y < 10) {
                        uint8_t *dst = A2 + ((y * 10 + x) * S + s) * 16;          // [r][x][sample]
#pragma unroll
                        for (int c8 = 0; c8 < 4; c8++) {
                            uint32_t w[4];
#pragma unroll
                            for (int j = 0; j < 4; j++)
                                w[j] = pack_relu_bf16(__uint_as_float(v[c8 * 8 + 2 * j]) + bias[16 + c8 * 8 + 2 * j],
                                                      __uint_as_float(v[c8 * 8 + 2 * j + 1]) + bias[16 + c8 * 8 + 2 * j + 1]);
                            *reinterpret_cast<uint4 *>(dst + c8 * A2_PLANE) = make_uint4(w[0], w[1], w[2], w[3]);
                        }
                    }
                }
            }
            acc_it += TILES2;
            fence_proxy_async();
            tc_fence_before();
            __syncthreads();                        // A2 complete; every conv2 MMA has completed (its epilogue ran), A1 is free
            if (warp == 4) E17_STAMP(3);
        }

        // ================= conv3: 32 -> 64, 6x6, valid; stationary weights, tile after tile =================
        if (warp == 0) {
            if (real) {
                tc_fence_after();
#pragma unroll 1
                for (int t = 0; t < 6; t++) {
                    const uint32_t u = c3_it + t;
                    const int b = t & 1;
                    mbar_wait(&c3_empty[b], ((u >> 1) & 1) ^ 1);
                    tc_fence_after();
                    E17_STAMP(8 + t);
                    const uint32_t d = tmem + TM_C3 + b * 80;
                    const uint64_t bt = dA2 + (uint64_t)(t * 10 * S);       // input row t (16-byte units: one per pixel-sample)
                    if (elect_one()) {
#pragma unroll
                        for (int j = 0; j < 3; j++)
#pragma unroll
                            for (int k1 = 0; k1 < 6; k1++)
#pragma unroll
                                for (int m = 0; m < 2; m++)
                                    umma_bf16_ts(d, tmem + TM_W3 + ((j * 6 + k1) * 2 + m) * 8,
                                                 bt + (uint64_t)((2 * j * 10 + k1) * S + 2 * m * (A2_PLANE / 16)),
                                                 idesc_bf16(128, 80), (j | k1 | m) ? 1u : 0u);
                        umma_commit(&c3_full[b]);
                        if (t == 5) umma_commit(c3_done);
                    }
                    __syncwarp();
                    E17_STAMP(16 + t);
                }
            }
        } else {
            // next iteration's conv1 on the CUDA cores (A1 is free: see the barrier above)
            if (conv1_warp && it + gridDim.x < n_iter) {
                e16::conv1_pixmajor<E17_SPREAD != 0>(a, (it + gridDim.x) * S, A1, w7 * 32 + lane, NC1W * 32);
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(a1_full);
                if (warp == 13) E17_STAMP(6);
            }
            if (real && warp >= 4 && warp < 12) {
                // Tile t: lanes 0..63 (warps q = 0,1) hold the even-k2 part of output row t, lanes 64..127 (q = 2,3) the odd-k2
                // part of row t-1.  The q < 2 warps park their half (+ bias) in one of two shared-memory buffers; one tile later
                // the q >= 2 warps add it to theirs, relu, and write the finished row.  A thread and the thread that parked for
                // it have the same lane index, so one 128-thread named barrier per group and tile orders the hand-over:
                // passing it at tile t means tile t-1's half is parked and tile t-2's has been read.
                const int grp = (warp - 4) >> 2, q = warp & 3;
                const int c_lo = grp == 0 ? 0 : 3, c_hi = grp == 0 ? 3 : 5;  // 16-column chunks (= output column x) of this group
                const int oc = (q & 1) * 32 + lane;
                const float bo = bias[48 + oc];
                const int live = (int)(a.n - s0 < 16 ? a.n - s0 : 16);
                const uint32_t scr = smem_u32(smem + OFF_SCR) + oc * 4;
#pragma unroll 1
                for (int t = 0; t < 6; t++) {
                    const uint32_t u = c3_it + t;
                    const int b = t & 1;
                    mbar_wait(&c3_full[b], (u >> 1) & 1);
                    tc_fence_after();
                    if (warp == 6) E17_STAMP(24 + t);
                    nbar_sync(1 + grp, 128);
                    const uint32_t my = tmem + ((uint32_t)(q * 32) << 16) + TM_C3 + b * 80;
                    if (q < 2 && t < 5) {
                        const uint32_t park = scr + (uint32_t)((t & 1) * SCR);
#pragma unroll 1
                        for (int h = c_lo; h < c_hi; h++) {
                            uint32_t v[16];
                            tmem_ld16(my + h * 16, v);
                            tmem_ld_wait();
                            if (h == c_hi - 1) {                                 // accumulator drained
                                tc_fence_before();
                                __syncwarp();
                                if (lane == 0) { mbar_arrive(&c3_empty[b]); if (t >= 4) mbar_arrive(&c3_drained[b]); }
                            }
#pragma unroll
                            for (int i = 0; i < 16; i++) sts_f32(park + (h * 16 + i) * 256, __uint_as_float(v[i]) + bo);
                        }
                        if (warp == 4) E17_STAMP(56 + t);
                    } else if (q >= 2 && t >= 1) {
                        const uint32_t park = scr + (uint32_t)(((t - 1) & 1) * SCR);
                        const int y = t - 1;
                        if (warp == 6) E17_STAMP(32 + t);
#pragma unroll 1
                        for (int h = c_lo; h < c_hi; h++) {                      // h = output column x
                            uint32_t v[16];
                            float other[16];
                            tmem_ld16(my + h * 16, v);
                            lds16_stride256(park + h * 16 * 256, other);
                            tmem_ld_wait();
                            if (h == c_hi - 1) {
                                tc_fence_before();
                                __syncwarp();
                                if (lane == 0) { mbar_arrive(&c3_empty[b]); if (t >= 4) mbar_arrive(&c3_drained[b]); }
                                if (warp == 6) E17_STAMP(40 + t);
                            }
                            uint16_t *dst = reinterpret_cast<uint16_t *>(a.out3 + s0 * 1600 + (y * 5 + h) * 64 + oc);
#pragma unroll
                            for (int i = 0; i < 16; i += 2) {                    // i = sample
                                const uint32_t pk = cvt_relu_bf16x2(__uint_as_float(v[i + 1]) + other[i + 1], __uint_as_float(v[i]) + other[i]);
                                if (E17_NOSTORE) continue;
                                if (i < live) dst[i * 1600] = (uint16_t)pk;
                                if (i + 1 < live) dst[(i + 1) * 1600] = (uint16_t)(pk >> 16);
                            }
                        }
                        if (warp == 6) E17_STAMP(48 + t);
                    } else {
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) { mbar_arrive(&c3_empty[b]); if (t >= 4) mbar_arrive(&c3_drained[b]); }
                    }
                }
            }
        }
        if (real) c3_it += 6;
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 0) {
        tc_fence_after();
        tmem_dealloc(tmem, 512);
    }
}
}  // namespace e17

// ---- kernel B: Dense(1600,64,relu) + Dense(64,3) ---------------------------------------------------------
// SPLIT = false: X = out3 [N][1600] bf16, W4' [64][1600] bf16, N = 64 accumulator columns.
// SPLIT = true (Float32-faithful): X = out3 [2N][1600] fp16 (row 2s = hi, row 2s+1 = 2^11 lo of sample s), W4' [128][1600]
// fp16 (rows 0..63 = hi, 64..127 = lo halves of the weights: ONE N = 128 operand, so X is read once); the epilogue adds
// accumulator columns j and j + 64 (weight halves) and lanes l and l ^ 1 (activation halves).  A 128-row tile covers 64 samples.
constexpr int HB_M = 128, HB_K = 64, HB_STAGES = 6;
constexpr int HB_THREADS = 192;
template <bool SPLIT>
struct HeadCfg {
    static constexpr int N = SPLIT ? 128 : 64;                           // accumulator columns per tile
    static constexpr int STAGE_BYTES = HB_M * 128 + N * 128;             // A tile 16 KB + W4 tile (SWIZZLE_128B rows of 64 16-bit elements)
    static constexpr int SMEM = HB_STAGES * STAGE_BYTES + 1024 + 256 + 64 * 4 + 3 * 64 * 4 + 16;
};

struct HeadArgs {
    const uint8_t *params;
    float *q_out;               // (3, N)
    long long n;
};

template <bool SPLIT>
__global__ void __launch_bounds__(HB_THREADS, 1) k_qnet_head(const __grid_constant__ CUtensorMap map_x,   // out3, box 128 x 64
                                                             const __grid_constant__ CUtensorMap map_w,   // W4', box N x 64
                                                             const HeadArgs a) {
    using C = HeadCfg<SPLIT>;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = (uint8_t *)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t *bars = (uint64_t *)(smem + HB_STAGES * C::STAGE_BYTES);
    uint64_t *full = bars, *empty = bars + HB_STAGES, *acc_full = bars + 2 * HB_STAGES, *acc_empty = acc_full + 2;
    uint32_t *tmem_slot = (uint32_t *)(acc_empty + 2);
    float *s_b4 = (float *)(tmem_slot + 4), *s_w5 = s_b4 + 64, *s_b5 = s_w5 + 192;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long n_rows = SPLIT ? 2 * a.n : a.n;
    const long long n_tiles = (n_rows + HB_M - 1) / HB_M;
    constexpr int KB = 1600 / HB_K;             // 25 k-blocks
    constexpr uint32_t IDESC = SPLIT ? idesc_f16(128, 128) : idesc_bf16(128, 64);

    for (int i = tid; i < 64; i += HB_THREADS) s_b4[i] = reinterpret_cast<const float *>(a.params + P_B4)[i];
    for (int i = tid; i < 192; i += HB_THREADS) s_w5[i] = reinterpret_cast<const float *>(a.params + P_W5)[i];
    if (tid < 3) s_b5[tid] = reinterpret_cast<const float *>(a.params + P_B5)[tid];
    if (tid == 0) {
        for (int s = 0; s < HB_STAGES; s++) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        for (int s = 0; s < 2; s++) { mbar_init(&acc_full[s], 1); mbar_init(&acc_empty[s], 4); }
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc(tmem_slot, 2 * C::N);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0) {
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x)
                for (int kb = 0; kb < KB; kb++) {
                    mbar_wait(&empty[stage], phase ^ 1);
                    uint8_t *st = smem + stage * C::STAGE_BYTES;
                    mbar_expect_tx(&full[stage], C::STAGE_BYTES);
                    tma_load_2d(&map_x, &full[stage], st, kb * HB_K, (int)((n_tiles - 1 - t) * HB_M));   // newest rows first, see below
                    tma_load_2d(&map_w, &full[stage], st + HB_M * 128, kb * HB_K, 0);
                    if (++stage == HB_STAGES) { stage = 0; phase ^= 1; }
                }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            int stage = 0, acc = 0;
            uint32_t phase = 0, acc_phase = 0;
            for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
                mbar_wait(&acc_empty[acc], acc_phase ^ 1);
                tc_fence_after();
                for (int kb = 0; kb < KB; kb++) {
                    mbar_wait(&full[stage], phase);
                    tc_fence_after();
                    const uint32_t base = smem_u32(smem + stage * C::STAGE_BYTES);
#pragma unroll
                    for (int k = 0; k < HB_K / 16; k++)          // 128-byte swizzled rows: 8-row atoms 1024 B apart
                        umma_bf16(tmem + acc * C::N, desc_sw<1024, LAYOUT_SW128>(base) + (uint64_t)(2 * k),
                                  desc_sw<1024, LAYOUT_SW128>(base + HB_M * 128) + (uint64_t)(2 * k), IDESC, (kb | k) ? 1u : 0u);
                    umma_commit(&empty[stage]);
                    if (++stage == HB_STAGES) { stage = 0; phase ^= 1; }
                }
                umma_commit(&acc_full[acc]);
                if (++acc == 2) { acc = 0; acc_phase ^= 1; }
            }
        }
    } else {
        const int q = warp & 3;
        int acc = 0;
        uint32_t acc_phase = 0;
        for (long long t = blockIdx.x; t < n_tiles; t += gridDim.x) {
            mbar_wait(&acc_full[acc], acc_phase);
            tc_fence_after();
            float q0 = s_b5[0], q1 = s_b5[1], q2 = s_b5[2];
#pragma unroll
            for (int h = 0; h < 4; h++) {
                uint32_t v[16], vl[16];
                const uint32_t src = tmem + ((uint32_t)(q * 32) << 16) + acc * C::N + h * 16;
                tmem_ld16(src, v);
                if (SPLIT) tmem_ld16(src + 64, vl);                                   // the lo-weight half of the same outputs
                tmem_ld_wait();
#pragma unroll
                for (int j = 0; j < 16; j++) {
                    const int c = h * 16 + j;
                    float x = __uint_as_float(v[j]);
                    if (SPLIT) {                                                      // even lane: high-half row, odd lane: low-half row
                        x = (x + __uint_as_float(vl[j])) * ((lane & 1) ? 1.0f / 2048.0f : 1.0f);
                        x += __shfl_xor_sync(0xffffffffu, x, 1);
                    }
                    const float hv = fmaxf(x + s_b4[c], 0.f);                        // Dense(1600,64,relu)
                    q0 = fmaf(s_w5[c * 3 + 0], hv, q0);                              // Dense(64,3); W5 stored (3,64) column-major
                    q1 = fmaf(s_w5[c * 3 + 1], hv, q1);
                    q2 = fmaf(s_w5[c * 3 + 2], hv, q2);
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&acc_empty[acc]);
            // tiles are taken from the END of the batch: the conv kernel wrote out3 in sample order and the last ~100 MB of it
            // are still in L2 when this kernel starts; reading front to back would evict them before they are reached
            const long long row = (n_tiles - 1 - t) * HB_M + q * 32 + lane;
            const long long s = SPLIT ? row >> 1 : row;
            if (s < a.n && !(SPLIT && (lane & 1))) { a.q_out[3 * s] = q0; a.q_out[3 * s + 1] = q1; a.q_out[3 * s + 2] = q2; }
            if (++acc == 2) { acc = 0; acc_phase ^= 1; }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc(tmem, 2 * C::N);
    }
}

// ---- parameter packing: k_qnet_train_apply at create, after every update and in set_params --------------------------
__device__ static inline uint16_t f2bf(float f) {            // round-to-nearest-even
    uint32_t u;
    memcpy(&u, &f, 4);
    if ((u & 0x7F800000u) == 0x7F800000u) return (uint16_t)(u >> 16);
    u += 0x7FFFu + ((u >> 16) & 1u);
    return (uint16_t)(u >> 16);
}
// w = hi + lo in fp16 (lo unscaled): part 0 = lo, part 1 = hi
__device__ static inline uint16_t f2h_part(float w, int part) {
    const __half h = __float2half_rn(w);
    if (part) return __half_as_ushort(h);
    return __half_as_ushort(__float2half_rn(w - __half2float(h)));
}

// The one definition of every device layout of the weights, as a scatter from a parameter's Flux index p (theta =
// Flux.destructure(q_net): W1(3,3,2,16) b1 W2(3,3,16,32) b2 W3(6,6,32,64) b3 W4(64,1600) b4 W5(3,64) b5, column-major): writes
// every byte derived from theta[p].  `theta` is the handle's extended copy (the two re-ordered W3 copies behind it).
__device__ __forceinline__ void scatter_param(float w, int p, float *theta, uint8_t *params) {
    using namespace qgrad;
    auto h = [&](size_t off) { return reinterpret_cast<uint16_t *>(params + off); };
    auto f = [&](size_t off) { return reinterpret_cast<float *>(params + off); };
    theta[p] = w;
    if (p < O_B1) {                                     // W1 (3,3,2,16) -> [tap = k2*3 + k1][c][o], flipped: k = 2 - a
        const int a1 = p % 3, a2 = (p / 3) % 3, c = (p / 9) % 2, o = p / 18;
        f(P_W1)[(((2 - a2) * 3 + (2 - a1)) * 2 + c) * 16 + o] = w;
    } else if (p < O_W2) {
        f(P_BIAS)[p - O_B1] = w;
    } else if (p < O_B2) {                              // W2 (3,3,16,32) -> [k2][k1][chunk][o][8]; split: [k2][k1][chunk][hi|lo o][8]
        const int i = p - O_W2, a1 = i % 3, a2 = (i / 3) % 3, c = (i / 9) % 16, o = i / 144;
        const int kc = ((2 - a2) * 3 + (2 - a1)) * 2 + c / 8;
        h(P_W2)[(kc * 32 + o) * 8 + c % 8] = f2bf(w);
        h(P_S_W2)[(kc * 64 + o) * 8 + c % 8] = f2h_part(w, 1);
        h(P_S_W2)[(kc * 64 + 32 + o) * 8 + c % 8] = f2h_part(w, 0);
    } else if (p < O_W3) {
        f(P_BIAS)[16 + p - O_B2] = w;
    } else if (p < O_B3) {                              // W3 (6,6,32,64): the gradient kernel's two copies and both tensor-core layouts
        const int i = p - O_W3, t = i % 36, c = (i / 36) % 32, o = i / 1152;
        theta[O_W3OF + (c * 36 + t) * 64 + o] = w;
        theta[O_W3CF + (o * 36 + t) * 32 + c] = w;
        const int k1 = 5 - t % 6, k2 = 5 - t / 6, m = c / 16, kk = c % 16;
        auto core = [&](int R) { return (((kk / 8) * 16 + R / 8) * 8 + R % 8) * 8 + kk % 8; };
        h(P_W3B)[(size_t)(((k2 / 2) * 6 + k1) * 2 + m) * 2048 + core(64 * (k2 % 2) + o)] = f2bf(w);
        const size_t blk = (size_t)((k2 * 6 + k1) * 2 + m) * 2048;
        h(P_S_W3)[blk + core(o)] = f2h_part(w, 1);
        h(P_S_W3)[blk + core(64 + o)] = f2h_part(w, 0);
    } else if (p < O_W4) {
        f(P_BIAS)[48 + p - O_B3] = w;
    } else if (p < O_B4) {                              // W4 (64,1600), kF = x + 5 y + 25 c -> [n][(y*5 + x)*64 + c]
        const int i = p - O_W4, n = i % 64, kF = i / 64;
        const size_t k = (size_t)((kF / 5) % 5 * 5 + kF % 5) * 64 + kF / 25;
        h(P_W4)[(size_t)n * 1600 + k] = f2bf(w);
        h(P_S_W4)[(size_t)n * 1600 + k] = f2h_part(w, 1);
        h(P_S_W4)[(size_t)(64 + n) * 1600 + k] = f2h_part(w, 0);
    } else if (p < O_W5) {
        f(P_B4)[p - O_B4] = w;
    } else if (p < O_B5) {
        f(P_W5)[p - O_W5] = w;
    } else {
        f(P_B5)[p - O_B5] = w;
    }
}

// A running sum: [NP] Float64 sums of the rows, [NP] the loss, [NP + 1] the number of samples summed so far (exact in Float64).
constexpr int SUM_LEN = qgrad::NP + 2;

struct ApplyArgs {
    const float *theta_src;      // non-NULL: no update, theta_src is the new theta (snk_qnet_set_params)
    const float *rows;           // [nrows][NP] per-sample gradient rows of one chunk of the minibatch (k_sample_grads)
    const float *losses;         // [nrows] per-sample losses
    int nrows;                   // 0 in the last pass of a learner group: the chain's final sum is the whole minibatch
    const double *sum_in;        // [SUM_LEN] the running sum this chunk continues (a peer's in a learner group), NULL: 0
    double *sum_out;             // [SUM_LEN] where a pass that is not the last leaves its running sum
    int last;                    // the sum is complete: apply it, B = its sample count
    float *acc;                  // RMSProp state of theta
    double eta, rho, one_m_rho, eps;
    float *grad_out, *loss_out;  // optional
    float *theta;                // the handle's extended theta
    uint8_t *params;             // the handle's packed blob
    int *overflow;               // SNK_QNET_F32: a parameter left the fp16 range of the split operands; NULL in bf16 mode
};

// One thread per parameter (thread NP: the loss and the sample count).  g = Float32(sum_i J_i / B), the sum a Float64 running
// sum in sample order, rounded once: the order depends on B only, wherever the chunks of the sum were added (one handle's
// scratch chunks, or the ranks of a learner group, each continuing its predecessor's sum).  Then Flux.Optimise's RMSProp
// (apply! + update!, utils.jl:466) with Julia's promotions: Float64 hyper-parameters, Float32 arrays, every operation rounded
// on its own (no FMA contraction).
constexpr int APPLY_THREADS = 256;
__global__ void __launch_bounds__(APPLY_THREADS) k_qnet_train_apply(const ApplyArgs a) {
    using qgrad::NP;
    const int p = blockIdx.x * APPLY_THREADS + threadIdx.x;
    if (p > NP) return;
    float w;
    if (a.theta_src == nullptr) {
        const float *src = p < NP ? a.rows + p : a.losses;
        const long long ld = p < NP ? NP : 1;
        double s = a.sum_in != nullptr ? a.sum_in[p] : 0.0;
#pragma unroll 8
        for (int r = 0; r < a.nrows; r++) s = __dadd_rn(s, (double)src[r * ld]);
        const double count = (a.sum_in != nullptr ? a.sum_in[NP + 1] : 0.0) + (double)a.nrows;
        if (!a.last) {
            a.sum_out[p] = s;
            if (p == NP) a.sum_out[NP + 1] = count;
            return;
        }
        const float g = (float)__ddiv_rn(s, count);
        if (p == NP) {
            if (a.loss_out != nullptr) *a.loss_out = g;
            return;
        }
        if (a.grad_out != nullptr) a.grad_out[p] = g;
        const double gd = (double)g;
        // acc = rho acc + (1 - rho) g g;  delta = g (eta / (sqrt(acc) + eps)), sqrt in Float32;  theta -= delta
        const float acc = (float)__dadd_rn(__dmul_rn(a.rho, (double)a.acc[p]), __dmul_rn(__dmul_rn(a.one_m_rho, gd), gd));
        a.acc[p] = acc;
        const float delta = (float)__dmul_rn(gd, __ddiv_rn(a.eta, __dadd_rn((double)__fsqrt_rn(acc), a.eps)));
        w = __fsub_rn(a.theta[p], delta);
    } else {
        if (p == NP) return;
        w = a.theta_src[p];
    }
    if (a.overflow != nullptr && !(fabsf(w) <= 65504.0f)) *a.overflow = 1;
    scatter_param(w, p, a.theta, a.params);
}

// ---- the data-parallel learner group (snk_qnet_group_*, DESIGN §5f) ----------------------------------------------------
// Rank r of R continues the running sum rank r - 1 published with its own rows and publishes the result; every rank then
// applies the sum of rank R - 1.  The peer memory of a rank is ONE snk_ipc_alloc allocation (one 64-byte handle):
//   [0, 8 MAX_WORLD)                   flags: slot q = the last update (epoch) whose running sum rank q has published
//   GROUP_OFF_SUM + k GROUP_SUM_BYTES   the running sum (SUM_LEN doubles) this rank published at an update of parity k
// Double buffering by parity is enough: a rank overwrites its sum of update e at update e + 2, and before that (in update
// e + 1) it has waited for rank R - 1's sum of e + 1.  Rank R - 1 published e + 1 only after every rank had, and each rank
// published e + 1 only after its last reads of update e (its predecessor's sum, rank R - 1's final sum) had finished.
constexpr size_t GROUP_OFF_SUM = 256, GROUP_SUM_BYTES = (size_t)SUM_LEN * 8;
constexpr size_t GROUP_PEER_BYTES = GROUP_OFF_SUM + 2 * GROUP_SUM_BYTES;

struct GroupFlags {
    unsigned long long *p[MAX_WORLD];
};

// One CTA, run on the rank's stream between the kernels of an update (a spinning kernel of one CTA leaves the GPU to the
// other virtual ranks of one process, whatever stream each of them is on).  signal: thread q tells rank q that this rank has
// published its sum of `epoch`; then thread 0 waits until rank `wait_for` (>= 0) has published its sum of `epoch`.
__global__ void k_group_sync(GroupFlags peers, const unsigned long long *mine, int world, int rank, int signal, int wait_for,
                             unsigned long long epoch, int *timed_out) {
    const int q = threadIdx.x;
    if (signal && q < world) peer_signal(peers.p[q] + rank, epoch);
    if (q == 0 && wait_for >= 0) peer_wait(mine + wait_for, epoch, timed_out);
}

}  // namespace qnet
}  // namespace snk

using namespace snk;
using namespace snk::qnet;

struct snk_qnet_s {
    __half2 w1h[144], b1h[8];    // conv1 weights of the bf16 mode (kernel parameters)
    float w1f[288], b1f[16];     // the same in FP32 for the Float32-faithful mode
    long long *timing;
    int device;
    int precision;               // SNK_QNET_BF16 | SNK_QNET_F32
    uint8_t *params;
    float *theta;                // Flux.destructure(q_net) as given, Float32 on the device, followed by two re-ordered copies of W3 (per-sample gradients)
    void *out3;                  // conv3 activations: bf16 [cap][1600] or fp16 [2 cap][1600]
    long long out3_cap;          // in samples
    int *d_overflow;             // SNK_QNET_F32: an activation left the fp16 range
    int sms;
    // learner (snk_qnet_train_step): per-sample gradient rows of one chunk of the minibatch, grown on demand up to 2 * sms samples
    float *rows;
    float *row_loss;
    double *gsum;                // the running sum (SUM_LEN) carried between chunks
    long long rows_cap;          // in samples
    // conv1's weights are kernel parameters read from w1h / b1h / w1f / b1f (DESIGN §5b): every write of the weights on the device
    // copies them into conv1_host and records conv1_ready; create, and after an update the next forward, waits for that event and
    // rebuilds the host fields (fetch_conv1)
    float *conv1_host;           // pinned: P_W1 (288) then b1 (16)
    cudaEvent_t conv1_ready;
    int conv1_pending;
};

// one rank of a data-parallel learner (DESIGN §5f); the layout of `mem` is described at k_group_sync
struct snk_qnet_group_s {
    snk_qnet_s *q;
    int world, rank, device;
    bool connected;
    unsigned long long epoch;    // updates so far
    uint8_t *mem;                // this rank's flags and published sums (snk_ipc_alloc)
    uint8_t *peer_mem[MAX_WORLD];
    void *opened[MAX_WORLD];     // snk_ipc_import mappings to close
    int *d_timed_out;
    // ALL of this rank's rows stay resident (B_local x 0.73 MB): it cannot reduce a chunk before its predecessor's sum arrives
    float *rows, *row_loss;
    long long rows_cap;          // in samples
};

static void set_conv1(snk_qnet_s *q, const float *w1f, const float *b1f) {
    for (int i = 0; i < 144; i++) q->w1h[i] = __floats2half2_rn(w1f[2 * i], w1f[2 * i + 1]);
    for (int i = 0; i < 8; i++) q->b1h[i] = __floats2half2_rn(b1f[2 * i], b1f[2 * i + 1]);
    memcpy(q->w1f, w1f, sizeof(q->w1f));
    memcpy(q->b1f, b1f, sizeof(q->b1f));
}

// after k_qnet_train_apply: bring conv1's new weights to the host (the forward launches read them from there)
static int enqueue_conv1_refresh(snk_qnet_s *q, cudaStream_t st) {
    SNK_CUDA(cudaMemcpyAsync(q->conv1_host, q->params + P_W1, 288 * 4, cudaMemcpyDeviceToHost, st));
    SNK_CUDA(cudaMemcpyAsync(q->conv1_host + 288, q->params + P_BIAS, 16 * 4, cudaMemcpyDeviceToHost, st));
    SNK_CUDA(cudaEventRecord(q->conv1_ready, st));
    q->conv1_pending = 1;
    return SNK_OK;
}

static int fetch_conv1(snk_qnet_s *q) {
    SNK_CUDA(cudaEventSynchronize(q->conv1_ready));
    set_conv1(q, q->conv1_host, q->conv1_host + 288);
    q->conv1_pending = 0;
    return SNK_OK;
}

static ApplyArgs rmsprop_args(float *acc, double eta, double rho, double epsilon, float *grad_out, float *loss_out) {
    ApplyArgs a = {};
    a.acc = acc; a.eta = eta; a.rho = rho; a.one_m_rho = 1.0 - rho; a.eps = epsilon;
    a.grad_out = grad_out; a.loss_out = loss_out;
    return a;
}

static int launch_apply(snk_qnet_s *q, ApplyArgs &a, cudaStream_t st) {
    a.theta = q->theta;
    a.params = q->params;
    a.overflow = q->precision == SNK_QNET_F32 ? q->d_overflow : nullptr;
    k_qnet_train_apply<<<(qgrad::NP + APPLY_THREADS) / APPLY_THREADS, APPLY_THREADS, 0, st>>>(a);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

extern "C" {

int snk_qnet_create(snk_qnet *out, const float *theta_host, int64_t n_params, int device, int precision) {
    SNK_REQUIRE(out != nullptr && theta_host != nullptr, "null argument");
    SNK_REQUIRE(n_params == 181395, "theta must be Flux.destructure of the two-frame Q-net (181,395 parameters, structs.jl:127-139)");
    SNK_REQUIRE(precision == SNK_QNET_BF16 || precision == SNK_QNET_F32, "precision must be SNK_QNET_BF16 or SNK_QNET_F32");
    *out = nullptr;
    if (precision == SNK_QNET_F32)
        for (int64_t i = 0; i < n_params; i++)
            if (!(fabsf(theta_host[i]) <= 65504.0f))
                return fail(SNK_ERR_UNSUPPORTED, "snk_qnet_create: parameter %lld = %g is outside the fp16 range of the split operands",
                            (long long)i, (double)theta_host[i]);
    DeviceGuard guard(device);
    SNK_CUDA(cudaGetLastError());
    snk_qnet_s *q = new (std::nothrow) snk_qnet_s();      // value-initialised: every member zero, so destroy frees what exists
    if (q == nullptr) return fail(SNK_ERR_INVALID, "out of host memory");
    q->device = device;
    q->precision = precision;
    cudaDeviceGetAttribute(&q->sms, cudaDevAttrMultiProcessorCount, device);
    auto build = [&]() -> int {
        SNK_CUDA(cudaMalloc((void **)&q->params, P_END));
        SNK_CUDA(cudaMemset(q->params, 0, P_END));                       // the padding no layout writes
        SNK_CUDA(cudaMalloc((void **)&q->theta, qgrad::THETA_EXT * 4));
        SNK_CUDA(cudaMemset(q->theta, 0, qgrad::THETA_EXT * 4));         // the gap [NP, O_W3OF)
        SNK_CUDA(cudaMalloc((void **)&q->d_overflow, sizeof(int)));
        SNK_CUDA(cudaMemset(q->d_overflow, 0, sizeof(int)));
        SNK_CUDA(cudaMallocHost((void **)&q->conv1_host, 304 * 4));
        SNK_CUDA(cudaEventCreateWithFlags(&q->conv1_ready, cudaEventDisableTiming));
        SNK_CUDA(cudaMemcpy(q->theta, theta_host, qgrad::NP * 4, cudaMemcpyHostToDevice));
        // in place on the legacy stream behind the copies: thread p reads theta_src[p] before it writes theta[p], and its
        // other writes lie at >= O_W3OF, which no thread reads
        ApplyArgs a = {};
        a.theta_src = q->theta;
        int rc;
        if ((rc = launch_apply(q, a, 0)) != SNK_OK) return rc;
        if ((rc = enqueue_conv1_refresh(q, 0)) != SNK_OK) return rc;
        return fetch_conv1(q);
    };
    const int rc = build();
    if (rc != SNK_OK) {
        snk_qnet_destroy(q);
        return rc;
    }
    *out = q;
    return SNK_OK;
}

int snk_qnet_destroy(snk_qnet q) {
    if (q == nullptr) return SNK_OK;
    DeviceGuard guard(q->device);
    if (q->params) cudaFree(q->params);
    if (q->theta) cudaFree(q->theta);
    if (q->out3) cudaFree(q->out3);
    if (q->d_overflow) cudaFree(q->d_overflow);
    if (q->rows) cudaFree(q->rows);
    if (q->row_loss) cudaFree(q->row_loss);
    if (q->gsum) cudaFree(q->gsum);
    if (q->conv1_ready) cudaEventDestroy(q->conv1_ready);
    if (q->conv1_host) cudaFreeHost(q->conv1_host);
    delete q;
    return SNK_OK;
}

// Flux.gradient of mean(huber(q_net(s)[a], y)) + update!(RMSProp(eta, rho, epsilon), theta, g) (utils.jl:452-466): the
// per-sample rows of k_sample_grads, chunk by chunk, reduced and applied by k_qnet_train_apply, which also re-derives every
// device layout of the weights
int snk_qnet_train_step(snk_qnet q, const float *states, const uint8_t *actions, const double *targets, int64_t B, float *acc,
                        double eta, double rho, double epsilon, float *grad_out, float *loss_out, void *cuda_stream) {
    SNK_REQUIRE(B >= 1, "B must be >= 1");
    SNK_REQUIRE(eta > 0.0 && rho >= 0.0 && rho < 1.0 && epsilon >= 0.0, "RMSProp needs eta > 0, 0 <= rho < 1 and epsilon >= 0");
    SNK_REQUIRE(q != nullptr && states != nullptr && actions != nullptr && targets != nullptr && acc != nullptr, "null argument");
    DeviceGuard guard(q->device);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const long long chunk = 2ll * q->sms;          // one CTA of k_sample_grads per sample and slot; bounds the scratch (215 MB)
    const long long need = B < chunk ? B : chunk;
    if (q->rows_cap < need) {
        SNK_CUDA(cudaStreamSynchronize(st));
        if (q->rows) { SNK_CUDA(cudaFree(q->rows)); q->rows = nullptr; }
        if (q->row_loss) { SNK_CUDA(cudaFree(q->row_loss)); q->row_loss = nullptr; }
        q->rows_cap = 0;
        SNK_CUDA(cudaMalloc((void **)&q->rows, (size_t)need * qgrad::NP * 4));
        SNK_CUDA(cudaMalloc((void **)&q->row_loss, (size_t)need * 4));
        if (q->gsum == nullptr) SNK_CUDA(cudaMalloc((void **)&q->gsum, SUM_LEN * sizeof(double)));
        q->rows_cap = need;
    }
    ApplyArgs a = rmsprop_args(acc, eta, rho, epsilon, grad_out, loss_out);
    a.rows = q->rows; a.losses = q->row_loss; a.sum_out = q->gsum;
    for (long long s0 = 0; s0 < B; s0 += chunk) {
        const long long n = B - s0 < chunk ? B - s0 : chunk;
        int rc = qgrad::launch_sample_grads(q->theta, states + s0 * 200, actions + s0, targets + s0, n, nullptr, nullptr, 0, q->rows,
                                            qgrad::NP, q->row_loss, q->sms, st);
        if (rc != SNK_OK) return rc;
        a.nrows = (int)n; a.sum_in = s0 == 0 ? nullptr : q->gsum; a.last = s0 + n == B;
        if ((rc = launch_apply(q, a, st)) != SNK_OK) return rc;
    }
    return enqueue_conv1_refresh(q, st);
}

// theta <- theta_dev (update_target_net!, utils.jl:469-472): the same kernel without a gradient re-derives every layout
int snk_qnet_set_params(snk_qnet q, const float *theta_dev, void *cuda_stream) {
    SNK_REQUIRE(q != nullptr && theta_dev != nullptr, "null argument");
    DeviceGuard guard(q->device);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    ApplyArgs a = {};
    a.theta_src = theta_dev;
    int rc = launch_apply(q, a, st);
    if (rc != SNK_OK) return rc;
    return enqueue_conv1_refresh(q, st);
}

int snk_qnet_params(snk_qnet q, const float **theta_dev) {
    SNK_REQUIRE(q != nullptr && theta_dev != nullptr, "null argument");
    *theta_dev = q->theta;
    return SNK_OK;
}

// per-sample gradients of huber(q_net(s_i)[a_i], y_i) (utils.jl:452-466), always from the Float32 weights: csrc/qnet_grads.cu
int snk_qnet_sample_grads(snk_qnet q, const float *states, const uint8_t *actions, const double *targets, int64_t B, void *hi,
                          void *lo, int64_t pitch_elems, float *J_f32, int64_t ldJ, float *loss, void *cuda_stream) {
    SNK_REQUIRE(q != nullptr && states != nullptr && actions != nullptr && targets != nullptr && B >= 0, "bad argument");
    SNK_REQUIRE((hi == nullptr) == (lo == nullptr), "hi and lo planes come together");
    SNK_REQUIRE(hi != nullptr || J_f32 != nullptr || loss != nullptr, "no output requested");
    SNK_REQUIRE(hi == nullptr || (pitch_elems >= 181395 && pitch_elems % 8 == 0 && (((uintptr_t)hi | (uintptr_t)lo) & 15u) == 0),
                "planes need a pitch >= 181395 that is a multiple of 8 elements and 16-byte aligned bases");
    SNK_REQUIRE(J_f32 == nullptr || ldJ >= 181395, "ldJ too small");
    if (B == 0) return SNK_OK;
    DeviceGuard guard(q->device);
    return qgrad::launch_sample_grads(q->theta, states, actions, targets, B, hi, lo, pitch_elems, J_f32, ldJ, loss, q->sms,
                                      (cudaStream_t)cuda_stream);
}

int snk_qnet_precision(snk_qnet q, int *precision) {
    SNK_REQUIRE(q != nullptr && precision != nullptr, "null argument");
    *precision = q->precision;
    return SNK_OK;
}

// SNK_QNET_F32: 1 if any forward since the last call produced an activation outside the fp16 range (then its Q-values are
// not valid); reads and clears the flag (synchronises the device)
int snk_qnet_overflow_host(snk_qnet q, int *flag) {
    SNK_REQUIRE(q != nullptr && flag != nullptr, "null argument");
    DeviceGuard guard(q->device);
    SNK_CUDA(cudaMemcpy(flag, q->d_overflow, sizeof(int), cudaMemcpyDeviceToHost));
    if (*flag) SNK_CUDA(cudaMemset(q->d_overflow, 0, sizeof(int)));
    return SNK_OK;
}

// debug (bf16 mode): device buffer of 512 int64 receiving clock64 stamps of the conv phases of CTA 0; NULL = off
int snk_qnet_debug_timing(snk_qnet q, long long *device_buf) {
    SNK_REQUIRE(q != nullptr, "null qnet");
    q->timing = device_buf;
    return SNK_OK;
}

int snk_qnet_forward(snk_qnet q, const float *obs_f32, int64_t N, float *q_out_3xN, void *cuda_stream) {
    SNK_REQUIRE(q != nullptr && obs_f32 != nullptr && q_out_3xN != nullptr && N > 0, "bad argument");
    DeviceGuard guard(q->device);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const bool f32 = q->precision == SNK_QNET_F32;
    if (q->conv1_pending) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        SNK_CUDA(cudaStreamIsCapturing(st, &cs));
        if (cs != cudaStreamCaptureStatusNone)
            return fail(SNK_ERR_INVALID, "snk_qnet_forward: the weights of this handle changed on the device (snk_qnet_train_step / "
                                         "snk_qnet_set_params) and conv1's kernel parameters must be fetched by the host first: "
                                         "run one forward outside the stream capture");
        const int rc = fetch_conv1(q);
        if (rc != SNK_OK) return rc;
    }
    const size_t row_bytes = f32 ? 2 * 1600 * 2 : 1600 * 2;             // per sample
    if (q->out3_cap < N) {
        if (q->out3) { SNK_CUDA(cudaStreamSynchronize(st)); SNK_CUDA(cudaFree(q->out3)); q->out3 = nullptr; q->out3_cap = 0; }
        long long cap = (N + 127) / 128 * 128;
        SNK_CUDA(cudaMalloc(&q->out3, (size_t)cap * row_bytes));
        SNK_CUDA(cudaMemsetAsync(q->out3, 0, (size_t)cap * row_bytes, st));
        q->out3_cap = cap;
    }
    int grid, rc;
    CUtensorMap mx, mw;
    auto make_map = [&](CUtensorMap *m, const void *base, long long rows, int box_rows) {     // rows of 1600 fp16 / bf16
        return make_map_2d_16bit(m, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, base, rows, 1600, 1600,
                                 box_rows, HB_K, CU_TENSOR_MAP_SWIZZLE_128B);
    };
    if (f32) {
        SplitArgs sa;
        sa.obs = obs_f32; sa.n = N; sa.params = q->params; sa.out3 = (__half *)q->out3; sa.overflow = q->d_overflow;
        sa.timing = q->timing;
        memcpy(sa.w1f, q->w1f, sizeof(sa.w1f));
        memcpy(sa.b1f, q->b1f, sizeof(sa.b1f));
        const long long n_iter = (N + split::SR - 1) / split::SR;
        grid = (int)(n_iter < q->sms ? n_iter : q->sms);
        SNK_CUDA(cudaFuncSetAttribute(split::k_qnet_convs_split, cudaFuncAttributeMaxDynamicSharedMemorySize, split::SMEM));
        split::k_qnet_convs_split<<<grid, THREADS, split::SMEM, st>>>(sa);
        SNK_CUDA(cudaGetLastError());
        if ((rc = make_map(&mx, q->out3, 2 * q->out3_cap, HB_M)) != SNK_OK) return rc;
        if ((rc = make_map(&mw, q->params + P_S_W4, 128, 128)) != SNK_OK) return rc;
    } else {
        ConvArgs ca;
        ca.obs = obs_f32; ca.n = N; ca.params = q->params; ca.out3 = (__nv_bfloat16 *)q->out3; ca.timing = q->timing;
        for (int i = 0; i < 144; i++) ca.w1h[i] = q->w1h[i];
        for (int i = 0; i < 8; i++) ca.b1h[i] = q->b1h[i];
        const long long n_iter = (N + e17::S - 1) / e17::S;
        grid = (int)(n_iter < q->sms ? n_iter : q->sms);
        SNK_CUDA(cudaFuncSetAttribute(e17::k_qnet_convs17, cudaFuncAttributeMaxDynamicSharedMemorySize, e17::SMEM));
        e17::k_qnet_convs17<<<grid, e17::NTHREADS, e17::SMEM, st>>>(ca);
        SNK_CUDA(cudaGetLastError());
        if ((rc = make_map(&mx, q->out3, q->out3_cap, HB_M)) != SNK_OK) return rc;
        if ((rc = make_map(&mw, q->params + P_W4, 64, 64)) != SNK_OK) return rc;
    }
    HeadArgs ha;
    ha.params = q->params; ha.q_out = q_out_3xN; ha.n = N;
    const long long n_tiles = ((f32 ? 2 * N : N) + HB_M - 1) / HB_M;
    grid = (int)(n_tiles < q->sms ? n_tiles : q->sms);
    if (f32) {
        SNK_CUDA(cudaFuncSetAttribute(k_qnet_head<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, HeadCfg<true>::SMEM));
        k_qnet_head<true><<<grid, HB_THREADS, HeadCfg<true>::SMEM, st>>>(mx, mw, ha);
    } else {
        SNK_CUDA(cudaFuncSetAttribute(k_qnet_head<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, HeadCfg<false>::SMEM));
        k_qnet_head<false><<<grid, HB_THREADS, HeadCfg<false>::SMEM, st>>>(mx, mw, ha);
    }
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

// ---- data-parallel learner group (DESIGN §5f) ----------------------------------------------------------------------------
int snk_qnet_group_create(snk_qnet_group *out, snk_qnet q, int world, int rank) {
    SNK_REQUIRE(out != nullptr, "null argument");
    *out = nullptr;
    SNK_REQUIRE(world >= 1 && world <= MAX_WORLD, "world must be 1 .. 16");
    SNK_REQUIRE(rank >= 0 && rank < world, "rank must be 0 .. world - 1");
    SNK_REQUIRE(q != nullptr, "null qnet");
    DeviceGuard guard(q->device);
    snk_qnet_group_s *g = new (std::nothrow) snk_qnet_group_s();
    if (g == nullptr) return fail(SNK_ERR_INVALID, "out of host memory");
    g->q = q; g->world = world; g->rank = rank; g->device = q->device;
    auto build = [&]() -> int {
        int rc;
        if ((rc = snk_ipc_alloc((void **)&g->mem, GROUP_PEER_BYTES)) != SNK_OK) return rc;
        SNK_CUDA(cudaMemset(g->mem, 0, GROUP_OFF_SUM));
        SNK_CUDA(cudaMalloc((void **)&g->d_timed_out, sizeof(int)));
        SNK_CUDA(cudaMemset(g->d_timed_out, 0, sizeof(int)));
        // load the update's kernels now (module loading is lazy): a first launch while a peer wait of this process spins
        // would block the host until that wait gives up
        cudaFuncAttributes fa;
        SNK_CUDA(cudaFuncGetAttributes(&fa, k_group_sync));
        SNK_CUDA(cudaFuncGetAttributes(&fa, k_qnet_train_apply));
        return qgrad::preload_sample_grads();
    };
    const int rc = build();
    if (rc != SNK_OK) {
        snk_qnet_group_destroy(g);
        return rc;
    }
    g->peer_mem[rank] = g->mem;
    g->connected = world == 1;
    *out = g;
    return SNK_OK;
}

int snk_qnet_group_destroy(snk_qnet_group g) {
    if (g == nullptr) return SNK_OK;
    DeviceGuard guard(g->device);
    cudaDeviceSynchronize();
    for (void *p : g->opened) if (p) snk_ipc_close(p);
    if (g->mem) snk_ipc_free(g->mem);
    if (g->d_timed_out) cudaFree(g->d_timed_out);
    if (g->rows) cudaFree(g->rows);
    if (g->row_loss) cudaFree(g->row_loss);
    delete g;
    return SNK_OK;
}

int snk_qnet_group_export_host(snk_qnet_group g, uint8_t *handle64) {
    SNK_REQUIRE(g != nullptr && handle64 != nullptr, "null argument");
    DeviceGuard guard(g->device);
    return snk_ipc_export(g->mem, handle64);
}

int snk_qnet_group_connect_host(snk_qnet_group g, const uint8_t *handles, int n_handles) {
    SNK_REQUIRE(g != nullptr && handles != nullptr, "null argument");
    SNK_REQUIRE(n_handles == g->world, "one handle per rank is needed");
    SNK_REQUIRE(!g->connected || g->world == 1, "already connected");
    DeviceGuard guard(g->device);
    for (int r = 0; r < g->world; r++) {
        if (r == g->rank) continue;
        void *p = nullptr;
        int rc = snk_ipc_import(handles + (size_t)r * SNK_QNET_GROUP_HANDLE_BYTES, &p);
        if (rc != SNK_OK) return rc;
        g->opened[r] = p;
        g->peer_mem[r] = (uint8_t *)p;
    }
    g->connected = true;
    return SNK_OK;
}

int snk_qnet_group_connect_local(snk_qnet_group g, const snk_qnet_group *peers, int n_peers) {
    SNK_REQUIRE(g != nullptr && peers != nullptr, "null argument");
    SNK_REQUIRE(n_peers == g->world, "one group per rank is needed");
    for (int r = 0; r < g->world; r++)
        SNK_REQUIRE(peers[r] != nullptr && peers[r]->rank == r && peers[r]->world == g->world && peers[r]->device == g->device,
                    "peer list does not match");
    SNK_REQUIRE(peers[g->rank] == g, "peer list does not match");
    for (int r = 0; r < g->world; r++) g->peer_mem[r] = peers[r]->mem;
    g->connected = true;
    return SNK_OK;
}

// k_sample_grads into the resident rows -> wait for rank - 1's sum -> continue it with my rows and publish -> wait for rank
// world - 1's sum -> apply it (RMSProp + every layout) -> conv1 refresh.  No host synchronisation.
int snk_qnet_group_train_step(snk_qnet_group g, const float *states, const uint8_t *actions, const double *targets,
                              int64_t B_local, float *acc, double eta, double rho, double epsilon, float *grad_out,
                              float *loss_out, void *cuda_stream) {
    SNK_REQUIRE(g != nullptr, "null group");
    SNK_REQUIRE(g->connected, "group not connected (snk_qnet_group_connect_host / connect_local)");
    SNK_REQUIRE(B_local >= 1 && B_local <= (1ll << 30), "B_local must be 1 .. 2^30");
    SNK_REQUIRE(eta > 0.0 && rho >= 0.0 && rho < 1.0 && epsilon >= 0.0, "RMSProp needs eta > 0, 0 <= rho < 1 and epsilon >= 0");
    SNK_REQUIRE(states != nullptr && actions != nullptr && targets != nullptr && acc != nullptr, "null argument");
    DeviceGuard guard(g->device);
    snk_qnet_s *q = g->q;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    if (g->rows_cap < B_local) {
        // only a buffer in use needs the wait: the first call must not block the host, whose stream may already wait on the
        // device for a peer's call the same host thread has yet to enqueue (a replay group's sample, DESIGN §5g)
        if (g->rows != nullptr) SNK_CUDA(cudaStreamSynchronize(st));
        if (g->rows) { SNK_CUDA(cudaFree(g->rows)); g->rows = nullptr; }
        if (g->row_loss) { SNK_CUDA(cudaFree(g->row_loss)); g->row_loss = nullptr; }
        g->rows_cap = 0;
        SNK_CUDA(cudaMalloc((void **)&g->rows, (size_t)B_local * qgrad::NP * 4));
        SNK_CUDA(cudaMalloc((void **)&g->row_loss, (size_t)B_local * 4));
        g->rows_cap = B_local;
    }
    int rc = qgrad::launch_sample_grads(q->theta, states, actions, targets, B_local, nullptr, nullptr, 0, g->rows, qgrad::NP,
                                        g->row_loss, q->sms, st);
    if (rc != SNK_OK) return rc;
    const unsigned long long e = ++g->epoch;
    const size_t sum_off = GROUP_OFF_SUM + (e & 1) * GROUP_SUM_BYTES;
    GroupFlags peers;
    for (int r = 0; r < g->world; r++) peers.p[r] = (unsigned long long *)g->peer_mem[r];
    const unsigned long long *mine = (const unsigned long long *)g->mem;
    auto sync = [&](int signal, int wait_for) -> int {
        k_group_sync<<<1, 32, 0, st>>>(peers, mine, g->world, g->rank, signal, wait_for, e, g->d_timed_out);
        SNK_CUDA(cudaGetLastError());
        return SNK_OK;
    };
    if (g->rank > 0 && (rc = sync(0, g->rank - 1)) != SNK_OK) return rc;
    ApplyArgs a = rmsprop_args(acc, eta, rho, epsilon, grad_out, loss_out);
    a.rows = g->rows; a.losses = g->row_loss; a.nrows = (int)B_local;
    a.sum_in = g->rank > 0 ? (const double *)(g->peer_mem[g->rank - 1] + sum_off) : nullptr;
    a.sum_out = (double *)(g->mem + sum_off);
    if ((rc = launch_apply(q, a, st)) != SNK_OK) return rc;
    if ((rc = sync(1, g->world - 1)) != SNK_OK) return rc;
    a.rows = a.losses = nullptr; a.nrows = 0;
    a.sum_in = (const double *)(g->peer_mem[g->world - 1] + sum_off); a.sum_out = nullptr; a.last = 1;
    if ((rc = launch_apply(q, a, st)) != SNK_OK) return rc;
    return enqueue_conv1_refresh(q, st);
}

int snk_qnet_group_status_host(snk_qnet_group g, int *timed_out) {
    SNK_REQUIRE(g != nullptr && timed_out != nullptr, "null argument");
    DeviceGuard guard(g->device);
    SNK_CUDA(cudaMemcpy(timed_out, g->d_timed_out, 4, cudaMemcpyDeviceToHost));
    if (*timed_out) return fail(SNK_ERR_TIMEOUT, "snk_qnet_group: a peer did not publish its running sum within ~20 s");
    return SNK_OK;
}

}  // extern "C"
