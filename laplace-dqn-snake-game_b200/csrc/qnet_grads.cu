// qnet_grads.cu — per-sample gradients of the DQN loss, the rows of the matrix J whose Gram BASELINE config 5b names
// ("Gram/D matrix of per-sample gradients ... over a 50k-transition buffer").
//
// Reference: the loss of train! (utils.jl:452-466; dup compute_D.jl:102-116, la_utils.jl:193-207)
//     q_pred = q_net(states);  q_sel = q_pred[a_i, i];  Flux.huber_loss(q_sel, q_target)         (delta = 1)
// through the network of structs.jl:127-139.  Row i of J is d huber(q_net(s_i)[a_i], y_i) / d theta with theta in
// Flux.destructure order (W1 b1 W2 b2 W3 b3 W4 b4 W5 b5, column-major) — the per-sample term, without the 1/B of the batch
// mean.  The reference itself never forms per-sample gradients (Zygote returns their mean); the oracle is a Float64
// torch.func evaluation of the same expression (tests/test_sample_grads_gpu.py) — parity unpinned by the reference.
//
// One CTA (10 warps) per sample, all activations and back-propagated signals of the sample in shared memory, plain FP32 FMAs: per
// sample the contractions are 25..2304 deep — CUDA-core work; the kernel is bound by FP32 issue (14.6 MFLOP per sample) and
// by the 725 KB (two bf16 planes) it writes per sample.  The row goes STRAIGHT into the bf16 hi / lo planes the Gram
// kernel consumes (hi = bf16(v), lo = bf16(v - hi): the same split as k_gram_pack), optionally also as Float32.
// Where the weights come from (measured: what bounded the first version was not FP32 issue but the load/store unit — a
// warp-wide load whose lanes touch 32 different cache lines costs ~32 cycles, and one shared-memory load per FMA saturates
// the shared-memory pipe):
//   W1, W2 (19 KB)  staged in shared memory once per CTA, W2 as [c][tap][o] so that the forward pass (lanes = output
//                   channels) and the backward-data pass (lanes = input channels) both read it without bank conflicts;
//   W3 (295 KB)     read from L2 through two re-ordered copies appended to theta by snk_qnet_create: output channel
//                   fastest for the forward pass, input channel fastest for the backward-data pass — the 32 lanes of a warp
//                   read one 128-byte line;
//   W4 (410 KB)     rows of 64 consecutive floats, read by half warps (forward: lanes = output units).
// The conv passes are register-tiled (a thread owns 5-25 outputs) so that one shared-memory load feeds 3-6 FMAs.
#include <cuda_bf16.h>

#include "common.h"
#include "qnet_theta.h"

namespace snk {
namespace qgrad {

constexpr int NT = 320, NW = NT / 32;      // 10 warps: the conv3 backward-data pass has 32 x 10 row tasks
// shared memory map (floats)
constexpr int S_XIN = 0;                       // [2][12][12]   input, zero padded by 1
constexpr int S_A1 = S_XIN + 2 * 144;          // [16][12][12]  relu(conv1), zero padded by 1
constexpr int S_A2 = S_A1 + 16 * 144;          // [32][10][10]  relu(conv2)
constexpr int S_A3 = S_A2 + 3200;              // [64][5][5]    relu(conv3) = Flux.flatten order x + 5 y + 25 c
constexpr int S_HID = S_A3 + 1600;             // [64]          relu(dense1)
constexpr int S_GH = S_HID + 64;               // [64]          d loss / d (dense1 pre-activation)
constexpr int S_Q = S_GH + 64;                 // [4]           q-values, [3] = d loss / d q[a]
constexpr int S_RED = S_Q + 4;                 // [320]         reduction scratch
constexpr int S_G3 = S_RED + 320;              // [64][5][5]    d loss / d (conv3 pre-activation)
constexpr int S_PART = S_G3 + 1600;            // [256][25]     conv3 forward: partial sums of the four channel quarters
constexpr int G2C = 145;                       // channel stride of the padded conv2 gradient: odd, so lanes that differ in the channel hit different banks
constexpr int S_G2 = S_PART + 256 * 25;        // [32][145]     d loss / d (conv2 pre-activation), [12][12] zero padded by 1
constexpr int S_G1 = S_G2 + 32 * G2C;          // [16][10][10]  d loss / d (conv1 pre-activation)
constexpr int S_END = S_G1 + 1600;             // everything below is re-zeroed / rewritten per CTA start
constexpr int S_W1 = S_END;                    // [288]      W1, Flux order, staged once per CTA
constexpr int W2C = 290;                       // W2s[c*290 + tap*32 + o]: 290 = 2 mod 32 (16 input channels -> 16 banks), even (8-byte loads of o pairs)
constexpr int S_W2 = S_W1 + 288;               // [16][290]  W2, tap = a1 + 3 a2
constexpr int S_TOTAL = S_W2 + 16 * W2C;
constexpr int SMEM_BYTES = S_TOTAL * 4;        // 107.8 KB: two CTAs per SM

struct GradArgs {
    const float *theta;          // 181,395 Float32, Flux.destructure order
    const float *states;         // (10,10,2,B) f32
    const uint8_t *actions;      // (B) 0-based index into available_actions
    const double *targets;       // (B) Float64 (what snk_masked_target returns)
    long long B;
    __nv_bfloat16 *hi, *lo;     // planes [B][pitch] or NULL
    long long pitch;
    float *J;                    // [B][ldJ] Float32 or NULL
    long long ldJ;
    float *loss;                 // (B) or NULL
};

struct Row {
    __nv_bfloat16 *hi, *lo;
    float *J;
};
// (hi, lo) of two values, each pair packed into 32 bits.  The packed conversion (one F2FP for two values, on the ALU pipe)
// instead of four scalar F2F: the kernel converts 363,000 values per sample and F2F issues at a quarter of the rate.
__device__ __forceinline__ uint32_t split2(float v0, float v1, uint32_t &lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
    const uint32_t hb = *reinterpret_cast<const uint32_t *>(&h);
    const __nv_bfloat162 l = __floats2bfloat162_rn(v0 - __uint_as_float(hb << 16), v1 - __uint_as_float(hb & 0xffff0000u));
    lo = *reinterpret_cast<const uint32_t *>(&l);
    return hb;
}
__device__ __forceinline__ void emit1(const Row &r, int idx, float v) {
    if (r.hi != nullptr) {
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        r.hi[idx] = h;
        r.lo[idx] = __float2bfloat16_rn(v - __bfloat162float(h));
    }
    if (r.J != nullptr) r.J[idx] = v;
}
template <int N>      // N = 4 or 8 consecutive values, idx a multiple of N
__device__ __forceinline__ void emitv(const Row &r, int idx, const float (&v)[N]) {
    if (r.hi != nullptr) {
        uint32_t h[N / 2], l[N / 2];
#pragma unroll
        for (int j = 0; j < N / 2; j++) h[j] = split2(v[2 * j], v[2 * j + 1], l[j]);
        if (N == 8) {
            *reinterpret_cast<uint4 *>(r.hi + idx) = make_uint4(h[0], h[1], h[2], h[3]);
            *reinterpret_cast<uint4 *>(r.lo + idx) = make_uint4(l[0], l[1], l[2], l[3]);
        } else {
            *reinterpret_cast<uint2 *>(r.hi + idx) = make_uint2(h[0], h[1]);
            *reinterpret_cast<uint2 *>(r.lo + idx) = make_uint2(l[0], l[1]);
        }
    }
    if (r.J != nullptr) {
#pragma unroll
        for (int j = 0; j < N; j++) r.J[idx + j] = v[j];
    }
}

// out(x, y, o) = relu(b[o] + sum_{c,a2,a1} W[a1 + K (a2 + K (c + CIN o))] * in[c][y + K-1-a2][x + K-1-a1])   (true convolution;
// `in` is the zero-padded input plane, row pitch IP, channel stride IC).  A warp owns an output channel, its lanes up to PPL
// output positions each; the weight is a warp-uniform shared-memory load (W staged by the caller).
template <int K, int CIN, int COUT, int OW, int IP, int IC, int PPL>
__device__ __forceinline__ void conv_forward(const float *W, const float *__restrict__ b, const float *in, float *out,
                                             int out_pitch, int out_cs, int out_off, int warp, int lane) {
    for (int o = warp; o < COUT; o += NW) {
        float acc[PPL];
        int base[PPL];
        bool live[PPL];
#pragma unroll
        for (int j = 0; j < PPL; j++) {
            const int p = lane + 32 * j;
            live[j] = p < OW * OW;
            const int y = live[j] ? p / OW : 0, x = live[j] ? p - OW * (p / OW) : 0;
            base[j] = (y + K - 1) * IP + (x + K - 1);
            acc[j] = __ldg(b + o);
        }
        const float *w = W + (size_t)K * K * CIN * o;
        for (int c = 0; c < CIN; c++)
#pragma unroll
            for (int a2 = 0; a2 < K; a2++)
#pragma unroll
                for (int a1 = 0; a1 < K; a1++) {
                    const float wv = w[a1 + K * (a2 + K * c)];
#pragma unroll
                    for (int j = 0; j < PPL; j++) acc[j] = fmaf(wv, in[c * IC + base[j] - a2 * IP - a1], acc[j]);
                }
#pragma unroll
        for (int j = 0; j < PPL; j++)
            if (live[j]) {
                const int p = lane + 32 * j, y = p / OW, x = p - OW * y;
                out[o * out_cs + y * out_pitch + x + out_off] = fmaxf(acc[j], 0.f);
            }
    }
}

// d loss / d W[a1 + K (a2 + K (c + CIN o))] = sum_{x,y} g(x, y, o) * in[c][y + K-1-a2][x + K-1-a1]; g read from its padded
// array (gp + g_off = position (0,0)).  One task = (input channel c, NO consecutive output channels): K*K*NO accumulators in
// registers; lanes of a warp differ in o, so the input reads are broadcasts.
template <int K, int CIN, int COUT, int OW, int IP, int IC, int GP, int GC, int NO>
__device__ __forceinline__ void conv_backward_weights(const float *gp, int g_off, const float *in, const Row &row, int w_off, int tid) {
    constexpr int OG = COUT / NO;
    for (int task = tid; task < CIN * OG; task += NT) {
        const int og = task % OG, c = task / OG;
        float acc[NO][K * K];
#pragma unroll
        for (int n = 0; n < NO; n++)
#pragma unroll
            for (int t = 0; t < K * K; t++) acc[n][t] = 0.f;
        for (int y = 0; y < OW; y++)
            for (int x = 0; x < OW; x++) {
                float g[NO];
#pragma unroll
                for (int n = 0; n < NO; n++) g[n] = gp[(og * NO + n) * GC + g_off + y * GP + x];
                const float *ip = in + c * IC + (y + K - 1) * IP + (x + K - 1);
#pragma unroll
                for (int a2 = 0; a2 < K; a2++)
#pragma unroll
                    for (int a1 = 0; a1 < K; a1++) {
                        const float v = ip[-a2 * IP - a1];
#pragma unroll
                        for (int n = 0; n < NO; n++) acc[n][a2 * K + a1] = fmaf(g[n], v, acc[n][a2 * K + a1]);
                    }
            }
#pragma unroll
        for (int n = 0; n < NO; n++) {
            const int idx = w_off + K * K * (c + CIN * (og * NO + n));
            if ((K * K) % 4 == 0) {
#pragma unroll
                for (int t = 0; t < K * K; t += 4) {
                    const float v4[4] = {acc[n][t], acc[n][t + 1], acc[n][t + 2], acc[n][t + 3]};
                    emitv<4>(row, idx + t, v4);
                }
            } else {
#pragma unroll
                for (int t = 0; t < K * K; t++) emit1(row, idx + t, acc[n][t]);
            }
        }
    }
}

// bias gradient: sum over the positions of one channel of a (padded) gradient array
template <int C, int OW, int GP, int GC>
__device__ __forceinline__ void bias_grad(const float *gp, int g_off, const Row &row, int b_off, int warp, int lane) {
    for (int o = warp; o < C; o += NW) {
        float s = 0.f;
        for (int p = lane; p < OW * OW; p += 32) s += gp[o * GC + g_off + (p / OW) * GP + (p % OW)];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
        if (lane == 0) emit1(row, b_off + o, s);
    }
}

// conv3 forward, register-tiled: a3(x, y, o) = relu(b3[o] + sum_{c,a2,a1} W3[a1 + 6 (a2 + 6 (c + 32 o))] * a2in[c][y+5-a2][x+5-a1]).
// Thread = (output channel o, quarter of the input channels): all 25 outputs of the channel in registers; per (c, a2) the thread
// reads the 6 weights of ITS channel from the o-fastest copy (the 32 lanes of a warp = 32 consecutive o: one line per load) and
// the five input rows y+5-a2 are warp-uniform shared-memory reads: 150 FMAs per 50 broadcast loads + 6 weights.
// The four quarter sums are added through shared memory.
__device__ __forceinline__ void conv3_forward_tiled(const float *__restrict__ W3of, const float *__restrict__ b3, const float *a2s,
                                                    float *part, float *a3s, int tid) {
    if (tid < 256) {
        const int o = tid & 63, cq = tid >> 6;
        float acc[25];
#pragma unroll
        for (int i = 0; i < 25; i++) acc[i] = 0.f;
        const float *w = W3of + 36 * 64 * (8 * cq) + o;
#pragma unroll 1
        for (int c = 0; c < 8; c++) {
            const float *in = a2s + (8 * cq + c) * 100;
#pragma unroll 3
            for (int a2 = 0; a2 < 6; a2++) {                     // 18 weight loads in flight (all 36 spill the accumulators)
                float wv[6];
#pragma unroll
                for (int a1 = 0; a1 < 6; a1++) wv[a1] = __ldg(w + 64 * (36 * c + 6 * a2 + a1));
#pragma unroll
                for (int y = 0; y < 5; y++) {
                    float row[10];                           // five 8-byte broadcasts (rows are 40 bytes: 8-byte aligned)
#pragma unroll
                    for (int i = 0; i < 5; i++) {
                        const float2 t2 = *reinterpret_cast<const float2 *>(in + (y + 5 - a2) * 10 + 2 * i);
                        row[2 * i] = t2.x; row[2 * i + 1] = t2.y;
                    }
#pragma unroll
                    for (int a1 = 0; a1 < 6; a1++)
#pragma unroll
                        for (int x = 0; x < 5; x++) acc[y * 5 + x] = fmaf(wv[a1], row[x + 5 - a1], acc[y * 5 + x]);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 25; i++) part[i * 256 + tid] = acc[i];        // [position][quarter][o]: conflict-free
    }
    __syncthreads();
    for (int k = tid; k < 1600; k += NT) {
        const int o = k / 25, i = k - 25 * o;
        const float *p = part + i * 256 + o;
        a3s[k] = fmaxf(p[0] + p[64] + p[128] + p[192] + __ldg(b3 + o), 0.f);
    }
}

// conv3 weight gradient, register-tiled: d loss / d W3[a1 + 6 (a2 + 6 (c + 32 o))] = sum_{y,x} g3(x, y, o) a2in[c][y+5-a2][x+5-a1].
// Task = (fifth of the output channels, input channel c, kernel row a2): 5 x 192 = 960 tasks = exactly three rounds of the 320
// threads (one task per (c, a2) left 128 threads idle and the other 192 with 9,600 FMAs each).  The task holds the five input
// rows y+5-a2 (50 values) in registers; per o the 25 gradient values are warp-uniform shared-memory reads (192 = 6 warps, so a
// warp never straddles two fifths): 150 FMAs per 25 loads.  The six a1 of a task are consecutive in theta: 12 bytes per plane
// and o, consecutive tasks are consecutive in memory.
__device__ __forceinline__ void conv3_weight_grad_tiled(const float *g3, const float *a2s, const Row &row, int tid) {
    for (int task = tid; task < 960; task += NT) {
        const int og = task / 192, r = task - 192 * og, c = r / 6, a2 = r - 6 * c;
        const int o0 = 13 * og, o1 = o0 + 13 < 64 ? o0 + 13 : 64;          // 13, 13, 13, 13, 12 output channels
        float in[5][10];
#pragma unroll
        for (int y = 0; y < 5; y++)
#pragma unroll
            for (int i = 0; i < 5; i++) {
                const float2 t2 = *reinterpret_cast<const float2 *>(a2s + c * 100 + (y + 5 - a2) * 10 + 2 * i);
                in[y][2 * i] = t2.x; in[y][2 * i + 1] = t2.y;
            }
        for (int o = o0; o < o1; o++) {
            float acc[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int y = 0; y < 5; y++)
#pragma unroll
                for (int x = 0; x < 5; x++) {
                    const float gv = g3[o * 25 + y * 5 + x];
#pragma unroll
                    for (int a1 = 0; a1 < 6; a1++) acc[a1] = fmaf(gv, in[y][x + 5 - a1], acc[a1]);
                }
            const int idx = O_W3 + 6 * a2 + 36 * (c + 32 * o);            // even: 4-byte aligned in the bf16 planes
            if (row.hi != nullptr) {
#pragma unroll
                for (int j = 0; j < 3; j++) {
                    uint32_t lo;
                    const uint32_t hi = split2(acc[2 * j], acc[2 * j + 1], lo);
                    *reinterpret_cast<uint32_t *>(row.hi + idx + 2 * j) = hi;
                    *reinterpret_cast<uint32_t *>(row.lo + idx + 2 * j) = lo;
                }
            }
            if (row.J != nullptr) {
#pragma unroll
                for (int j = 0; j < 6; j++) row.J[idx + j] = acc[j];
            }
        }
    }
}

// conv3 backward-data without the zero padding: d loss / d a2(u, v, c) = sum_o sum_{y, x} W3[x+5-u, y+5-v, c, o] g3(x, y, o), only
// over the taps that exist (0 <= y+5-v <= 5; x+5-u is always a tap).  Thread = (input channel c, input row v): the ten u of the
// row in registers; per (o, y) five broadcast reads of a g3 row and six weights from the c-fastest copy (the 32 lanes of a warp
// = the 32 input channels: one line per load; from the Flux layout each lane sat in its own line and the load unit, ~32 cycles
// per such instruction, took 178k of a sample's 570k cycles) give 30 FMAs.  Masked by relu'(a2) and stored into the padded
// conv2-gradient plane.
__device__ __forceinline__ void conv3_backward_data_tiled(const float *__restrict__ W3cf, const float *g3, const float *a2s, float *g2p, int tid) {
    const int c = tid & 31, v = tid >> 5;                     // NT = 320: v = 0..9 = the warp index
    float acc[10];
#pragma unroll
    for (int i = 0; i < 10; i++) acc[i] = 0.f;
    const int y_lo = v - 5 > 0 ? v - 5 : 0, y_hi = v < 4 ? v : 4;
    // batches of four output channels, software-pipelined by hand: the 24 weight loads of batch b + 1 are issued before the
    // 120 FMAs of batch b (left to the compiler, every batch waited a full L2 latency: the warps of rows 4 and 5 have 80
    // batches each and everybody else waits for them at the barrier).  Batch b: y = y_lo + b / 16, o = 4 (b % 16) ..+3.
    const int n_b = (y_hi - y_lo + 1) * 16;
    auto load = [&](float (&w)[4][6], int b) {
        const float *p = W3cf + 32 * (36 * 4 * (b & 15) + 6 * (y_lo + (b >> 4) + 5 - v)) + c;
#pragma unroll
        for (int j = 0; j < 4; j++)
#pragma unroll
            for (int a1 = 0; a1 < 6; a1++) w[j][a1] = __ldg(p + 32 * (36 * j + a1));
    };
    auto fma = [&](const float (&w)[4][6], int b) {
        const float *gr = g3 + 100 * (b & 15) + 5 * (y_lo + (b >> 4));
#pragma unroll
        for (int j = 0; j < 4; j++)
#pragma unroll
            for (int x = 0; x < 5; x++) {
                const float gv = gr[25 * j + x];
#pragma unroll
                for (int a1 = 0; a1 < 6; a1++) acc[x + 5 - a1] = fmaf(w[j][a1], gv, acc[x + 5 - a1]);
            }
    };
    float wa[4][6], wb[4][6];
    load(wa, 0);
#pragma unroll 1
    for (int b = 0; b < n_b; b += 2) {
        load(wb, b + 1);
        fma(wa, b);
        load(wa, b + 2 < n_b ? b + 2 : b);                     // the last prefetch re-reads a valid batch and is dropped
        fma(wb, b + 1);
    }
#pragma unroll
    for (int u = 0; u < 10; u++) g2p[c * G2C + (v + 1) * 12 + (u + 1)] = a2s[c * 100 + v * 10 + u] > 0.f ? acc[u] : 0.f;
}

// conv2 forward, register-tiled: a2(x, y, o) = relu(b2[o] + sum_{c,a2,a1} W2[a1 + 3 (a2 + 3 (c + 16 o))] * a1p[c][y+2-a2][x+2-a1]).
// Thread = (pair of output channels, half an output row = 5 positions): 16 x 20 = 320 tasks.  Per (c, a2) seven input values
// (two distinct addresses per warp: broadcasts) and three 8-byte weight loads feed 30 FMAs.
__device__ __forceinline__ void conv2_forward_tiled(const float *w2s, const float *__restrict__ b2, const float *a1p, float *a2s, int tid) {
    const int og = tid & 15, seg = tid >> 4, y = seg >> 1, x0 = (seg & 1) * 5;
    float acc[2][5];
    const float b0 = __ldg(b2 + 2 * og), b1 = __ldg(b2 + 2 * og + 1);
#pragma unroll
    for (int x = 0; x < 5; x++) { acc[0][x] = b0; acc[1][x] = b1; }
#pragma unroll 4
    for (int c = 0; c < 16; c++) {
#pragma unroll
        for (int a2 = 0; a2 < 3; a2++) {
            const float *ip = a1p + c * 144 + (y + 2 - a2) * 12 + x0;
            float in[7];
#pragma unroll
            for (int i = 0; i < 7; i++) in[i] = ip[i];
#pragma unroll
            for (int a1 = 0; a1 < 3; a1++) {
                const float2 w = *reinterpret_cast<const float2 *>(w2s + c * W2C + (3 * a2 + a1) * 32 + 2 * og);
#pragma unroll
                for (int x = 0; x < 5; x++) {
                    acc[0][x] = fmaf(w.x, in[x + 2 - a1], acc[0][x]);
                    acc[1][x] = fmaf(w.y, in[x + 2 - a1], acc[1][x]);
                }
            }
        }
    }
#pragma unroll
    for (int n = 0; n < 2; n++)
#pragma unroll
        for (int x = 0; x < 5; x++) a2s[(2 * og + n) * 100 + y * 10 + x0 + x] = fmaxf(acc[n][x], 0.f);
}

// conv2 backward-data: d loss / d a1(u, v, c) = sum_{o,a2,a1} W2[a1 + 3 (a2 + 3 (c + 16 o))] * g2p[o][v + a2][u + a1] (g2p zero
// padded by 1), masked by relu'(a1).  Thread = (input channel c, half an input row): 16 x 20 = 320 tasks; per (o, a2) seven
// gradient values (broadcasts) and three weights (lanes = 16 channels: 16 banks) feed 15 FMAs.
__device__ __forceinline__ void conv2_backward_data_tiled(const float *w2s, const float *g2p, const float *a1p, float *g1s, int tid) {
    const int c = tid & 15, seg = tid >> 4, v = seg >> 1, u0 = (seg & 1) * 5;
    float acc[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int o = 0; o < 32; o++) {
#pragma unroll
        for (int a2 = 0; a2 < 3; a2++) {
            const float *gp = g2p + o * G2C + (v + a2) * 12 + u0;
            float g[7];
#pragma unroll
            for (int i = 0; i < 7; i++) g[i] = gp[i];
#pragma unroll
            for (int a1 = 0; a1 < 3; a1++) {
                const float w = w2s[c * W2C + (3 * a2 + a1) * 32 + o];
#pragma unroll
                for (int u = 0; u < 5; u++) acc[u] = fmaf(w, g[u + a1], acc[u]);
            }
        }
    }
#pragma unroll
    for (int u = 0; u < 5; u++)
        g1s[c * 100 + v * 10 + u0 + u] = a1p[c * 144 + (v + 1) * 12 + (u0 + u + 1)] > 0.f ? acc[u] : 0.f;
}

// conv2 weight gradient: d loss / d W2[a1 + 3 (a2 + 3 (c + 16 o))] = sum_{y,x} g2(x, y, o) a1p[c][y+2-a2][x+2-a1].
// Thread = (input channel c, pair of output channels): 256 tasks, 18 accumulators.  Per output row the three input rows it
// touches are loaded (9 x 16-byte broadcasts) and slide under the ten positions: 180 FMAs per 29 loads (one scalar load
// per FMA before).  The lanes of a warp differ in the output channel: stride 145 in g2p, no bank conflicts.
__device__ __forceinline__ void conv2_weight_grad_tiled(const float *g2p, const float *a1p, const Row &row, int tid) {
    if (tid >= 256) return;
    const int og = tid & 15, c = tid >> 4;
    float acc[2][9];
#pragma unroll
    for (int n = 0; n < 2; n++)
#pragma unroll
        for (int t = 0; t < 9; t++) acc[n][t] = 0.f;
    for (int y = 0; y < 10; y++) {
        const float *g0 = g2p + (2 * og) * G2C + 13 + y * 12, *g1 = g0 + G2C;
        float ga[10], gb[10];
#pragma unroll
        for (int x = 0; x < 10; x++) { ga[x] = g0[x]; gb[x] = g1[x]; }
#pragma unroll
        for (int a2 = 0; a2 < 3; a2++) {                       // one input row at a time keeps the live set at 12 + 20 + 18 registers
            float in[12];
#pragma unroll
            for (int q4 = 0; q4 < 3; q4++) {
                const float4 t4 = *reinterpret_cast<const float4 *>(a1p + c * 144 + (y + 2 - a2) * 12 + 4 * q4);
                in[4 * q4] = t4.x; in[4 * q4 + 1] = t4.y; in[4 * q4 + 2] = t4.z; in[4 * q4 + 3] = t4.w;
            }
#pragma unroll
            for (int x = 0; x < 10; x++)
#pragma unroll
                for (int a1 = 0; a1 < 3; a1++) {
                    acc[0][3 * a2 + a1] = fmaf(ga[x], in[x + 2 - a1], acc[0][3 * a2 + a1]);
                    acc[1][3 * a2 + a1] = fmaf(gb[x], in[x + 2 - a1], acc[1][3 * a2 + a1]);
                }
        }
    }
#pragma unroll
    for (int n = 0; n < 2; n++)
#pragma unroll
        for (int t = 0; t < 9; t++) emit1(row, O_W2 + 9 * (c + 16 * (2 * og + n)) + t, acc[n][t]);
}

// d loss / d a3[k] = sum_n W4[n + 64 k] gh[n], through relu.  A half warp reads the 64 consecutive weights of one k as 16-byte
// loads (two lines per k; a thread per k had every lane in its own line) and reduces with four shuffles.
__device__ __forceinline__ void dense1_backward_data(const float *__restrict__ W4, const float *gh, const float *a3s, float *g3, int warp, int lane) {
    const int hl = lane & 15, half = lane >> 4;
    const float4 gv = *reinterpret_cast<const float4 *>(gh + 4 * hl);
#pragma unroll 8
    for (int k = 2 * warp + half; k < 1600; k += 2 * NW) {
        const float4 w = __ldg(reinterpret_cast<const float4 *>(W4 + 64 * k) + hl);
        float acc = fmaf(w.x, gv.x, fmaf(w.y, gv.y, fmaf(w.z, gv.z, w.w * gv.w)));
#pragma unroll
        for (int d = 8; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
        if (hl == 0) g3[k] = a3s[k] > 0.f ? acc : 0.f;         // k = o*25 + y*5 + x
    }
}

// -DGRADS_PHASES: CTA 0 prints the cycles of every phase of its second sample (development aid, off in the product build)
#ifdef GRADS_PHASES
#define PHASE(name)                                                                  \
    do {                                                                             \
        __syncthreads();                                                             \
        if (n_ph < 16) { ph_name[n_ph] = name; ph_t[n_ph++] = clock64(); }           \
    } while (0)
#else
#define PHASE(name)
#endif

__global__ void __launch_bounds__(NT, 2) k_sample_grads(const GradArgs a) {
    extern __shared__ float sm[];
    float *xin = sm + S_XIN, *a1p = sm + S_A1, *a2s = sm + S_A2, *a3s = sm + S_A3, *hid = sm + S_HID, *gh = sm + S_GH;
    float *qv = sm + S_Q, *red = sm + S_RED, *g3 = sm + S_G3, *part = sm + S_PART, *g2p = sm + S_G2, *g1s = sm + S_G1;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const float *th = a.theta;
    for (int i = tid; i < S_END; i += NT) sm[i] = 0.f;            // the zero borders of the padded arrays stay zero
    for (int i = tid; i < 288; i += NT) sm[S_W1 + i] = __ldg(th + O_W1 + i);
    for (int i = tid; i < 4608; i += NT) {                        // theta index a1 + 3 (a2 + 3 (c + 16 o)) -> [c][tap][o]
        const int tap = i % 9, c = (i / 9) % 16, o = i / 144;
        sm[S_W2 + c * W2C + tap * 32 + o] = __ldg(th + O_W2 + i);
    }
#ifdef GRADS_PHASES
    long long ph_t[16], t_phase = 0;
    const char *ph_name[16];
    int n_ph = 0;
#endif
    for (long long s = blockIdx.x; s < a.B; s += gridDim.x) {
        __syncthreads();
#ifdef GRADS_PHASES
        t_phase = clock64();
        n_ph = 0;
#endif
        Row row;
        row.hi = a.hi != nullptr ? a.hi + s * a.pitch : nullptr;
        row.lo = a.lo != nullptr ? a.lo + s * a.pitch : nullptr;
        row.J = a.J != nullptr ? a.J + s * a.ldJ : nullptr;
        // ---------------- forward (structs.jl:127-139) ----------------
        for (int i = tid; i < 200; i += NT) {
            const int c = i / 100, p = i - 100 * c, y = p / 10, x = p - 10 * y;
            xin[c * 144 + (y + 1) * 12 + (x + 1)] = a.states[s * 200 + i];
        }
        __syncthreads();
        conv_forward<3, 2, 16, 10, 12, 144, 4>(sm + S_W1, th + O_B1, xin, a1p, 12, 144, 13, warp, lane);
        __syncthreads();
        PHASE("load + conv1 fwd");
        conv2_forward_tiled(sm + S_W2, th + O_B2, a1p, a2s, tid);
        __syncthreads();
        PHASE("conv2 fwd");
        conv3_forward_tiled(th + O_W3OF, th + O_B3, a2s, part, a3s, tid);
        __syncthreads();
        PHASE("conv3 fwd");
        {   // Dense(1600, 64, relu): thread = (n, fifth of k); two interleaved chains so that 16 coalesced loads are in flight
            const int n = tid & 63, kq = tid >> 6;
            float acc0 = 0.f, acc1 = 0.f;
#pragma unroll 8
            for (int k = kq * 320; k < kq * 320 + 320; k += 2) {
                acc0 = fmaf(__ldg(th + O_W4 + n + 64 * k), a3s[k], acc0);
                acc1 = fmaf(__ldg(th + O_W4 + n + 64 * (k + 1)), a3s[k + 1], acc1);
            }
            red[tid] = acc0 + acc1;
            __syncthreads();
            if (tid < 64)
                hid[tid] = fmaxf(red[tid] + red[tid + 64] + red[tid + 128] + red[tid + 192] + red[tid + 256] + __ldg(th + O_B4 + tid), 0.f);
            __syncthreads();
        }
        PHASE("dense 1600x64 fwd");
        const int act = a.actions[s] < 3 ? a.actions[s] : 0;
        if (warp == 0) {   // Dense(64, 3), Huber loss (delta = 1) on the selected action (utils.jl:452-458)
            float q3[3];
#pragma unroll
            for (int k = 0; k < 3; k++) {
                float p = fmaf(__ldg(th + O_W5 + k + 3 * lane), hid[lane], 0.f) + fmaf(__ldg(th + O_W5 + k + 3 * (lane + 32)), hid[lane + 32], 0.f);
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) p += __shfl_xor_sync(0xffffffffu, p, d);
                q3[k] = p + __ldg(th + O_B5 + k);
            }
            if (lane == 0) {
                // q_target is Float64 in the reference (the 0.97 literal promotes, utils.jl:451), so the loss is evaluated in
                // Float64 and its gradient projected back to the Float32 of q_pred
                const double d = (double)q3[act] - a.targets[s];
                const double ad = fabs(d);
                qv[0] = q3[0]; qv[1] = q3[1]; qv[2] = q3[2];
                qv[3] = (float)(ad < 1.0 ? d : copysign(1.0, d));          // d huber / d q_sel
                if (a.loss != nullptr) a.loss[s] = (float)(ad < 1.0 ? 0.5 * d * d : ad - 0.5);
            }
        }
        __syncthreads();
        // ---------------- backward ----------------
        PHASE("head + loss");
        const float g = qv[3];
        if (tid < 192) emit1(row, O_W5 + tid, (tid % 3) == act ? g * hid[tid / 3] : 0.f);       // W5 is (3,64) column-major
        if (tid < 3) emit1(row, O_B5 + tid, tid == act ? g : 0.f);
        if (tid >= 192 && tid < 192 + 45 && NP + (tid - 192) < a.pitch && row.hi != nullptr) {   // padding columns of the planes
            row.hi[NP + tid - 192] = __float2bfloat16_rn(0.f);
            row.lo[NP + tid - 192] = __float2bfloat16_rn(0.f);
        }
        if (tid < 64) {
            const float v = hid[tid] > 0.f ? __ldg(th + O_W5 + act + 3 * tid) * g : 0.f;
            gh[tid] = v;
            emit1(row, O_B4 + tid, v);
        }
        __syncthreads();
        // grad W4[n + 64 k] = gh[n] a3[k]: 8 consecutive n per store
        for (int i = tid; i < 1600 * 8; i += NT) {
            const int k = i >> 3, n0 = (i & 7) * 8;
            const float ak = a3s[k];
            float v8[8];
#pragma unroll
            for (int j = 0; j < 8; j++) v8[j] = gh[n0 + j] * ak;
            emitv<8>(row, O_W4 + n0 + 64 * k, v8);
        }
        PHASE("W4 grad emit");
        dense1_backward_data(th + O_W4, gh, a3s, g3, warp, lane);
        __syncthreads();
        PHASE("d a3");
        bias_grad<64, 5, 5, 25>(g3, 0, row, O_B3, warp, lane);
        PHASE("b3 grad");
        conv3_weight_grad_tiled(g3, a2s, row, tid);
        PHASE("conv3 weight grad");
        conv3_backward_data_tiled(th + O_W3CF, g3, a2s, g2p, tid);
        __syncthreads();
        PHASE("conv3 bwd data");
        bias_grad<32, 10, 12, G2C>(g2p, 13, row, O_B2, warp, lane);
        conv2_weight_grad_tiled(g2p, a1p, row, tid);
        PHASE("conv2 weight grad + b2");
        conv2_backward_data_tiled(sm + S_W2, g2p, a1p, g1s, tid);
        __syncthreads();
        PHASE("conv2 bwd data");
        bias_grad<16, 10, 10, 100>(g1s, 0, row, O_B1, warp, lane);
        conv_backward_weights<3, 2, 16, 10, 12, 144, 10, 100, 1>(g1s, 0, xin, row, O_W1, tid);
        PHASE("conv1 weight grad + b1");
#ifdef GRADS_PHASES
        if (blockIdx.x == 0 && tid == 0 && s == (long long)gridDim.x) {
            for (int i = 0; i < n_ph; i++) printf("%-28s %8lld\n", ph_name[i], ph_t[i] - (i ? ph_t[i - 1] : t_phase));
            printf("%-28s %8lld\n", "sample total", ph_t[n_ph - 1] - t_phase);
        }
#endif
    }
}

// loads k_sample_grads now: module loading is lazy, and a first launch behind a kernel that spins on a peer would wait for it
int preload_sample_grads() {
    cudaFuncAttributes fa;
    SNK_CUDA(cudaFuncGetAttributes(&fa, k_sample_grads));
    return SNK_OK;
}
int launch_sample_grads(const float *theta_dev, const float *states, const uint8_t *actions, const double *targets, long long B,
                        void *hi, void *lo, long long pitch, float *J, long long ldJ, float *loss, int sms, cudaStream_t st) {
    GradArgs a;
    a.theta = theta_dev; a.states = states; a.actions = actions; a.targets = targets; a.B = B;
    a.hi = (__nv_bfloat16 *)hi; a.lo = (__nv_bfloat16 *)lo; a.pitch = pitch; a.J = J; a.ldJ = ldJ; a.loss = loss;
    SNK_CUDA(cudaFuncSetAttribute(k_sample_grads, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    const long long max_grid = 2ll * sms;                    // 2 CTAs of 88 KB (and <= 102 registers x 320 threads) per SM
    const int grid = (int)(B < max_grid ? B : max_grid);
    k_sample_grads<<<grid, NT, SMEM_BYTES, st>>>(a);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

}  // namespace qgrad
}  // namespace snk
