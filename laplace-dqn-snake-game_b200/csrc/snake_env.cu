// snake_env.cu — batched Snake environment for B200 (sm_100a): kernels + C ABI.
//
// Replaces, for N independent envs at once, the reference's per-game Julia methods
// (lucagiorgetti/Laplace-DQN-Snake-game):
//   structs.jl:33-99   SnakeGame()            -> k_reset / auto-reset in k_step
//   utils.jl:7-10      available_actions      -> av_dir(), k_available_actions
//   utils.jl:13-40     sample_food!           -> food_search()
//   utils.jl:43-109    update_board!/check_collision/grow_maybe!/move_wrapper!/step! -> env_step()
//   utils.jl:112-132   virtual_step           -> losing_mask3()
//   utils.jl:135-149   assemble_state(s)      -> board planes + expand_obs()
//   utils.jl:153-172   epsilon_greedy         -> select_idx()
//   utils.jl:448-451   masked max-Q target    -> k_masked_target
//
// Design (see DESIGN.md): the game state is struct-of-arrays, 52 B/env:
//   occ   u64  snake occupancy of the 8x8 interior, bit = (r-1) + 8(c-1)   (r,c 0-based board coords)
//   pocc  u64  the same for the previous board (frame 1 of the two-frame state)
//   clo/chi    128-bit chain of 2-bit directions, entry j = move that took segment j+1 to segment j
//   cons  u64  which food_list entries have been used ("deleteat!") this episode
//   misc  u64  head, tail, food, previous food (4-bit r,c each), prev_dir, length, step count, done, error bits
//   ret   f32  running episode reward
// One thread steps one env with bit-board arithmetic (phase A, coalesced 8-byte loads/stores), drops two
// 100-cell boards as 2 bit-planes into shared memory, and then the whole CTA streams the (10,10,2,N)
// observation out as fully coalesced 16-byte stores through a 256-entry nibble->float4 table (phase B).
#include <stdarg.h>
#include <string.h>

#include <new>
#include <mutex>
#include <type_traits>
#include <unordered_map>

#include <cuda.h>

#include "common.h"
#include "sm100.h"

// how phase B stores the observation: 0 = st.global.cs (streaming), 1 = plain st.global (default), 2 = st.global.wt.
// Measured at 2^20 envs on B200: 166.5 us with .cs, 162.8 us with plain or .wt stores (87.4 % of the HBM copy peak); into
// compressible outputs (snk_device_alloc) 118.0 / 117.8 / 117.8 us.
#ifndef SNK_OBS_STORE_MODE
#define SNK_OBS_STORE_MODE 1
#endif
#if SNK_OBS_STORE_MODE == 1
#define SNK_OBS_STORE(p, v) (*(p) = (v))
#elif SNK_OBS_STORE_MODE == 2
#define SNK_OBS_STORE(p, v) __stwt((p), (v))
#else
#define SNK_OBS_STORE(p, v) __stcs((p), (v))
#endif

namespace snk {

static thread_local char g_err[512];
char *err_buf() { return g_err; }
int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

// ------------------------------------------------------------------------------------------------
#ifndef SNK_TPB
#define SNK_TPB 256            // measured on B200 at 2^20 envs into plain memory: 256 threads ~1-2 % faster than 128, 64 and 512 slower
                               // (Float32 into compressible outputs at unroll 2: 128 threads 114.7 us, 256 117.8; not adopted, the
                               // small formats' occupancy also depends on it and they were not re-measured)
#endif
#ifndef SNK_MINB
#define SNK_MINB 1
#endif
#ifndef SNK_UNROLL
#define SNK_UNROLL 4           // Float32 phase B into compressible outputs, 2^20 envs on B200: 1 / 2 / 4 -> 123.9 / 117.8 / 115.1 us;
                               // into plain memory 151.1 / 150.4 / 150.2 us.  Against unroll 2 (bench.py, with compressible outputs):
                               // config 2 at 4,096 envs 4.96 -> 4.98 G env-steps/s, the host-buffer Float32 step (e2e
                               // full_f32_obs_variant) 6.81 -> 6.82e7; the rollout kernels pass their own unroll (5); the
                               // stand-alone state kernel (snk_state) was not timed
#endif
constexpr int PHASE_B_UNROLL = SNK_UNROLL;
constexpr int TPB = SNK_TPB;      // envs (= threads) per CTA (tuning knobs: -DSNK_TPB / -DSNK_MINB / -DSNK_UNROLL)
constexpr int MAX_FOOD = 64;
constexpr int PLANE_WORDS = 16;   // per env in smem: [frame 0/1][plane 0/1][4 x u32]

// misc field layout
constexpr int M_HR = 0, M_HC = 4, M_TR = 8, M_TC = 12, M_FR = 16, M_FC = 20, M_PFR = 24, M_PFC = 28;
constexpr int M_PD = 32, M_LEN = 34, M_T = 41, M_DONE = 51, M_ERR = 52;

// walls of the 10x10 board in full-board bit space k = r + 10 c
constexpr u64 wall_bits(int lo_hi) {
    u64 lo = 0, hi = 0;
    for (int c = 0; c < 10; c++)
        for (int r = 0; r < 10; r++)
            if (r == 0 || r == 9 || c == 0 || c == 9) {
                int k = r + 10 * c;
                if (k < 64) lo |= 1ull << k; else hi |= 1ull << (k - 64);
            }
    return lo_hi ? hi : lo;
}
constexpr u64 WALL_LO = wall_bits(0), WALL_HI = wall_bits(1);

// R1 initial state (structs.jl:37-66): snake [(8,2),(9,2)] 1-based = head (7,1), tail (8,1) 0-based, food (4,5) -> (3,4)
constexpr u64 INIT_OCC = (1ull << (6 + 0)) | (1ull << (7 + 0));
constexpr u64 INIT_MISC = (7ull << M_HR) | (1ull << M_HC) | (8ull << M_TR) | (1ull << M_TC) | (3ull << M_FR) |
                          (4ull << M_FC) | (3ull << M_PFR) | (4ull << M_PFC) | (0ull << M_PD) | (2ull << M_LEN);

struct FoodTable {
    uint8_t bit[MAX_FOOD];   // interior bit index of list entry i
    int n;
    __host__ __device__ u64 mask() const { return n >= 64 ? ~0ull : ((1ull << n) - 1ull); }   // the entries of the list
};

struct EnvState {
    u64 *occ, *pocc, *clo, *chi, *cons, *misc;
    float *ret;
};

// bytes of one env's observation; 0 for SNK_OBS_NONE and unknown formats
__host__ __device__ constexpr int obs_bytes(int fmt) {
    switch (fmt) {
        case SNK_OBS_F32: return 800;
        case SNK_OBS_I8: return 200;
        case SNK_OBS_I64: return 1600;
        case SNK_OBS_PACKED2: return 50;
        case SNK_OBS_BITS: return 24;
        default: return 0;
    }
}

// the per-step outputs of the step and rollout kernels, any of them NULL
struct StepOutputs {
    float *reward;
    uint8_t *done;
    void *obs;
    uint8_t *mask;
    float *ep_return;
    int32_t *ep_score;
};

struct StepArgs {
    EnvState s;
    const uint8_t *act;      // input action (idx or abs dir) when !SELECT
    const float *q;          // (3,N) when SELECT
    const float *u;          // (N) or NULL
    const uint8_t *ridx;     // (N) or NULL
    float eps;
    uint8_t *act_out;
    StepOutputs out;
    long long env_begin, env_end;
    u64 seed, step_counter;
    int auto_reset, is_abs;
    // transition sink = replay ring (store!, utils.jl:267-277): one 128-byte record per env per step
    uint4 *sink;
    long long sink_base, sink_cap, sink_n;   // transitions stored before this step; ring capacity; envs in this step
    FoodTable food;
};

// 128-byte transition record (one cache line): three boards as 2 x 128-bit planes each, then the scalars
//   [0,32) board_{t-2}  [32,64) board_{t-1}  [64,96) board_t      state = (b_{t-2}, b_{t-1}), next_state = (b_{t-1}, b_t)
//   [96] reward f32 | [100] action idx u8 | [101] done u8 | [102] next_is_suicidal bits u8 | [103] prev_dir at action time u8
//   [104] episode return f32 | [108] score i32 | [112] env id u32 | [116] step-in-episode u16
constexpr int REC_U4 = 8;

// ------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ u64 splitmix64(u64 x) {
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}

__device__ __forceinline__ void dir_delta(int d, int &dr, int &dc) {   // utils.jl:8 order U D L R
    int s = (d & 1) ? 1 : -1;
    dr = (d & 2) ? 0 : s;
    dc = (d & 2) ? s : 0;
}
// available_actions (utils.jl:7-10): [U,D,L,R] minus the reverse of prev_dir, order kept
__device__ __forceinline__ int av_dir(int prev_dir, int idx) { return idx + (idx >= (prev_dir ^ 1) ? 1 : 0); }

__device__ __forceinline__ int chain_get(u64 lo, u64 hi, int i) {
    int pos = 2 * i;
    return (int)(((pos < 64) ? (lo >> pos) : (hi >> (pos - 64))) & 3ull);
}

// sample_food! (utils.jl:13-40): first not-yet-used list entry whose cell is empty on the pre-update board.
// blocked = cells that are not 0 there (old snake incl. tail, and the eaten food cell).  Returns the list
// index or -1 (BoundsError in the reference), -2 when no cell is empty at all (utils.jl:18-21).
__device__ __forceinline__ int food_search(u64 blocked, u64 cons, u64 list_mask, const uint8_t *s_food_bit) {
    if (~blocked == 0ull) return -2;
    u64 cand = ~cons & list_mask;
    while (cand) {
        int i = __ffsll((long long)cand) - 1;
        if (!((blocked >> s_food_bit[i]) & 1ull)) return i;
        cand &= cand - 1;
    }
    return -1;
}

// Julia argmax over 3 Float32 (findmax with isless: first maximum, NaN largest, -0.0 < 0.0)
__device__ __forceinline__ bool jl_isless(float a, float b) {
    if (a != a) return false;
    if (b != b) return true;
    if (a < b) return true;
    if (a == b) return (__float_as_uint(a) >> 31) && !(__float_as_uint(b) >> 31);
    return false;
}
__device__ __forceinline__ int select_idx(float q0, float q1, float q2, float eps, float u, int ridx) {
    if (u < eps) return ridx;
    int best = 0;
    float qb = q0;
    if (jl_isless(qb, q1)) { best = 1; qb = q1; }
    if (jl_isless(qb, q2)) { best = 2; }
    return best;
}
__device__ __forceinline__ void internal_draw(u64 seed, u64 step, long long env, float &u, int &ridx) {
    u64 x = splitmix64(seed ^ splitmix64((u64)env * 0x100000001B3ull + step));
    u = (float)(x >> 40) * 5.9604644775390625e-08f;   // 24 bits -> [0,1)
    ridx = (int)((x & 0xFFFFFFull) % 3ull);
}

// 8x8 interior bitmap -> 10x10 full-board bit space (k = r + 10c = b + 2(c-1) + 11)
__device__ __forceinline__ void to_full(u64 occ, u64 &lo, u64 &hi) {
    u64 b0 = occ & 0xFF, b1 = (occ >> 8) & 0xFF, b2 = (occ >> 16) & 0xFF, b3 = (occ >> 24) & 0xFF;
    u64 b4 = (occ >> 32) & 0xFF, b5 = (occ >> 40) & 0xFF, b6 = (occ >> 48) & 0xFF, b7 = occ >> 56;
    lo = (b0 << 11) | (b1 << 21) | (b2 << 31) | (b3 << 41) | (b4 << 51) | (b5 << 61);
    hi = (b5 >> 3) | (b6 << 7) | (b7 << 17);
}
__device__ __forceinline__ void set_k(int r, int c, u64 &lo, u64 &hi) {
    int k = r + 10 * c;
    u64 b = 1ull << (k & 63);
    if (k < 64) lo |= b; else hi |= b;
}
// Two bit-planes of one board in full-board bit space (cells 0..63 in lo, 64..99 in hi), code = 2*p1 + p0: 0 empty, 1 snake,
// 2 food, 3 wall.  The head is drawn last as snake, which reproduces update_board! overwriting the wall cell on a wall death
// (utils.jl:48-50).
__device__ __forceinline__ void board_bits(u64 occ, int fr, int fc, bool has_head, int hr, int hc, u64 &p0lo, u64 &p0hi,
                                           u64 &p1lo, u64 &p1hi) {
    u64 slo, shi;
    to_full(occ, slo, shi);
    if (has_head) set_k(hr, hc, slo, shi);
    u64 flo = WALL_LO, fhi = WALL_HI;
    if (fr != 0) set_k(fr, fc, flo, fhi);
    p0lo = slo | WALL_LO; p0hi = shi | WALL_HI;
    p1lo = flo & ~slo; p1hi = fhi & ~shi;
}
// nibble i of x -> byte i of the result (low nibble of each byte)
__device__ __forceinline__ u64 spread_nibbles(uint32_t x) {
    u64 v = x;
    v = (v | (v << 16)) & 0x0000FFFF0000FFFFull;
    v = (v | (v << 8)) & 0x00FF00FF00FF00FFull;
    v = (v | (v << 4)) & 0x0F0F0F0F0F0F0F0Full;
    return v;
}
// byte i of the result = nibble i of p0 | nibble i of p1 << 4  (8 unit bytes from 32 cells of both planes).  Even and odd
// nibbles are separated with two masks each and interleaved by two byte permutes: 6 instructions — the shift-and-mask
// spreading of each plane through a 64-bit word took 36, and the board conversion was the longest chain of a step's consumers.
__device__ __forceinline__ u64 unit_bytes(uint32_t p0, uint32_t p1) {
    const uint32_t ev = (p0 & 0x0F0F0F0Fu) | ((p1 << 4) & 0xF0F0F0F0u);      // byte k: nibbles 2k of both planes
    const uint32_t od = ((p0 >> 4) & 0x0F0F0F0Fu) | (p1 & 0xF0F0F0F0u);      // byte k: nibbles 2k+1
    return (u64)__byte_perm(ev, od, 0x5140) | ((u64)__byte_perm(ev, od, 0x7362) << 32);
}
// PERM = false keeps the shift-and-mask form: the fused step with Float32 / Int64 observations is bound by its stores, and there
// the SHORTER conversion measured 0.9 % slower in an A/B on one box (0.929 -> 0.921 of the HBM peak, three runs each); every
// other kernel gains (int8 step 0.73 -> 0.75, 4,096-env rollout 0.87 -> 0.80 us per step).
template <bool PERM>
__device__ __forceinline__ u64 unit_word(uint32_t p0, uint32_t p1) {
    return PERM ? unit_bytes(p0, p1) : (spread_nibbles(p0) | (spread_nibbles(p1) << 4));
}
// One board -> 25 "unit bytes" in shared memory (32-byte slot): unit q covers cells 4q..4q+3, its byte holds the
// plane-0 nibble in bits 0-3 and the plane-1 nibble in bits 4-7 — exactly the index of the 256-entry output tables,
// so phase B needs one byte load per 16-byte store.
template <bool PERM = true>
__device__ __forceinline__ void board_planes(u64 occ, int fr, int fc, bool has_head, int hr, int hc, uint32_t *dst) {
    u64 p0lo, p0hi, p1lo, p1hi;
    board_bits(occ, fr, fc, has_head, hr, hc, p0lo, p0hi, p1lo, p1hi);
    u64 *d = reinterpret_cast<u64 *>(dst);
    d[0] = unit_word<PERM>((uint32_t)p0lo, (uint32_t)p1lo);
    d[1] = unit_word<PERM>((uint32_t)(p0lo >> 32), (uint32_t)(p1lo >> 32));
    d[2] = unit_word<PERM>((uint32_t)p0hi, (uint32_t)p1hi);
    d[3] = unit_word<PERM>((uint32_t)(p0hi >> 32), (uint32_t)(p1hi >> 32));
}
// the same board as two 16-byte plane vectors (the transition record)
__device__ __forceinline__ void board_planes_reg(u64 occ, int fr, int fc, bool has_head, int hr, int hc, uint4 &a, uint4 &b) {
    u64 p0lo, p0hi, p1lo, p1hi;
    board_bits(occ, fr, fc, has_head, hr, hc, p0lo, p0hi, p1lo, p1hi);
    a = make_uint4((uint32_t)p0lo, (uint32_t)(p0lo >> 32), (uint32_t)p0hi, (uint32_t)(p0hi >> 32));
    b = make_uint4((uint32_t)p1lo, (uint32_t)(p1lo >> 32), (uint32_t)p1hi, (uint32_t)(p1hi >> 32));
}

__device__ __forceinline__ int cell_code(const uint32_t *pl, int k) {     // pl = one board's 32-byte unit slot
    const uint32_t b = reinterpret_cast<const uint8_t *>(pl)[k >> 2];
    const int j = k & 3;
    return (int)(((b >> j) & 1u) | (((b >> (4 + j)) & 1u) << 1));
}
__device__ __forceinline__ int code_value(int code) { return code == 3 ? -1 : code; }

// ------------------------------------------------------------------------------------------------
// Phase B: the CTA streams n_local envs' two boards out of shared memory in the requested format.
// The CTA's output region is contiguous (envs env0 .. env0+n_local-1), so unit j of the region is
// stored by thread j % TPB: every warp-wide store covers one contiguous 512-byte (f32) span.
struct ObsTables {
    float4 f32[256];         // (n1<<4 | n0) -> 4 cells as Float32
};
template <int OBS>
__device__ __forceinline__ void fill_tables(ObsTables &tb, int tid, int nt = TPB) {
    if (OBS == SNK_OBS_F32 || OBS == SNK_OBS_I8 || OBS == SNK_OBS_PACKED2) {
        for (int i = tid; i < 256; i += nt) {
            int n0 = i & 15, n1 = i >> 4;
            float v[4];
            uint32_t bytes = 0, packed = 0;
            for (int j = 0; j < 4; j++) {
                int code = ((n0 >> j) & 1) | (((n1 >> j) & 1) << 1);
                v[j] = (float)code_value(code);
                bytes |= (uint32_t)(uint8_t)(int8_t)code_value(code) << (8 * j);
                packed |= (uint32_t)code << (2 * j);
            }
            if (OBS == SNK_OBS_F32) tb.f32[i] = make_float4(v[0], v[1], v[2], v[3]);
            else if (OBS == SNK_OBS_I8) reinterpret_cast<uint32_t *>(tb.f32)[i] = bytes;
            else reinterpret_cast<uint8_t *>(tb.f32)[i] = (uint8_t)packed;
        }
    }
}

template <bool STREAM, typename T>
__device__ __forceinline__ void obs_store(T *p, const T &v) {
    if (STREAM) __stcs(p, v); else SNK_OBS_STORE(p, v);
}
// unit q (0..49) of env e -> its byte in the shared-memory planes = index of the output tables
__device__ __forceinline__ uint32_t unit_index(const uint32_t *s_planes, int j) {
    const int e = (int)(((unsigned)j * 5243u) >> 18);     // j / 50 for j < 2^15
    const int qq = j - e * 50;
    const int f = qq >= 25;
    return reinterpret_cast<const uint8_t *>(s_planes)[e * (PLANE_WORDS * 4) + f * 32 + (qq - 25 * f)];
}
template <int OBS, int NT = TPB, int UNROLL = PHASE_B_UNROLL, bool STREAM = false>
__device__ __forceinline__ void expand_obs(void *obs, long long env0, int n_local, const uint32_t *s_planes,
                                           const ObsTables &tb, int tid) {
    if (OBS == SNK_OBS_F32) {
        // unit = 4 consecutive cells = one nibble of each plane; 50 units per env; one 16-byte store per unit, unit j of the CTA's
        // region by thread j % NT.  (A division-free mapping — thread = fixed unit of every fifth env — measured 1.6 % slower
        // here: this format is HBM-bound and the independent iterations of this loop keep more stores in flight.)
        const int total = n_local * 50;
        float4 *o32 = reinterpret_cast<float4 *>(obs) + env0 * 50;
#pragma unroll UNROLL
        for (int j = tid; j < total; j += NT) obs_store<STREAM>(o32 + j, tb.f32[unit_index(s_planes, j)]);
    } else if (OBS == SNK_OBS_I8) {
        // int8 observations are bound by instruction issue, not by HBM: one thread gathers 4 units = 16 output bytes and stores
        // one uint4.  Two envs are 25 such vectors; thread t < GP*25 owns vector t % 25 of env pair t / 25 of every group of
        // GP pairs, with its four byte offsets computed once.
        constexpr int GP = NT / 25;                                // env pairs per pass (10 at 256 threads)
        uint8_t *base = reinterpret_cast<uint8_t *>(obs) + env0 * 200;
        const int n_pairs = (NT % 25 > 10) ? 0 : n_local >> 1;   // (see above; then everything goes through the per-unit loop below)
        if ((reinterpret_cast<uintptr_t>(base) & 15u) == 0) {
            if (tid < GP * 25) {
                const int p0 = tid / 25, w = tid - 25 * p0;
                int off[4];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const int uu = 4 * w + k, e2 = uu >= 50, qq = uu - 50 * e2;
                    off[k] = e2 * (PLANE_WORDS * 4) + (qq >= 25 ? 7 : 0) + qq;
                }
                const uint8_t *src = reinterpret_cast<const uint8_t *>(s_planes) + p0 * (2 * PLANE_WORDS * 4);
                const uint32_t *t32 = reinterpret_cast<const uint32_t *>(tb.f32);
                uint4 *o = reinterpret_cast<uint4 *>(base);
#pragma unroll 2
                for (int p = p0; p < n_pairs; p += GP, src += GP * (2 * PLANE_WORDS * 4))
                    obs_store<STREAM>(o + p * 25 + w, make_uint4(t32[src[off[0]]], t32[src[off[1]]], t32[src[off[2]]], t32[src[off[3]]]));
            }
        }
        // an odd last env, or a region that is not 16-byte aligned: one unit per store
        const int done_units = (reinterpret_cast<uintptr_t>(base) & 15u) == 0 ? n_pairs * 100 : 0;
        for (int j = done_units + tid; j < n_local * 50; j += NT)
            reinterpret_cast<uint32_t *>(base)[j] = reinterpret_cast<const uint32_t *>(tb.f32)[unit_index(s_planes, j)];
    } else if (OBS == SNK_OBS_PACKED2) {
        // 2-bit codes: 16 units per 16-byte vector; the CTA's output region is one contiguous byte range
        uint8_t *base = reinterpret_cast<uint8_t *>(obs) + env0 * 50;
        const int total = n_local * 50;
        int done_units = 0;
        if ((reinterpret_cast<uintptr_t>(base) & 15u) == 0) {
            const int nvec = total / 16;
            uint4 *o = reinterpret_cast<uint4 *>(base);
#pragma unroll 2
            for (int v = tid; v < nvec; v += NT) {
                uint32_t w[4];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    uint32_t x = 0;
#pragma unroll
                    for (int b = 0; b < 4; b++)
                        x |= (uint32_t)reinterpret_cast<const uint8_t *>(tb.f32)[unit_index(s_planes, v * 16 + k * 4 + b)] << (8 * b);
                    w[k] = x;
                }
                obs_store<STREAM>(o + v, make_uint4(w[0], w[1], w[2], w[3]));
            }
            done_units = nvec * 16;
        }
        for (int j = done_units + tid; j < total; j += NT) base[j] = reinterpret_cast<const uint8_t *>(tb.f32)[unit_index(s_planes, j)];
    } else if (OBS == SNK_OBS_I64) {
        // unit = 2 consecutive cells (16 bytes); 100 units per env
        const int total = n_local * 100;
        longlong2 *o = reinterpret_cast<longlong2 *>(obs) + env0 * 100;
        for (int j = tid; j < total; j += NT) {
            int e = j / 100;
            int p = j - e * 100;
            int f = p >= 50;
            int k = 2 * (p - 50 * f);
            const uint32_t *pl = s_planes + e * PLANE_WORDS + f * 8;
            longlong2 v;
            v.x = code_value(cell_code(pl, k));
            v.y = code_value(cell_code(pl, k + 1));
            obs_store<STREAM>(o + j, v);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// losing mask of a live state (virtual_step, utils.jl:112-132), closed form:
// action k loses iff it hits a wall, or hits the body after the conditional tail pop, or the
// history-length rule fires (t >= 499 steps already taken).  A virtual eat runs sample_food! on the
// copy, which can raise the reference's BoundsError -> error bit.
__device__ __forceinline__ uint32_t losing_mask3(u64 occ, u64 cons, int hr, int hc, int tr, int tc, int fr, int fc,
                                                 int pd, int t, u64 list_mask, const uint8_t *s_food_bit, int &err) {
    const bool cap = t >= 499;
    const u64 occ_nt = occ & ~(1ull << ((tr - 1) + 8 * (tc - 1)));
    uint32_t m = 0;
#pragma unroll
    for (int k = 0; k < 3; k++) {
        int d = av_dir(pd, k), dr, dc;
        dir_delta(d, dr, dc);
        int nr = hr + dr, nc = hc + dc;
        bool lose;
        if (nr == 0 || nr == 9 || nc == 0 || nc == 9) {
            lose = true;
        } else {
            int b = (nr - 1) + 8 * (nc - 1);
            if (fr != 0 && nr == fr && nc == fc) {
                lose = cap;
                if (food_search(occ | (1ull << b), cons, list_mask, s_food_bit) == -1) err |= SNK_ENV_ERR_FOOD;
            } else {
                lose = cap || ((occ_nt >> b) & 1ull);
            }
        }
        m |= (lose ? 1u : 0u) << k;
    }
    return m;
}

// next_is_suicidal bits m3 as 3 bytes
__device__ __forceinline__ void store_mask3(uint8_t *m, uint32_t m3) {
    m[0] = (uint8_t)(m3 & 1u); m[1] = (uint8_t)((m3 >> 1) & 1u); m[2] = (uint8_t)((m3 >> 2) & 1u);
}
// the scalar outputs of env i's step (row i of a step's outputs)
__device__ __forceinline__ void store_step_outputs(const StepOutputs &o, long long i, float reward, int done, uint32_t m3, float ret,
                                                   int score) {
    if (o.reward != nullptr) o.reward[i] = reward;
    if (o.done != nullptr) o.done[i] = (uint8_t)done;
    if (o.mask != nullptr) store_mask3(o.mask + 3 * i, m3);
    if (o.ep_return != nullptr) o.ep_return[i] = ret;
    if (o.ep_score != nullptr) o.ep_score[i] = score;
}

// ---- one env in registers ---------------------------------------------------------------------------
constexpr int CHI_FROM_LEN = 32;          // see env_load
struct Env {
    u64 occ, pocc, clo, chi, cons;
    float ret;
    int hr, hc, tr, tc, fr, fc, pfr, pfc, pd, len, t, dn, err;
};
// POCC_ALWAYS = false: the previous board is only read for an env that is frozen (done, no auto-reset) — a live env overwrites
// it with the current board before anything looks at it (env_advance), so the 8 bytes are not fetched for it
// CHI_LAZY = true: the second word of the direction chain (entries 32..63) only carries live entries for a snake of 34 or more
// segments, and an entry that is live when it crosses from clo into chi does so at length >= 33: the word is fetched (and,
// see env_store, written back) only from length 32 on.  Below that its content in memory is never looked at by anybody.
__device__ __forceinline__ void env_unpack(Env &e, u64 misc) {
    e.hr = (int)(misc >> M_HR) & 15; e.hc = (int)(misc >> M_HC) & 15;
    e.tr = (int)(misc >> M_TR) & 15; e.tc = (int)(misc >> M_TC) & 15;
    e.fr = (int)(misc >> M_FR) & 15; e.fc = (int)(misc >> M_FC) & 15;
    e.pfr = (int)(misc >> M_PFR) & 15; e.pfc = (int)(misc >> M_PFC) & 15;
    e.pd = (int)(misc >> M_PD) & 3; e.len = (int)(misc >> M_LEN) & 127; e.t = (int)(misc >> M_T) & 1023;
    e.dn = (int)(misc >> M_DONE) & 1; e.err = (int)(misc >> M_ERR) & 15;
}
template <bool POCC_ALWAYS = true, bool CHI_LAZY = false>
__device__ __forceinline__ void env_load(Env &e, const EnvState &s, long long i) {
    e.occ = s.occ[i]; e.clo = s.clo[i]; e.cons = s.cons[i]; e.ret = s.ret[i];
    const u64 misc = s.misc[i];
    e.pocc = (POCC_ALWAYS || ((misc >> M_DONE) & 1ull)) ? s.pocc[i] : 0ull;
    e.chi = (!CHI_LAZY || ((int)(misc >> M_LEN) & 127) >= CHI_FROM_LEN) ? s.chi[i] : 0ull;
    env_unpack(e, misc);
}
__device__ __forceinline__ void env_store(const Env &e, const EnvState &s, long long i, bool store_chi = true, bool store_cons = true) {
    const u64 misc = ((u64)e.hr << M_HR) | ((u64)e.hc << M_HC) | ((u64)e.tr << M_TR) | ((u64)e.tc << M_TC) |
                     ((u64)e.fr << M_FR) | ((u64)e.fc << M_FC) | ((u64)e.pfr << M_PFR) | ((u64)e.pfc << M_PFC) |
                     ((u64)e.pd << M_PD) | ((u64)e.len << M_LEN) | ((u64)e.t << M_T) | ((u64)e.dn << M_DONE) |
                     ((u64)e.err << M_ERR);
    s.occ[i] = e.occ; s.pocc[i] = e.pocc; s.clo[i] = e.clo; s.misc[i] = misc;
    if (store_chi) s.chi[i] = e.chi;
    if (store_cons) s.cons[i] = e.cons;
    s.ret[i] = e.ret;
}
// a fresh SnakeGame() (structs.jl:33-99, utils.jl:199); error bits are sticky
__device__ __forceinline__ void env_reset(Env &e) {
    e.occ = INIT_OCC; e.pocc = INIT_OCC; e.clo = 0; e.chi = 0; e.cons = 0; e.ret = 0.0f;
    e.hr = 7; e.hc = 1; e.tr = 8; e.tc = 1; e.fr = 3; e.fc = 4; e.pfr = 3; e.pfc = 4; e.pd = 0; e.len = 2; e.t = 0; e.dn = 0;
}
// step!(game, action) + virtual_step for one live env (utils.jl:100-109, 112-132): returns the reward, m3 = the
// next_is_suicidal bits.  aidx: index into available_actions, or an absolute direction when is_abs.
template <bool WITH_MASK = true>
__device__ __forceinline__ float env_advance(Env &e, int &aidx, int is_abs, u64 list_mask, const uint8_t *s_food_bit,
                                             uint32_t &m3) {
    int d;
    if (is_abs) {
        d = aidx;
        if (d > 3) { e.err |= SNK_ENV_ERR_ACTION; d = 0; }
    } else {
        if (aidx > 2) { e.err |= SNK_ENV_ERR_ACTION; aidx = 0; }
        d = av_dir(e.pd, aidx);
    }
    // grow_maybe! (utils.jl:66-81) on the board of the previous step
    int dr, dc;
    dir_delta(d, dr, dc);
    const int nr = e.hr + dr, nc = e.hc + dc;
    const bool wall = (nr == 0) | (nr == 9) | (nc == 0) | (nc == 9);
    const u64 nbit = wall ? 0ull : (1ull << ((nr - 1) + 8 * (nc - 1)));
    const bool eat = (e.fr != 0) & (nr == e.fr) & (nc == e.fc);
    const bool reverse = d == (e.pd ^ 1);                           // utils.jl:57, third clause
    e.pocc = e.occ; e.pfr = e.fr; e.pfc = e.fc;                    // this board becomes frame 1
    e.chi = (e.chi << 2) | (e.clo >> 62);                           // pushfirst!(snake, new_head)
    e.clo = (e.clo << 2) | (u64)d;
    e.len++;
    bool self = false;
    float reward;
    if (eat) {
        reward = 1.0f;                                              // eating_reward
        e.fr = 0; e.fc = 0;
        int i = food_search(e.occ | nbit, e.cons, list_mask, s_food_bit);
        if (i >= 0) {
            e.cons |= 1ull << i;                                    // deleteat!(food_list, idx)
            int b = s_food_bit[i];
            e.fr = (b & 7) + 1; e.fc = (b >> 3) + 1;
        } else if (i == -1) {
            e.err |= SNK_ENV_ERR_FOOD;
        }
        e.occ |= nbit;
    } else {
        e.occ &= ~(1ull << ((e.tr - 1) + 8 * (e.tc - 1)));          // remove_tail!
        int c = chain_get(e.clo, e.chi, e.len - 2), er, ec;
        dir_delta(c, er, ec);
        e.tr += er; e.tc += ec;
        e.len--;
        reward = -0.01f;                                            // male_di_vivere
        self = (e.occ & nbit) != 0ull;                              // count(==(head), snake) > 1
        e.occ |= nbit;
    }
    e.t++;
    const bool lost = wall | self | reverse | (e.t >= 500);         // utils.jl:88 (history length > 500)
    if (lost) reward = -1.0f;                                       // suicide_penalty
    e.hr = nr; e.hc = nc; e.pd = d; e.dn = lost;
    e.ret += reward;
    m3 = 7u;
    if (WITH_MASK && !lost) m3 = losing_mask3(e.occ, e.cons, e.hr, e.hc, e.tr, e.tc, e.fr, e.fc, e.pd, e.t, list_mask, s_food_bit, e.err);
    return reward;
}

// The Float32 / Int64 observation formats are HBM-bound at 3 CTAs per SM; the small formats are bound by instruction issue and
// latency: capping them at 64 registers buys a fourth CTA per SM (no spills).
// SNK_OBS_BITS: the two boards in the library's own bit-board form plus the step's scalars, 24 bytes per env (see the
// header).  Written by the env's own thread in phase A: no table expansion, no phase B.
__device__ __forceinline__ void store_bits_record(void *obs, long long env, u64 pocc, int pfr, int pfc, u64 occ, int fr, int fc,
                                                  int hr, int hc, uint32_t m3, bool done, int aidx, float reward) {
    u64 *rec = reinterpret_cast<u64 *>(obs) + 3 * env;
    const uint32_t cells = (uint32_t)(pfr | (pfc << 4)) | ((uint32_t)(fr | (fc << 4)) << 8) | ((uint32_t)(hr | (hc << 4)) << 16) |
                           (((m3 & 7u) | ((uint32_t)done << 3) | (((uint32_t)aidx & 3u) << 4)) << 24);
    rec[0] = pocc;
    rec[1] = occ;
    rec[2] = (u64)cells | ((u64)__float_as_uint(reward) << 32);
}
__host__ __device__ constexpr bool obs_expands(int fmt) { return fmt != SNK_OBS_NONE && fmt != SNK_OBS_BITS; }   // formats that go through phase B

template <int OBS, bool SELECT, bool SINK>
__global__ void __launch_bounds__(TPB, (OBS == SNK_OBS_F32 || OBS == SNK_OBS_I64) ? SNK_MINB : 4) k_step(const __grid_constant__ StepArgs a) {
    __shared__ __align__(16) uint32_t s_planes[TPB * PLANE_WORDS];
    __shared__ ObsTables s_tb;
    __shared__ uint8_t s_food_bit[MAX_FOOD];

    const int tid = threadIdx.x;
    const long long env0 = a.env_begin + (long long)blockIdx.x * TPB;
    const long long rem = a.env_end - env0;
    const int n_local = rem < TPB ? (int)rem : TPB;
    const long long env = env0 + tid;

    if (tid < MAX_FOOD) s_food_bit[tid] = a.food.bit[tid];
    if (obs_expands(OBS)) fill_tables<OBS>(s_tb, tid);
    __syncthreads();

    if (tid < n_local) {
        // ---- phase A: one thread, one env ------------------------------------------------------
        Env e;
        env_load<SINK, true>(e, a.s, env);                         // the transition record needs board_{t-2}
        const bool chi_live = e.len >= CHI_FROM_LEN;
        const u64 cons_loaded = e.cons;                             // changes only when an apple is eaten or the env resets
        const u64 list_mask = a.food.mask();
        const u64 occ_tm2 = e.pocc;                                 // board_{t-2}, for the transition record
        const int fr_tm2 = e.pfr, fc_tm2 = e.pfc, pd_before = e.pd;

        int aidx;
        if (SELECT) {
            float q0 = a.q[3 * env], q1 = a.q[3 * env + 1], q2 = a.q[3 * env + 2];
            float u;
            int ri;
            if (a.u != nullptr && a.ridx != nullptr) {
                u = a.u[env];
                ri = a.ridx[env];
            } else {
                internal_draw(a.seed, a.step_counter, env, u, ri);
                if (a.u != nullptr) u = a.u[env];
                if (a.ridx != nullptr) ri = a.ridx[env];
            }
            aidx = select_idx(q0, q1, q2, a.eps, u, ri);
            if (a.act_out != nullptr) a.act_out[env] = (uint8_t)aidx;
        } else {
            aidx = a.act[env];
        }

        float reward = 0.0f;
        uint32_t m3 = 7u;
        if (!e.dn) reward = env_advance(e, aidx, a.is_abs, list_mask, s_food_bit, m3);

        // (not store_step_outputs: through it ptxas gives the SINK kernels of three formats one or two registers more or less)
        if (a.out.reward != nullptr) a.out.reward[env] = reward;
        if (a.out.done != nullptr) a.out.done[env] = (uint8_t)e.dn;
        if (a.out.mask != nullptr) store_mask3(a.out.mask + 3 * env, m3);
        if (a.out.ep_return != nullptr) a.out.ep_return[env] = e.ret;
        if (a.out.ep_score != nullptr) a.out.ep_score[env] = e.len - 2;

        if (obs_expands(OBS)) {
            constexpr bool PERM = OBS != SNK_OBS_F32 && OBS != SNK_OBS_I64;
            board_planes<PERM>(e.pocc, e.pfr, e.pfc, false, 0, 0, s_planes + tid * PLANE_WORDS);
            board_planes<PERM>(e.occ, e.fr, e.fc, true, e.hr, e.hc, s_planes + tid * PLANE_WORDS + 8);
        }
        if (OBS == SNK_OBS_BITS)
            store_bits_record(a.out.obs, env, e.pocc, e.pfr, e.pfc, e.occ, e.fr, e.fc, e.hr, e.hc, m3, e.dn, aidx, reward);

        if (SINK) {
            // store!(rpb, exp) for envs in index order == ring slot (stored_so_far + env) mod capacity; when the
            // step holds more envs than the ring, the later env wins exactly as sequential store! calls would
            const long long k = env - a.env_begin;
            if (k + a.sink_cap >= a.sink_n) {
                uint4 *rec = a.sink + ((a.sink_base + k) % a.sink_cap) * REC_U4;
                uint4 p0, p1;
                board_planes_reg(occ_tm2, fr_tm2, fc_tm2, false, 0, 0, p0, p1);
                rec[0] = p0; rec[1] = p1;
                board_planes_reg(e.pocc, e.pfr, e.pfc, false, 0, 0, p0, p1);
                rec[2] = p0; rec[3] = p1;
                board_planes_reg(e.occ, e.fr, e.fc, true, e.hr, e.hc, p0, p1);
                rec[4] = p0; rec[5] = p1;
                rec[6] = make_uint4(__float_as_uint(reward),
                                    (uint32_t)aidx | ((uint32_t)e.dn << 8) | (m3 << 16) | ((uint32_t)pd_before << 24),
                                    __float_as_uint(e.ret), (uint32_t)(e.len - 2));
                rec[7] = make_uint4((uint32_t)env, (uint32_t)e.t, 0u, 0u);
            }
        }

        if (e.dn && a.auto_reset) env_reset(e);
        env_store(e, a.s, env, chi_live || e.len >= CHI_FROM_LEN, e.cons != cons_loaded);
    }

    if (obs_expands(OBS)) {
        __syncthreads();
        expand_obs<OBS>(a.out.obs, env0, n_local, s_planes, s_tb, tid);
    }
}

// ---- T steps in one launch (small batches are launch-latency bound: the env stays in registers) ----------
// EPB envs per CTA of TPB threads: phase A uses the first EPB threads, phase B all TPB of them.
// Step-major I/O: act (T,N) u8; reward (T,N), done (T,N), mask (T,3,N) bytes, obs (T, N x 200) — any output NULL.
struct RolloutArgs {
    EnvState s;
    const uint8_t *act;
    StepOutputs out;
    long long n;
    int steps, auto_reset, is_abs;
    long long *prof;         // debug (snk_debug_rollout_timing): cycle counts of CTA 0's logic warp / expander thread 0
    FoodTable food;
};
#ifndef SNK_RTPB
#define SNK_RTPB 128
#endif
#ifndef SNK_WS_EPB
#define SNK_WS_EPB 16           // measured at 4,096 envs: 4 -> 2.26 us per step, 8 -> 1.44, 16 -> 1.29, 32 -> 1.31 (more CTAs per SM only add issue contention: the step time is the logic warp's instruction chain)
#endif
constexpr int WS_EPB = SNK_WS_EPB; // envs per CTA of the warp-specialised small-batch rollout kernel
constexpr int RTPB = SNK_RTPB;    // threads per CTA of the rollout kernel (latency-bound: tuned separately from k_step)
template <int OBS, int EPB>
__global__ void __launch_bounds__(RTPB) k_rollout(const __grid_constant__ RolloutArgs a) {
    __shared__ __align__(16) uint32_t s_planes[EPB * PLANE_WORDS];
    __shared__ ObsTables s_tb;
    __shared__ uint8_t s_food_bit[MAX_FOOD];
    const int tid = threadIdx.x;
    const long long env0 = (long long)blockIdx.x * EPB;
    const long long rem = a.n - env0;
    const int n_local = rem < EPB ? (int)rem : EPB;
    const long long env = env0 + tid;
    const bool mine = tid < n_local;
    if (tid < MAX_FOOD) s_food_bit[tid] = a.food.bit[tid];
    if (OBS != SNK_OBS_NONE) fill_tables<OBS>(s_tb, tid, RTPB);
    __syncthreads();
    const u64 list_mask = a.food.mask();
    Env e;
    if (mine) env_load(e, a.s, env);
    const size_t obs_step = (size_t)a.n * obs_bytes(OBS);
    for (int t = 0; t < a.steps; t++) {
        if (mine) {
            const long long o = (long long)t * a.n + env;
            int aidx = a.act[o];
            float reward = 0.0f;
            uint32_t m3 = 7u;
            if (!e.dn) reward = env_advance(e, aidx, a.is_abs, list_mask, s_food_bit, m3);
            store_step_outputs(a.out, o, reward, e.dn, m3, e.ret, e.len - 2);
            if (OBS != SNK_OBS_NONE) {
                board_planes(e.pocc, e.pfr, e.pfc, false, 0, 0, s_planes + tid * PLANE_WORDS);
                board_planes(e.occ, e.fr, e.fc, true, e.hr, e.hc, s_planes + tid * PLANE_WORDS + 8);
            }
            if (e.dn && a.auto_reset) env_reset(e);
        }
        if (OBS != SNK_OBS_NONE) {
            __syncthreads();
            expand_obs<OBS, RTPB, 5, true>((uint8_t *)a.out.obs + (size_t)t * obs_step, env0, n_local, s_planes, s_tb, tid);
            __syncthreads();
        }
    }
    if (mine) env_store(e, a.s, env);
}

// ---- small batches: warp-specialised multi-step rollout -------------------------------------------------------------
// At 4,096 envs (BASELINE config 2) a step moves 3.5 MB: the time per step is a serial instruction chain, not memory.  So
// three chains run side by side in a CTA (EPB envs, one per lane): warp 0 only advances the envs (260 instructions per step)
// and drops a 48-byte record per env into a double-buffered hand-over slot; warp 1 computes next_is_suicidal from the record
// (three virtual steps: a chain as long as the step's) and writes the per-env scalars; warps 2.. turn the record into the two
// boards as unit bytes and expand the observation — all while warp 0 is already in the next step.  Actions are prefetched two
// steps ahead.  Named barriers: FULL[b] (warp 0 arrives, every consumer waits), EMPTY[b] (the consumers arrive once they
// have read the record, warp 0 waits two steps later), and one among the expansion warps.
// Measured: without an observation a step costs 1,010 cycles = warp 0's chain (170 instructions) + hand-over; with Float32
// observations 1,470.  ncu's warp-stall sampling per instruction (profiles/r02_ncu_rollout_ws_stalls.txt) shows why: warp 0
// then spends a third of its time blocked at EMPTY — the pace is set by the consumers' chain FULL -> board conversion (190
// instructions on one warp per board) -> barrier -> expansion -> barrier.  (The clock64 counters of tools/rollout_probe.py
// cannot see that wait: after BAR.SYNC.DEFER_BLOCKING the clock read issues before the warp blocks, so it is booked as work.)
// Tried on top and not kept, Float32 observations, us per step: the board conversion spread over 8 threads per env 1.03 (its
// instructions land on the schedulers of warps 0 and 1); expansion warps only on the schedulers warps 0 and 1 do not use
// (groups of four warps, the other two idle) 1.35; the CTA's region of a step staged in shared memory and sent off as one
// bulk asynchronous copy 1.04; actions preloaded into shared memory 0.87 (no change); plain instead of streaming stores 0.87;
// (after the shorter board conversion, 0.80) the per-env scalars written by the idle upper lanes of the first role warp
// instead of the mask warp 0.87 — whatever lengthens the role warps' chain FULL -> boards -> barrier -> expansion costs.
struct __align__(16) Handoff {
    u64 occ, pocc, cons;
    uint32_t pk;             // hr hc fr fc pfr pfc (4 bits each) | done << 24
    uint32_t pk2;            // tr tc (4 bits each) | prev_dir << 8 | step count << 10
    float reward, ret;
    int score, pad;
};
#ifndef SNK_WS_XW
#define SNK_WS_XW 5              // expansion warps per CTA; measured at 4,096 envs, Float32 observations: 2 -> 1.13 us per step, 3 -> 1.02, 4 -> 0.90, 5 -> 0.87, 6 -> 0.97, 8 -> 0.98
#endif
constexpr int WS_XW = SNK_WS_XW;
constexpr bool WS_STREAM = true;        // streaming (.cs) and plain stores measure the same here
// warp 0 logic, warp 1 mask + scalars, warps 2 .. 1+XW boards + expansion, warp 2+XW a second mask warp for the small observation
// formats: the two take turns (even / odd steps).  Once the board conversion got shorter the single mask warp was the busiest chain
// of the CTA (ncu: 88 % of its samples outside barriers, 206 instructions per step); each now has two steps' time for one step.
constexpr int WS_THREADS = 32 * (3 + WS_XW);   // launched
constexpr int WS_BAR = 32 * (2 + WS_XW);       // threads meeting at a FULL / EMPTY barrier: logic + ONE mask warp + expansion

template <int OBS, int EPB>
__global__ void __launch_bounds__(WS_THREADS) k_rollout_ws(const __grid_constant__ RolloutArgs a) {
    static_assert(EPB <= 32, "one env per lane of the logic warp");
    constexpr int NX = 32 * WS_XW;                           // expansion threads
    // Measured, us per step at 4,096 envs with one / two mask warps: no observation 0.61 / 0.45, packed 0.65 / 0.57, int8 0.66 /
    // 0.65, Float32 0.80 / 0.82 — with the large formats the expansion chain sets the pace and the extra warp only adds
    // contention, so the second mask warp stays idle there (it waits at the final barrier).
    constexpr bool TWO_MASK = OBS != SNK_OBS_F32 && OBS != SNK_OBS_I64;
    __shared__ Handoff s_hand[2][EPB];
    __shared__ __align__(16) uint32_t s_planes[EPB * PLANE_WORDS];
    __shared__ ObsTables s_tb;
    __shared__ uint8_t s_food_bit[MAX_FOOD];
    __shared__ int s_err[EPB];                               // error bits found by the virtual steps (utils.jl:23,37 inside virtual_step)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long env0 = (long long)blockIdx.x * EPB;
    const long long rem = a.n - env0;
    const int n_local = rem < EPB ? (int)rem : EPB;
    if (tid < MAX_FOOD) s_food_bit[tid] = a.food.bit[tid];
    if (tid < EPB) s_err[tid] = 0;
    if (OBS != SNK_OBS_NONE) fill_tables<OBS>(s_tb, tid, WS_THREADS);
    __syncthreads();
    // barrier ids: FULL+b (warp 0 arrives, every consumer waits), EMPTY+b (the consumers arrive once they have read slot b,
    // warp 0 waits two steps later), XB among the expansion warps.  Consumers that have nothing to do for this format
    // (expansion warps without an observation) still take part in FULL / EMPTY so that the counts stay WS_BAR.
    constexpr int FULL = 1, EMPTY = 3, XB = 5;
    const u64 list_mask = a.food.mask();
    Env e;
    const bool mine = warp == 0 && lane < n_local;
    const long long env = env0 + (mine ? lane : 0);
    if (warp == 0) {
        env_load(e, a.s, env);
        // loop invariants pinned in registers: re-reading a kernel parameter is a uniform constant load (LDCU, tens of cycles
        // of latency in front of the compare that uses it) — on a chain where every cycle counts
        int steps = a.steps, is_abs = a.is_abs, auto_reset = a.auto_reset;
        const uint8_t *actp = a.act + env;
        long long astride = a.n;
        asm volatile("" : "+r"(steps), "+r"(is_abs), "+r"(auto_reset), "+l"(actp), "+l"(astride));
        int a0 = steps > 0 ? actp[0] : 0, a1 = steps > 1 ? actp[astride] : 0;
        const uint8_t *act2 = actp + 2 * astride;
        const bool prof = a.prof != nullptr && blockIdx.x == 0 && lane == 0;
        long long p_wait = 0, p_work = 0, p_arr = 0, p_t0 = prof ? clock64() : 0;
        for (int t = 0; t < steps; t++, act2 += astride) {
            const int a2 = t + 2 < steps ? *act2 : 0;                       // in flight during two steps
            const int b = t & 1;
            const long long w0 = prof ? clock64() : 0;
            if (t >= 2) nbar_sync(EMPTY + b, WS_BAR);    // every consumer has read slot b (step t-2)
            const long long w1 = prof ? clock64() : 0;
            if (prof) p_wait += w1 - w0;
            int aidx = a0;
            float reward = 0.0f;
            uint32_t m3;
            if (!e.dn) reward = env_advance<false>(e, aidx, is_abs, list_mask, s_food_bit, m3);   // virtual_step is warp 1's job
            if (mine) {
                Handoff h;
                h.occ = e.occ; h.pocc = e.pocc; h.cons = e.cons;
                h.pk = (uint32_t)e.hr | ((uint32_t)e.hc << 4) | ((uint32_t)e.fr << 8) | ((uint32_t)e.fc << 12) |
                       ((uint32_t)e.pfr << 16) | ((uint32_t)e.pfc << 20) | ((uint32_t)e.dn << 24);
                h.pk2 = (uint32_t)e.tr | ((uint32_t)e.tc << 4) | ((uint32_t)e.pd << 8) | ((uint32_t)e.t << 10);
                h.reward = reward; h.ret = e.ret; h.score = e.len - 2; h.pad = 0;
                s_hand[b][lane] = h;
            }
            if (e.dn && auto_reset) env_reset(e);
            __syncwarp();
            const long long w2 = prof ? clock64() : 0;
            nbar_arrive(FULL + b, WS_BAR);
            if (prof) { p_work += w2 - w1; p_arr += clock64() - w2; }
            a0 = a1; a1 = a2;
        }
        if (prof) { a.prof[0] = clock64() - p_t0; a.prof[1] = p_wait; a.prof[6] = p_work; a.prof[7] = p_arr; }
    } else if (warp == 1 || (TWO_MASK && warp == 2 + WS_XW)) {
        // ---- mask warp: next_is_suicidal (three virtual steps: as long a chain as the step itself) and the per-env scalars,
        // beside the expansion of the same step, not in front of it
        const bool prof = a.prof != nullptr && blockIdx.x == 0 && lane == 0 && warp == 1;
        long long p_full = 0, p_role = 0;
        for (int t = (TWO_MASK && warp != 1) ? 1 : 0; t < a.steps; t += TWO_MASK ? 2 : 1) {   // two mask warps: even / odd steps
            const int b = t & 1;
            long long c0 = prof ? clock64() : 0;
            nbar_sync(FULL + b, WS_BAR);
            if (prof) { const long long c1 = clock64(); p_full += c1 - c0; c0 = c1; }
            Handoff h;
            if (lane < n_local) h = s_hand[b][lane];
            __syncwarp();
            if (t + 2 < a.steps) nbar_arrive(EMPTY + b, WS_BAR);       // the record is in registers
            if (lane < n_local) {
                const int hr = (int)h.pk & 15, hc = (int)(h.pk >> 4) & 15, fr = (int)(h.pk >> 8) & 15, fc = (int)(h.pk >> 12) & 15;
                const int dn = (int)(h.pk >> 24) & 1;
                uint32_t m3 = 7u;
                if (!dn) {
                    int err = 0;
                    m3 = losing_mask3(h.occ, h.cons, hr, hc, (int)h.pk2 & 15, (int)(h.pk2 >> 4) & 15, fr, fc, (int)(h.pk2 >> 8) & 3,
                                      (int)(h.pk2 >> 10) & 1023, list_mask, s_food_bit, err);
                    if (err) atomicOr(&s_err[lane], err);
                }
                store_step_outputs(a.out, (long long)t * a.n + env0 + lane, h.reward, dn, m3, h.ret, h.score);
            }
            if (prof) p_role += clock64() - c0;
        }
        if (prof) { a.prof[2] = p_full; a.prof[3] = p_role; }
    } else if (warp < 2 + WS_XW) {
        // ---- expansion warps: the two boards as unit bytes (threads 0..EPB-1 the older, 32..32+EPB-1 the newer), then the
        // expanded observation by all of them
        const int et = tid - 64;                             // 0..NX-1
        const bool prof = a.prof != nullptr && blockIdx.x == 0 && et == 0;
        long long p_exp = 0, p_xfull = 0;
        const size_t obs_step = (size_t)a.n * obs_bytes(OBS);
        for (int t = 0; t < a.steps; t++) {
            const int b = t & 1;
            long long c0 = prof ? clock64() : 0;
            nbar_sync(FULL + b, WS_BAR);
            if (prof) { const long long c1 = clock64(); p_xfull += c1 - c0; c0 = c1; }
            const int j = et & 31, role = et >> 5;
            if (OBS != SNK_OBS_NONE && j < n_local && role < 2) {
                const Handoff h = s_hand[b][j];
                if (role == 0) {
                    board_planes(h.pocc, (int)(h.pk >> 16) & 15, (int)(h.pk >> 20) & 15, false, 0, 0, s_planes + j * PLANE_WORDS);
                } else {
                    board_planes(h.occ, (int)(h.pk >> 8) & 15, (int)(h.pk >> 12) & 15, true, (int)h.pk & 15, (int)(h.pk >> 4) & 15,
                                 s_planes + j * PLANE_WORDS + 8);
                }
            }
            if (t + 2 < a.steps) nbar_arrive(EMPTY + b, WS_BAR);       // the record has been read: warp 0 may overwrite it at step t+2
            if (OBS != SNK_OBS_NONE) {
                // (Staging the CTA's contiguous region of the step in shared memory and sending it off as one bulk asynchronous
                // copy was measured slower: 1.04 against 0.90 us per step with Float32 observations.)
                nbar_sync(XB, NX);
                expand_obs<OBS, NX, 5, WS_STREAM>((uint8_t *)a.out.obs + (size_t)t * obs_step, env0, n_local, s_planes, s_tb, et);
                nbar_sync(XB, NX);
                if (prof) p_exp += clock64() - c0;
            }
        }
        if (prof) { a.prof[4] = p_exp; a.prof[5] = p_xfull; }
    }
    __syncthreads();
    if (mine) {
        e.err |= s_err[lane];
        env_store(e, a.s, env);
    }
}

// ---- stand-alone views of the state ------------------------------------------------------------
// k_state and k_losing_mask decode only the misc fields they use: decoding through env_unpack costs k_state<F32> and
// k_state<I64> 8 instructions and one or two registers more.
template <int OBS>
__global__ void __launch_bounds__(TPB) k_state(EnvState s, long long n, void *obs) {
    __shared__ __align__(16) uint32_t s_planes[TPB * PLANE_WORDS];
    __shared__ ObsTables s_tb;
    const int tid = threadIdx.x;
    const long long env0 = (long long)blockIdx.x * TPB;
    const int n_local = (n - env0) < TPB ? (int)(n - env0) : TPB;
    if (OBS == SNK_OBS_BITS) {           // boards of the current state; no step has produced scalars: flags = done bit only
        if (tid < n_local) {
            const long long env = env0 + tid;
            const u64 misc = s.misc[env];
            store_bits_record(obs, env, s.pocc[env], (int)(misc >> M_PFR) & 15, (int)(misc >> M_PFC) & 15, s.occ[env],
                              (int)(misc >> M_FR) & 15, (int)(misc >> M_FC) & 15, (int)(misc >> M_HR) & 15, (int)(misc >> M_HC) & 15,
                              0u, ((misc >> M_DONE) & 1ull) != 0, 0, 0.0f);
        }
        return;
    }
    fill_tables<OBS>(s_tb, tid);
    if (tid < n_local) {
        long long env = env0 + tid;
        u64 misc = s.misc[env];
        board_planes(s.pocc[env], (int)(misc >> M_PFR) & 15, (int)(misc >> M_PFC) & 15, false, 0, 0,
                     s_planes + tid * PLANE_WORDS);
        board_planes(s.occ[env], (int)(misc >> M_FR) & 15, (int)(misc >> M_FC) & 15, true, (int)(misc >> M_HR) & 15,
                     (int)(misc >> M_HC) & 15, s_planes + tid * PLANE_WORDS + 8);
    }
    __syncthreads();
    expand_obs<OBS>(obs, env0, n_local, s_planes, s_tb, tid);
}

// assemble_state! for the envs the last step re-initialised (auto-reset): rows of `obs` whose done flag is set are
// overwritten with the constructor state (init, init) (structs.jl:53-55), all other rows are left alone.  Turns the
// next_state output of one fused step into the acting state of the next one without re-expanding all N envs.
template <int OBS>
__global__ void __launch_bounds__(TPB) k_patch_reset(long long n, const uint8_t *__restrict__ done, void *obs) {
    __shared__ __align__(16) uint32_t s_pl[8];
    __shared__ ObsTables s_tb;
    __shared__ int s_list[TPB];
    __shared__ int s_cnt;
    const int tid = threadIdx.x;
    const long long env0 = (long long)blockIdx.x * TPB;
    if (OBS == SNK_OBS_BITS) {           // the boards of the record become (init, init); its flags and reward stay the step's
        if (env0 + tid < n && done[env0 + tid] != 0) {
            u64 *rec = reinterpret_cast<u64 *>(obs) + 3 * (env0 + tid);
            rec[0] = INIT_OCC;
            rec[1] = INIT_OCC;
            rec[2] = (rec[2] & ~0xFFFFFFull) | (u64)((3 | (4 << 4)) | ((3 | (4 << 4)) << 8) | ((7 | (1 << 4)) << 16));
        }
        return;
    }
    fill_tables<OBS>(s_tb, tid);
    if (tid == 0) {
        s_cnt = 0;
        board_planes(INIT_OCC, 3, 4, false, 0, 0, s_pl);
    }
    __syncthreads();
    if (env0 + tid < n && done[env0 + tid] != 0) s_list[atomicAdd(&s_cnt, 1)] = tid;
    __syncthreads();
    const int cnt = s_cnt;
    if (OBS == SNK_OBS_I64) {
        for (int j = tid; j < cnt * 100; j += TPB) {
            const int e = j / 100, p = j - e * 100, k = 2 * (p % 50);
            longlong2 v;
            v.x = code_value(cell_code(s_pl, k));
            v.y = code_value(cell_code(s_pl, k + 1));
            reinterpret_cast<longlong2 *>(obs)[(env0 + s_list[e]) * 100 + p] = v;
        }
    } else {
        for (int j = tid; j < cnt * 50; j += TPB) {
            const int e = j / 50, qq = j - e * 50;
            const uint32_t idx = reinterpret_cast<const uint8_t *>(s_pl)[qq % 25];
            const long long o = (env0 + s_list[e]) * 50 + qq;
            if (OBS == SNK_OBS_F32) reinterpret_cast<float4 *>(obs)[o] = s_tb.f32[idx];
            else if (OBS == SNK_OBS_I8) reinterpret_cast<uint32_t *>(obs)[o] = reinterpret_cast<const uint32_t *>(s_tb.f32)[idx];
            else reinterpret_cast<uint8_t *>(obs)[o] = reinterpret_cast<const uint8_t *>(s_tb.f32)[idx];
        }
    }
}

__global__ void k_reset(EnvState s, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    s.occ[i] = INIT_OCC; s.pocc[i] = INIT_OCC; s.clo[i] = 0; s.chi[i] = 0; s.cons[i] = 0;
    s.misc[i] = INIT_MISC; s.ret[i] = 0.0f;
}

__global__ void k_available_actions(EnvState s, long long n, uint8_t *out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int pd = (int)(s.misc[i] >> M_PD) & 3;
    for (int k = 0; k < 3; k++) out[3 * i + k] = (uint8_t)av_dir(pd, k);
}

__global__ void k_losing_mask(EnvState s, long long n, uint8_t *out, FoodTable food) {
    __shared__ uint8_t s_food_bit[MAX_FOOD];
    if (threadIdx.x < MAX_FOOD) s_food_bit[threadIdx.x] = food.bit[threadIdx.x];
    __syncthreads();
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u64 misc = s.misc[i];
    uint32_t m3 = 7u;
    if (!((misc >> M_DONE) & 1ull)) {
        int err = (int)(misc >> M_ERR) & 15, err0 = err;
        m3 = losing_mask3(s.occ[i], s.cons[i], (int)(misc >> M_HR) & 15, (int)(misc >> M_HC) & 15,
                          (int)(misc >> M_TR) & 15, (int)(misc >> M_TC) & 15, (int)(misc >> M_FR) & 15,
                          (int)(misc >> M_FC) & 15, (int)(misc >> M_PD) & 3, (int)(misc >> M_T) & 1023, food.mask(),
                          s_food_bit, err);
        if (err != err0) s.misc[i] = (misc & ~(15ull << M_ERR)) | ((u64)err << M_ERR);
    }
    store_mask3(out + 3 * i, m3);
}

__global__ void k_select(long long n, const float *q, float eps, const float *u, const uint8_t *ridx, u64 seed,
                         u64 step, uint8_t *out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float uu;
    int ri;
    internal_draw(seed, step, i, uu, ri);
    if (u != nullptr) uu = u[i];
    if (ridx != nullptr) ri = ridx[i];
    out[i] = (uint8_t)select_idx(q[3 * i], q[3 * i + 1], q[3 * i + 2], eps, uu, ri);
}

// which: 0 score (i32), 1 done (u8), 2 error flags (u8), 3 steps (i32)
__global__ void k_scalars(EnvState s, long long n, int which, void *out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    u64 misc = s.misc[i];
    if (which == 0) ((int32_t *)out)[i] = ((int)(misc >> M_LEN) & 127) - 2;
    else if (which == 1) ((uint8_t *)out)[i] = (uint8_t)((misc >> M_DONE) & 1ull);
    else if (which == 2) ((uint8_t *)out)[i] = (uint8_t)((misc >> M_ERR) & 15ull);
    else ((int32_t *)out)[i] = (int)(misc >> M_T) & 1023;
}

__global__ void k_count_errors(EnvState s, long long n, unsigned long long *count) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    bool e = i < n && ((s.misc[i] >> M_ERR) & 15ull) != 0ull;
    unsigned b = __ballot_sync(0xffffffffu, e);
    if ((threadIdx.x & 31) == 0 && b) atomicAdd(count, (unsigned long long)__popc(b));
}

// masked max-Q target (utils.jl:448-451).  Base.max: NaN-propagating, +0.0 > -0.0.
__device__ __forceinline__ float jl_max(float a, float b) {
    if (a != a || b != b) return a + b;
    if (a > b) return a;
    if (b > a) return b;
    return (__float_as_uint(a) >> 31) ? b : a;
}
__global__ void k_masked_target(const float *q, const uint8_t *mask, const float *r, const uint8_t *done, double gamma,
                                float fill, double *y64, float *y32, long long B) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    float q0 = mask[3 * i] ? fill : q[3 * i];
    float q1 = mask[3 * i + 1] ? fill : q[3 * i + 1];
    float q2 = mask[3 * i + 2] ? fill : q[3 * i + 2];
    float m = jl_max(jl_max(q0, q1), q2);
    // @. rewards + 0.97 * max_next_q * (1 - dones): Float64 per element, left to right, no FMA
    double tt = __dmul_rn(gamma, (double)m);
    tt = __dmul_rn(tt, (double)(1 - (int)(done[i] != 0)));
    double y = __dadd_rn((double)r[i], tt);
    if (y64 != nullptr) y64[i] = y;
    if (y32 != nullptr) y32[i] = (float)y;
}


// ---- replay ring: stack_exp (utils.jl:343-383) of the records at idx[0..B) ------------------------------
// One CTA per 32 samples; the records' planes go to shared memory, then states (10,10,2,B) and next_states are
// streamed out with the same nibble->float4 table as the step kernel.
constexpr int GATHER_S = 32;
__global__ void __launch_bounds__(128) k_replay_gather(const uint4 *__restrict__ ring, long long cap, const long long *__restrict__ idx,
                                                       long long B, float *states, float *next_states, uint8_t *actions,
                                                       float *rewards, uint8_t *dones, uint8_t *mask, float *ep_return,
                                                       int32_t *score, int *bad_index) {
    __shared__ __align__(16) uint32_t s_pl[GATHER_S * 24];        // per sample: 3 boards x (P0[4], P1[4])
    __shared__ ObsTables s_tb;
    const int tid = threadIdx.x;
    const long long b0 = (long long)blockIdx.x * GATHER_S;
    const int n_local = (B - b0) < GATHER_S ? (int)(B - b0) : GATHER_S;
    fill_tables<SNK_OBS_F32>(s_tb, tid, 128);
    // 4 threads per sample copy the 6 plane vectors + scalars
    if (tid < n_local * 4) {
        const int sl = tid >> 2, part = tid & 3;
        long long i = idx[b0 + sl];
        if (i < 0 || i >= cap) { *bad_index = 1; i = 0; }
        const uint4 *rec = ring + i * REC_U4;
        uint4 *dst = reinterpret_cast<uint4 *>(s_pl + sl * 24);
        if (part < 3) { dst[2 * part] = rec[2 * part]; dst[2 * part + 1] = rec[2 * part + 1]; }
        else {
            const uint4 sc = rec[6];
            const long long o = b0 + sl;
            if (rewards) rewards[o] = __uint_as_float(sc.x);
            if (actions) actions[o] = (uint8_t)(sc.y & 0xFF);
            if (dones) dones[o] = (uint8_t)((sc.y >> 8) & 0xFF);
            if (mask) { mask[3 * o] = (sc.y >> 16) & 1; mask[3 * o + 1] = (sc.y >> 17) & 1; mask[3 * o + 2] = (sc.y >> 18) & 1; }
            if (ep_return) ep_return[o] = __uint_as_float(sc.z);
            if (score) score[o] = (int32_t)sc.w;
        }
    }
    __syncthreads();
    // two outputs: states uses boards (0,1), next_states boards (1,2); 50 float4 units per sample each
    const int total = n_local * 50;
#pragma unroll 2
    for (int which = 0; which < 2; which++) {
        float *outp = which == 0 ? states : next_states;
        if (outp == nullptr) continue;
        float4 *o4 = reinterpret_cast<float4 *>(outp) + b0 * 50;
        for (int j = tid; j < total; j += 128) {
            int e = (int)(((unsigned)j * 5243u) >> 18);
            int qq = j - e * 50;
            int f = qq >= 25;
            int q = qq - 25 * f;
            const uint32_t *pl = s_pl + e * 24 + (which + f) * 8;
            int w = q >> 3, sh = (q & 7) * 4;
            uint32_t ix = ((pl[w] >> sh) & 15u) | (((pl[4 + w] >> sh) & 15u) << 4);
            SNK_OBS_STORE(o4 + j, s_tb.f32[ix]);
        }
    }
}

// B distinct slots in [0, n): a keyed bijection of [0, 2^k) (4-round Feistel on k bits, k even) cycle-walked
// into [0, n) and evaluated at counters 0..B-1 — sampling without replacement with no state and no rejection set.
__device__ __forceinline__ unsigned long long feistel_perm(unsigned long long x, int half_bits, u64 key) {
    const unsigned long long m = (1ull << half_bits) - 1ull;
    unsigned long long l = x >> half_bits, r = x & m;
#pragma unroll
    for (int round = 0; round < 4; round++) {
        unsigned long long f = splitmix64(r ^ (key + 0x9E3779B97F4A7C15ull * (u64)(round + 1))) & m;
        unsigned long long nl = r;
        r = l ^ f;
        l = nl;
    }
    return (l << half_bits) | r;
}
__global__ void k_replay_sample(long long n, long long B, u64 key, long long *out) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B) return;
    int bits = 2;
    while ((1ll << bits) < n) bits += 2;
    unsigned long long x = (unsigned long long)i;
    do { x = feistel_perm(x, bits / 2, key); } while (x >= (unsigned long long)n);
    out[i] = (long long)x;
}

// ---- checkpoint validation (snk_env_load_host, snk_replay_load_host; DESIGN §5e) ----------------------------------------
// A checkpoint comes from a file: input from outside the program.  The kernels decode coordinates, lengths and chain entries
// from the state and trust them, so a load accepts only states the step kernel can have stored.  Rule codes index
// kEnvRuleText / kReplayRuleText.
enum EnvRule { ER_OK, ER_BITS, ER_HEAD, ER_TAIL, ER_FOOD, ER_PFOOD, ER_LEN, ER_STEPS, ER_CONS, ER_PD, ER_CHAIN, ER_CHAIN_TAIL, ER_OCC };
enum ReplayRule { RR_OK, RR_ACTION, RR_DONE, RR_MASK, RR_PD };

__device__ __forceinline__ bool interior(int r, int c) { return r >= 1 && r <= 8 && c >= 1 && c <= 8; }
__device__ __forceinline__ u64 interior_bit(int r, int c) { return 1ull << ((r - 1) + 8 * (c - 1)); }

// the first rule env i's state breaks, ER_OK if none
__device__ __forceinline__ int env_rule(u64 occ, u64 clo, u64 chi, u64 cons, u64 misc, u64 list_mask) {
    Env e;
    env_unpack(e, misc);
    if (misc >> (M_ERR + 2)) return ER_BITS;                       // error bits beyond FOOD | ACTION, bits 56..63
    // a wall death draws the head on the wall ring (next to an interior cell: never a corner)
    const bool on_wall = ((e.hr == 0 || e.hr == 9) && e.hc >= 1 && e.hc <= 8) || ((e.hc == 0 || e.hc == 9) && e.hr >= 1 && e.hr <= 8);
    const bool head_in = interior(e.hr, e.hc);
    if (!head_in && !(e.dn && on_wall)) return ER_HEAD;
    if (!interior(e.tr, e.tc)) return ER_TAIL;
    if (!interior(e.fr, e.fc) && (e.fr | e.fc) != 0) return ER_FOOD;   // (0, 0) = no food on the board
    if (!interior(e.pfr, e.pfc) && (e.pfr | e.pfc) != 0) return ER_PFOOD;
    if (e.len < 2 || e.len > 64) return ER_LEN;
    if (e.t > (e.dn ? 500 : 499)) return ER_STEPS;                 // the 500th step loses (utils.jl:88)
    if (cons & ~list_mask) return ER_CONS;
    if (chain_get(clo, chi, 0) != e.pd) return ER_PD;              // prev_dir is the last move
    // the body from the head: segment j+1 = segment j - delta(entry j); distinct interior cells, the last one the tail
    int r = e.hr, c = e.hc;
    u64 body = 0;
    for (int j = 0; j < e.len - 1; j++) {
        int dr, dc;
        dir_delta(chain_get(clo, chi, j), dr, dc);
        r -= dr;
        c -= dc;
        if (!interior(r, c) || (body & interior_bit(r, c))) return ER_CHAIN;
        body |= interior_bit(r, c);
    }
    if (r != e.tr || c != e.tc) return ER_CHAIN_TAIL;
    // occ = body + head cell; only a lost head may share a cell with the body (it ran into it)
    if (head_in) {
        if (!e.dn && (body & interior_bit(e.hr, e.hc))) return ER_CHAIN;
        body |= interior_bit(e.hr, e.hc);
    }
    return occ == body ? ER_OK : ER_OCC;
}

// the lowest failing index of the launch and its rule, packed as index << 8 | rule: a block-wide OR skips clean CTAs, the
// others reduce in shared memory and issue one global atomicMin
__device__ __forceinline__ void report_first_bad(int rule, long long i, unsigned long long *first) {
    __shared__ unsigned long long s_min;
    if (!__syncthreads_or(rule != 0)) return;
    if (threadIdx.x == 0) s_min = ~0ull;
    __syncthreads();
    if (rule != 0) atomicMin(&s_min, ((unsigned long long)i << 8) | (unsigned)rule);
    __syncthreads();
    if (threadIdx.x == 0) atomicMin(first, s_min);
}

__global__ void __launch_bounds__(256) k_env_validate(EnvState s, long long n, u64 list_mask, unsigned long long *first) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int rule = i < n ? env_rule(s.occ[i], s.clo[i], s.chi[i], s.cons[i], s.misc[i], list_mask) : ER_OK;
    report_first_bad(rule, i, first);
}

// the scalar bytes of a 128-byte record (see REC_U4): word 1 of rec[6] = action | done << 8 | mask bits << 16 | prev_dir << 24
__global__ void __launch_bounds__(256) k_replay_validate(const uint4 *ring, long long n, unsigned long long *first) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    int rule = RR_OK;
    if (i < n) {
        const uint32_t w = ring[i * REC_U4 + 6].y;
        if ((w & 0xFF) > 2) rule = RR_ACTION;                      // k_sample_grads indexes the three Q-values with it
        else if (((w >> 8) & 0xFF) > 1) rule = RR_DONE;
        else if (((w >> 16) & 0xFF) > 7) rule = RR_MASK;
        else if ((w >> 24) > 3) rule = RR_PD;
    }
    report_first_bad(rule, i, first);
}

}  // namespace snk

// ================================================================================================
// C ABI
// ================================================================================================
using namespace snk;

struct snk_env {
    long long n;
    int device;
    uint32_t flags;
    EnvState s;
    FoodTable food;            // active list
    cudaStream_t own_stream, stream;
    cudaStream_t copy_stream[2];
    cudaEvent_t ev_in, ev_chunk[64], ev_up[64], ev_done;
    u64 seed, step_counter;
    unsigned long long *d_count;
    // staging for the _host entry points (allocated on first use)
    float *d_q, *d_u, *d_reward, *d_ep_return;
    uint8_t *d_ridx, *d_act, *d_done, *d_mask;
    int32_t *d_ep_score;
    void *d_obs;
    size_t d_obs_bytes;
};

// the replay ring (ReplayBuffer, structs.jl:104-116)
struct snk_replay_s {
    long long capacity;
    int device;
    uint4 *ring;             // capacity x 128-byte records
    long long total;         // transitions ever stored since the last clear
    u64 draws;               // sample calls so far (counter of the keyed permutation)
    int *d_bad;
    uint8_t *stage;          // device staging of snk_replay_gather_host
    size_t stage_bytes;
};

static const uint8_t kDefaultFoodRC[100] = {  // Xoshiro(42) list, structs.jl:70 (pinned by tests/test_oracle_golden.py)
    7, 5, 5, 7, 7, 3, 6, 7, 5, 4, 7, 7, 4, 4, 6, 2, 4, 3, 5, 5, 2, 6, 3, 6, 5, 4, 5, 8, 4, 6, 4, 3, 7, 4,
    2, 2, 7, 5, 7, 3, 6, 5, 8, 3, 4, 9, 4, 7, 8, 6, 4, 4, 6, 6, 4, 2, 2, 8, 9, 3, 7, 4, 4, 8, 7, 7, 4, 2,
    3, 9, 4, 8, 7, 8, 2, 7, 2, 6, 9, 5, 9, 9, 7, 5, 8, 6, 4, 2, 7, 6, 4, 6, 8, 5, 2, 5, 2, 8, 9, 4};

static int set_food(FoodTable &ft, const uint8_t *rc, int n) {
    if (n < 0 || n > MAX_FOOD) return fail(SNK_ERR_INVALID, "food list length %d not in 0..64", n);
    memset(&ft, 0, sizeof(ft));
    for (int i = 0; i < n; i++) {
        int r = rc[2 * i], c = rc[2 * i + 1];
        if (r < 2 || r > 9 || c < 2 || c > 9) return fail(SNK_ERR_INVALID, "food cell %d = (%d,%d) outside 2..9", i, r, c);
        ft.bit[i] = (uint8_t)((r - 2) + 8 * (c - 2));
    }
    ft.n = n;
    return SNK_OK;
}

static inline unsigned nblocks(long long n, int tpb) { return (unsigned)((n + tpb - 1) / tpb); }

// Runs f(std::integral_constant<int, FMT>()) for the FMT among FMTS that equals fmt, then checks the launches f made: a
// runtime observation format becomes a template argument.  Each caller lists the formats it has kernels for.
template <int... FMTS, class F>
static int launch_obs_fmt(int fmt, F &&f) {
    if (!((fmt == FMTS && (f(std::integral_constant<int, FMTS>()), true)) || ...))
        return fail(SNK_ERR_INVALID, "unknown obs_fmt %d", fmt);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

#define SNK_CHECK_HANDLE(h)                                                  \
    do {                                                                     \
        if ((h) == nullptr) return fail(SNK_ERR_INVALID, "%s: null handle", __func__); \
    } while (0);                                                             \
    snk::DeviceGuard guard__((h)->device)

template <typename T>
static cudaError_t ensure(T **p, size_t bytes) {
    if (*p != nullptr) return cudaSuccess;
    return cudaMalloc((void **)p, bytes);
}

// The device staging buffers of the host-buffer entry points are read by copies on copy_stream[0] that the handle's own
// stream does NOT wait for (so that later work on it — e.g. the minibatch gather — overlaps those copies): whoever is about
// to overwrite the staging buffers first orders itself behind the last such copy.
static int staging_guard(snk_handle h) {
    SNK_CUDA(cudaStreamWaitEvent(h->stream, h->ev_done, 0));
    return SNK_OK;
}

// device staging buffer of the host getters (grown on demand)
static int ensure_obs_staging(snk_handle h, size_t bytes) {
    if (h->d_obs_bytes >= bytes) return SNK_OK;
    if (h->d_obs) { SNK_CUDA(cudaStreamSynchronize(h->stream)); SNK_CUDA(cudaFree(h->d_obs)); h->d_obs = nullptr; h->d_obs_bytes = 0; }
    SNK_CUDA(cudaMalloc(&h->d_obs, bytes));
    h->d_obs_bytes = bytes;
    return SNK_OK;
}

// The host getters: run(dev), the device form, writes `bytes` into the staging buffer dev, which is then copied down
// (synchronously).  staging_guard comes first: nothing may write the staging buffer before it.
template <class Run>
static int get_host(snk_handle h, void *out_host, size_t bytes, Run &&run) {
    int rc = staging_guard(h);
    if (rc == SNK_OK) rc = ensure_obs_staging(h, bytes);
    if (rc == SNK_OK) rc = run(h->d_obs);
    if (rc != SNK_OK) return rc;
    SNK_CUDA(cudaMemcpyAsync(out_host, h->d_obs, bytes, cudaMemcpyDeviceToHost, h->stream));
    SNK_CUDA(cudaStreamSynchronize(h->stream));
    return SNK_OK;
}

#ifndef SNK_HOST_CHUNK_MB
#define SNK_HOST_CHUNK_MB 16u      // measured at 2^20 envs: packed2 observations 8 MB chunks 1.49 ms per step, 16 MB 1.37, 32 MB 1.39, 64 MB 1.42; bit records 4 MB 0.90, 8 MB 0.82, 16 MB 0.753, 32 MB 0.756
#endif
static long long *g_rollout_prof = nullptr;

// ---- device memory with generic L2 compression (snk_device_alloc) ---------------------------------------------------
// Blackwell's L2 compresses the lines of an allocation made with CU_MEM_ALLOCATION_COMP_GENERIC when it writes them back to
// DRAM.  It is lossless: kernels and copies see the same bytes.  k_step's Float32 observations are mostly zeros and a few
// repeated words; written into such memory, the step moves fewer bytes over the DRAM bus than it stores (DESIGN §3).
// The driver API comes from cudaGetDriverEntryPoint: the library does not link libcuda.
struct Vmm {
    CUresult (*device_get)(CUdevice *, int);
    CUresult (*get_attribute)(int *, CUdevice_attribute, CUdevice);
    CUresult (*granularity)(size_t *, const CUmemAllocationProp *, CUmemAllocationGranularity_flags);
    CUresult (*create)(CUmemGenericAllocationHandle *, size_t, const CUmemAllocationProp *, unsigned long long);
    CUresult (*properties)(CUmemAllocationProp *, CUmemGenericAllocationHandle);
    CUresult (*address_reserve)(CUdeviceptr *, size_t, size_t, CUdeviceptr, unsigned long long);
    CUresult (*map)(CUdeviceptr, size_t, size_t, CUmemGenericAllocationHandle, unsigned long long);
    CUresult (*set_access)(CUdeviceptr, size_t, const CUmemAccessDesc *, size_t);
    CUresult (*unmap)(CUdeviceptr, size_t);
    CUresult (*address_free)(CUdeviceptr, size_t);
    CUresult (*release)(CUmemGenericAllocationHandle);
};
static int vmm_api(const Vmm **out) {
    static Vmm api;
    static int state = 0;                       // 0 = not loaded yet, 1 = loaded, -1 = an entry point is missing
    static std::mutex mu;
    std::lock_guard<std::mutex> lk(mu);
    if (state == 0) {
        struct { const char *name; void **slot; } want[] = {
            {"cuDeviceGet", (void **)&api.device_get}, {"cuDeviceGetAttribute", (void **)&api.get_attribute},
            {"cuMemGetAllocationGranularity", (void **)&api.granularity}, {"cuMemCreate", (void **)&api.create},
            {"cuMemGetAllocationPropertiesFromHandle", (void **)&api.properties},
            {"cuMemAddressReserve", (void **)&api.address_reserve}, {"cuMemMap", (void **)&api.map},
            {"cuMemSetAccess", (void **)&api.set_access}, {"cuMemUnmap", (void **)&api.unmap},
            {"cuMemAddressFree", (void **)&api.address_free}, {"cuMemRelease", (void **)&api.release}};
        state = 1;
        for (auto &w : want) {
            cudaDriverEntryPointQueryResult q;
            if (cudaGetDriverEntryPoint(w.name, w.slot, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess ||
                *w.slot == nullptr) {
                cudaGetLastError();
                state = -1;
                return fail(SNK_ERR_CUDA, "driver entry point %s not available", w.name);
            }
        }
    }
    if (state < 0) return fail(SNK_ERR_CUDA, "driver virtual-memory entry points not available");
    *out = &api;
    return SNK_OK;
}
static int vmm_compression_supported(const Vmm &v, int device, int *yes) {
    CUdevice d;
    int vmm = 0, comp = 0;
    CUresult r = v.device_get(&d, device);
    if (r == CUDA_SUCCESS) r = v.get_attribute(&vmm, CU_DEVICE_ATTRIBUTE_VIRTUAL_MEMORY_MANAGEMENT_SUPPORTED, d);
    if (r == CUDA_SUCCESS) r = v.get_attribute(&comp, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, d);
    if (r != CUDA_SUCCESS) return fail(SNK_ERR_CUDA, "cuDeviceGetAttribute: CUresult %d", (int)r);
    *yes = vmm && comp;
    return SNK_OK;
}
// one live snk_device_alloc allocation; vmm = false: a cudaMalloc block
struct DevAlloc {
    CUmemGenericAllocationHandle handle;
    size_t size;                 // mapped (= reserved) bytes
    int device;
    bool vmm;
};
static std::mutex g_dev_allocs_mu;
static std::unordered_map<void *, DevAlloc> g_dev_allocs;

// *p stays NULL when the driver hands out memory that is not compressible: the caller then falls back to cudaMalloc
static int vmm_alloc_compressible(const Vmm &v, int device, size_t bytes, void **p, DevAlloc *a) {
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    prop.allocFlags.compressionType = CU_MEM_ALLOCATION_COMP_GENERIC;
    size_t g = 0;
    CUresult r = v.granularity(&g, &prop, CU_MEM_ALLOC_GRANULARITY_MINIMUM);
    if (r != CUDA_SUCCESS) return fail(SNK_ERR_CUDA, "cuMemGetAllocationGranularity: CUresult %d", (int)r);
    const size_t size = (bytes + g - 1) / g * g;
    CUmemGenericAllocationHandle h;
    r = v.create(&h, size, &prop, 0);
    if (r != CUDA_SUCCESS) return fail(SNK_ERR_CUDA, "cuMemCreate(%zu bytes, compressible): CUresult %d", size, (int)r);
    CUmemAllocationProp got = {};
    r = v.properties(&got, h);
    if (r != CUDA_SUCCESS || got.allocFlags.compressionType != CU_MEM_ALLOCATION_COMP_GENERIC) {   // the hint was not honoured
        v.release(h);
        return r == CUDA_SUCCESS ? SNK_OK : fail(SNK_ERR_CUDA, "cuMemGetAllocationPropertiesFromHandle: CUresult %d", (int)r);
    }
    CUdeviceptr d = 0;
    r = v.address_reserve(&d, size, 0, 0, 0);
    if (r != CUDA_SUCCESS) {
        v.release(h);
        return fail(SNK_ERR_CUDA, "cuMemAddressReserve: CUresult %d", (int)r);
    }
    r = v.map(d, size, 0, h, 0);
    CUmemAccessDesc acc = {};
    acc.location = prop.location;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    if (r == CUDA_SUCCESS) {
        r = v.set_access(d, size, &acc, 1);
        if (r != CUDA_SUCCESS) v.unmap(d, size);
    }
    if (r != CUDA_SUCCESS) {
        v.address_free(d, size);
        v.release(h);
        return fail(SNK_ERR_CUDA, "cuMemMap / cuMemSetAccess: CUresult %d", (int)r);
    }
    *p = (void *)d;
    *a = {h, size, device, true};
    return SNK_OK;
}

// ---- checkpoints (snk_env_* / snk_replay_* _checkpoint_bytes, _save_host, _load_host; DESIGN §5e) -----------------------
// Blob = header + raw device arrays.  The env arrays go in the order of EnvState, copied as they are in memory (also the lazily
// maintained chi of short snakes, which nobody reads), so a continued run's checkpoints equal an uninterrupted run's byte for byte.
constexpr uint32_t CKPT_VERSION = 1;
static const char kEnvMagic[8] = {'s', 'n', 'k', '-', 'e', 'n', 'v', 0};
static const char kReplayMagic[8] = {'s', 'n', 'k', '-', 'r', 'p', 'l', 0};
struct EnvCkptHeader {
    char magic[8];
    uint32_t version, flags;            // CKPT_VERSION; the snk_create flags
    int64_t n;
    uint64_t seed, step_counter;        // the internal generator's key and call count
    int32_t food_n, reserved;
    uint8_t food_rc[2 * MAX_FOOD];      // the food list, 1-based (row, col) pairs as snk_set_food_list_host takes it
};
struct ReplayCkptHeader {
    char magic[8];
    uint32_t version, record_bytes;
    int64_t capacity, total;            // transitions stored since the last clear
    uint64_t draws;                     // snk_replay_sample_indices calls so far
};
static_assert(sizeof(EnvCkptHeader) == 176 && sizeof(ReplayCkptHeader) == 40, "blob headers are part of the format");
constexpr size_t ENV_STATE_BYTES = 52;  // per env: occ pocc clo chi cons misc (u64) + ret (f32)
static const char *const kEnvRuleText[] = {
    "", "unused bits of misc set (error bits beyond 3, bits 56..63)", "head outside the board (the wall only for a lost env)",
    "tail not an interior cell", "food neither an interior cell nor the no-food code", "previous food neither an interior cell nor the no-food code",
    "length outside 2..64", "step count above 500 (499 for a live env)", "consumed food entries outside the food list",
    "previous direction is not the chain's last move", "direction chain leaves the board or crosses itself",
    "direction chain does not end on the tail", "occupancy disagrees with the direction chain"};
static const char *const kReplayRuleText[] = {"", "action index above 2", "done above 1", "mask bits above 7", "previous direction above 3"};

// the env arrays in blob order: device pointer and bytes per env
static void env_arrays(const EnvState &s, void *p[7], size_t b[7]) {
    void *q[7] = {s.occ, s.pocc, s.clo, s.chi, s.cons, s.misc, s.ret};
    for (int k = 0; k < 7; k++) { p[k] = q[k]; b[k] = k < 6 ? 8 : 4; }
}

// device scratch of a load: the validation result (8 bytes, set to ~0 = no failure) and, 256 bytes in, the blob's arrays;
// freed by the destructor on every path
struct LoadScratch {
    uint8_t *p = nullptr;
    ~LoadScratch() { if (p) cudaFree(p); }
    unsigned long long *first() const { return reinterpret_cast<unsigned long long *>(p); }
    uint8_t *data() const { return p + 256; }
};
static int load_scratch(LoadScratch &sc, const void *src_host, size_t bytes, cudaStream_t st) {
    SNK_CUDA(cudaMalloc((void **)&sc.p, 256 + bytes));
    SNK_CUDA(cudaMemsetAsync(sc.p, 0xFF, 8, st));
    if (bytes) SNK_CUDA(cudaMemcpyAsync(sc.data(), src_host, bytes, cudaMemcpyHostToDevice, st));
    return SNK_OK;
}
// the validation result: index of the lowest failing record (-1 if none) and its rule
static int load_verdict(const LoadScratch &sc, cudaStream_t st, long long *idx, int *rule) {
    SNK_CUDA(cudaGetLastError());
    unsigned long long f = 0;
    SNK_CUDA(cudaMemcpyAsync(&f, sc.first(), 8, cudaMemcpyDeviceToHost, st));
    SNK_CUDA(cudaStreamSynchronize(st));
    *idx = f == ~0ull ? -1 : (long long)(f >> 8);
    *rule = (int)(f & 0xFF);
    return SNK_OK;
}

extern "C" {

// profiling aid: device buffer of 8 int64 receiving cycle counts of CTA 0 of the small-batch rollout kernel
// ([0] logic warp total, [1] its wait for the consumers, [2] mask warp: wait for the logic warp, [3] mask warp: mask + scalars,
// [4] expansion warps: boards + expansion, [5] expansion warps: wait for the logic warp)
int snk_debug_rollout_timing(long long *device_buf) {
    g_rollout_prof = device_buf;
    return SNK_OK;
}

int snk_version(void) { return SNK_VERSION; }
const char *snk_last_error(void) { return err_buf(); }

int snk_default_food_list_host(uint8_t *cells_rc_host, int *n) {
    SNK_REQUIRE(cells_rc_host != nullptr && n != nullptr, "null argument");
    memcpy(cells_rc_host, kDefaultFoodRC, 100);
    *n = 50;
    return SNK_OK;
}

int snk_create(snk_handle *out, int64_t n_envs, int device, uint32_t flags) {
    SNK_REQUIRE(out != nullptr, "null out");
    SNK_REQUIRE(n_envs > 0 && n_envs <= (1ll << 31), "n_envs must be in 1..2^31");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(SNK_ERR_NODEVICE, "no CUDA device (%s); libsnake_b200 has no CPU fallback", cudaGetErrorString(e));
    SNK_REQUIRE(device >= 0 && device < ndev, "device index out of range");
    cudaDeviceProp prop;
    SNK_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(SNK_ERR_NODEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major,
                    prop.minor);
    DeviceGuard guard(device);
    snk_env *h = new (std::nothrow) snk_env();
    if (h == nullptr) return fail(SNK_ERR_INVALID, "out of host memory");
    memset(h, 0, sizeof(*h));
    h->n = n_envs; h->device = device; h->flags = flags; h->seed = 42;
    set_food(h->food, kDefaultFoodRC, 50);
    size_t n = (size_t)n_envs;
    cudaError_t ce = cudaSuccess;
    auto A = [&](void **p, size_t bytes) { if (ce == cudaSuccess) ce = cudaMalloc(p, bytes); };
    A((void **)&h->s.occ, 8 * n); A((void **)&h->s.pocc, 8 * n); A((void **)&h->s.clo, 8 * n);
    A((void **)&h->s.chi, 8 * n); A((void **)&h->s.cons, 8 * n); A((void **)&h->s.misc, 8 * n);
    A((void **)&h->s.ret, 4 * n); A((void **)&h->d_count, 8);
    if (ce == cudaSuccess) ce = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
    for (int i = 0; i < 2 && ce == cudaSuccess; i++) ce = cudaStreamCreateWithFlags(&h->copy_stream[i], cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&h->ev_in, cudaEventDisableTiming);
    if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&h->ev_done, cudaEventDisableTiming);
    for (int i = 0; i < 64 && ce == cudaSuccess; i++) ce = cudaEventCreateWithFlags(&h->ev_chunk[i], cudaEventDisableTiming);
    for (int i = 0; i < 64 && ce == cudaSuccess; i++) ce = cudaEventCreateWithFlags(&h->ev_up[i], cudaEventDisableTiming);
    if (ce != cudaSuccess) {
        int rc = fail(SNK_ERR_CUDA, "snk_create: %s", cudaGetErrorString(ce));
        snk_destroy(h);
        return rc;
    }
    h->stream = h->own_stream;
    k_reset<<<nblocks(h->n, 256), 256, 0, h->stream>>>(h->s, h->n);
    SNK_CUDA(cudaGetLastError());
    *out = h;
    return SNK_OK;
}

int snk_destroy(snk_handle h) {
    if (h == nullptr) return SNK_OK;
    DeviceGuard guard(h->device);
    if (h->own_stream) cudaStreamSynchronize(h->own_stream);
    for (int i = 0; i < 2; i++) if (h->copy_stream[i]) cudaStreamSynchronize(h->copy_stream[i]);
    void *ptrs[] = {h->s.occ, h->s.pocc, h->s.clo, h->s.chi, h->s.cons, h->s.misc, h->s.ret, h->d_count, h->d_q, h->d_u,
                    h->d_reward, h->d_ep_return, h->d_ridx, h->d_act, h->d_done, h->d_mask, h->d_ep_score, h->d_obs};
    for (void *p : ptrs) if (p) cudaFree(p);
    for (int i = 0; i < 2; i++) if (h->copy_stream[i]) cudaStreamDestroy(h->copy_stream[i]);
    if (h->ev_in) cudaEventDestroy(h->ev_in);
    if (h->ev_done) cudaEventDestroy(h->ev_done);
    for (int i = 0; i < 64; i++) if (h->ev_chunk[i]) cudaEventDestroy(h->ev_chunk[i]);
    for (int i = 0; i < 64; i++) if (h->ev_up[i]) cudaEventDestroy(h->ev_up[i]);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    delete h;
    return SNK_OK;
}

int snk_reset(snk_handle h) {
    SNK_CHECK_HANDLE(h);
    k_reset<<<nblocks(h->n, 256), 256, 0, h->stream>>>(h->s, h->n);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

int snk_set_food_list_host(snk_handle h, const uint8_t *cells_rc_host, int n) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(cells_rc_host != nullptr || n == 0, "null list");
    FoodTable ft;
    int rc = set_food(ft, cells_rc_host, n);
    if (rc != SNK_OK) return rc;
    SNK_CUDA(cudaStreamSynchronize(h->stream));   // kernels in flight carry the old table by value; just order the change
    h->food = ft;
    return SNK_OK;
}

int snk_set_stream(snk_handle h, void *cuda_stream) {
    SNK_CHECK_HANDLE(h);
    SNK_CUDA(cudaStreamSynchronize(h->stream));
    h->stream = (cudaStream_t)cuda_stream;
    return SNK_OK;
}
int snk_use_own_stream(snk_handle h) {
    SNK_CHECK_HANDLE(h);
    SNK_CUDA(cudaStreamSynchronize(h->stream));
    h->stream = h->own_stream;
    return SNK_OK;
}
int snk_get_stream(snk_handle h, void **cuda_stream) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(cuda_stream != nullptr, "null out");
    *cuda_stream = (void *)h->stream;
    return SNK_OK;
}
int snk_set_seed(snk_handle h, uint64_t seed) {
    SNK_CHECK_HANDLE(h);
    h->seed = seed; h->step_counter = 0;
    return SNK_OK;
}
int snk_sync(snk_handle h) {
    SNK_CHECK_HANDLE(h);
    SNK_CUDA(cudaStreamSynchronize(h->stream));
    SNK_CUDA(cudaStreamSynchronize(h->copy_stream[0]));       // device->host copies of the host-buffer entry points
    return SNK_OK;
}
int64_t snk_num_envs(snk_handle h) { return h ? h->n : 0; }

int snk_available_actions(snk_handle h, uint8_t *dirs_3xN) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(dirs_3xN != nullptr, "null out");
    k_available_actions<<<nblocks(h->n, 256), 256, 0, h->stream>>>(h->s, h->n, dirs_3xN);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

// launches the fused kernel for envs [begin, end) on `st`
static int launch_step(StepArgs &a, int obs_fmt, bool select, long long begin, long long end, cudaStream_t st) {
    a.env_begin = begin; a.env_end = end;
    unsigned grid = nblocks(end - begin, TPB);
    if (grid == 0) return SNK_OK;
    return launch_obs_fmt<SNK_OBS_NONE, SNK_OBS_F32, SNK_OBS_I8, SNK_OBS_I64, SNK_OBS_PACKED2, SNK_OBS_BITS>(obs_fmt, [&](auto fmt) {
        constexpr int FMT = decltype(fmt)::value;
        if (a.sink != nullptr) {
            if (select) k_step<FMT, true, true><<<grid, TPB, 0, st>>>(a);
            else k_step<FMT, false, true><<<grid, TPB, 0, st>>>(a);
        } else {
            if (select) k_step<FMT, true, false><<<grid, TPB, 0, st>>>(a);
            else k_step<FMT, false, false><<<grid, TPB, 0, st>>>(a);
        }
    });
}

// The arguments of a step of every env of h.  q != NULL: act_idx receives the selected actions, else it holds the input
// actions.  r != NULL: the step also stores every env's transition into the replay ring r.
static StepArgs step_args(snk_handle h, const float *q, float eps, const float *u, const uint8_t *ridx, uint8_t *act_idx,
                          const StepOutputs &out, const snk_replay_s *r) {
    StepArgs a;
    memset(&a, 0, sizeof(a));
    a.s = h->s; a.food = h->food; a.seed = h->seed; a.step_counter = h->step_counter;
    a.auto_reset = (h->flags & SNK_AUTO_RESET) ? 1 : 0;
    a.q = q; a.eps = eps; a.u = u; a.ridx = ridx;
    if (q != nullptr) a.act_out = act_idx; else a.act = act_idx;
    a.out = out;
    if (r != nullptr) { a.sink = r->ring; a.sink_base = r->total; a.sink_cap = r->capacity; a.sink_n = h->n; }
    return a;
}

// snk_step / snk_step_abs: the step without an observation
static int step_plain(snk_handle h, const uint8_t *act, int is_abs, float *reward, uint8_t *done) {
    StepArgs a = step_args(h, nullptr, 0.0f, nullptr, nullptr, nullptr, {reward, done}, nullptr);
    a.act = act; a.is_abs = is_abs;
    int rc = launch_step(a, SNK_OBS_NONE, false, 0, h->n, h->stream);
    h->step_counter++;
    return rc;
}

int snk_step(snk_handle h, const uint8_t *act_idx, float *reward, uint8_t *done) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(act_idx != nullptr, "null actions");
    return step_plain(h, act_idx, 0, reward, done);
}

int snk_step_abs(snk_handle h, const uint8_t *dir, float *reward, uint8_t *done) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(dir != nullptr, "null directions");
    return step_plain(h, dir, 1, reward, done);
}

// The argument checks of the fused step entry points; fn names the entry point in the messages.
static int check_step_inputs(const char *fn, const float *q, const uint8_t *act_idx, const void *obs, int obs_fmt) {
    if (q == nullptr && act_idx == nullptr) return fail(SNK_ERR_INVALID, "%s: need q (select) or act_idx (input)", fn);
    if (obs_fmt != SNK_OBS_NONE && obs == nullptr) return fail(SNK_ERR_INVALID, "%s: obs_fmt given without an obs buffer", fn);
    return SNK_OK;
}
// `what` names the store in the SNK_ERR_UNSUPPORTED message
static int check_replay(const char *fn, snk_handle h, const snk_replay_s *r, const char *what) {
    if (r->device != h->device) return fail(SNK_ERR_INVALID, "%s: replay ring and env live on different devices", fn);
    if (!(h->flags & SNK_AUTO_RESET))
        return fail(SNK_ERR_UNSUPPORTED, "%s needs an env created with SNK_AUTO_RESET (every env must step)", what);
    return SNK_OK;
}

// The fused step with DEVICE buffers; with a replay ring r the same kernel also store!s every transition into it.
static int step_fused_impl(const char *fn, snk_handle h, snk_replay_s *r, const float *q, float eps, const float *u,
                           const uint8_t *ridx, uint8_t *act_idx, float *reward, uint8_t *done, void *obs, int obs_fmt,
                           uint8_t *mask, float *ep_return, int32_t *ep_score) {
    if (h == nullptr) return fail(SNK_ERR_INVALID, "%s: null handle", fn);
    DeviceGuard guard(h->device);
    int rc = r != nullptr ? check_replay(fn, h, r, fn) : SNK_OK;
    if (rc == SNK_OK) rc = check_step_inputs(fn, q, act_idx, obs, obs_fmt);
    if (rc != SNK_OK) return rc;
    if (obs_fmt != SNK_OBS_NONE && ((uintptr_t)obs & 15u) != 0) return fail(SNK_ERR_INVALID, "%s: obs must be 16-byte aligned", fn);
    StepArgs a = step_args(h, q, eps, u, ridx, act_idx, {reward, done, obs, mask, ep_return, ep_score}, r);
    rc = launch_step(a, obs ? obs_fmt : SNK_OBS_NONE, q != nullptr, 0, h->n, h->stream);
    h->step_counter++;
    if (rc == SNK_OK && r != nullptr) r->total += h->n;
    return rc;
}

int snk_step_fused(snk_handle h, const float *q, float eps, const float *u, const uint8_t *ridx, uint8_t *act_idx,
                   float *reward, uint8_t *done, void *obs, int obs_fmt, uint8_t *mask, float *ep_return,
                   int32_t *ep_score) {
    return step_fused_impl(__func__, h, nullptr, q, eps, u, ridx, act_idx, reward, done, obs, obs_fmt, mask, ep_return, ep_score);
}

int snk_rollout_fused(snk_handle h, const uint8_t *act_TxN, int64_t T, int is_abs, float *reward, uint8_t *done, void *obs,
                      int obs_fmt, uint8_t *mask, float *ep_return, int32_t *ep_score) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(act_TxN != nullptr && T > 0 && T <= (1 << 20), "bad argument");
    SNK_REQUIRE(obs_fmt == SNK_OBS_NONE || obs != nullptr, "obs_fmt given without an obs buffer");
    SNK_REQUIRE(obs == nullptr || ((uintptr_t)obs & 15u) == 0, "obs must be 16-byte aligned");
    RolloutArgs a;
    memset(&a, 0, sizeof(a));
    a.s = h->s; a.food = h->food; a.act = act_TxN; a.out = {reward, done, obs, mask, ep_return, ep_score};
    a.n = h->n; a.steps = (int)T; a.is_abs = is_abs;
    a.prof = g_rollout_prof;
    a.auto_reset = (h->flags & SNK_AUTO_RESET) ? 1 : 0;
    // small batches: the warp-specialised kernel, WS_EPB envs per CTA (4,096 envs -> 256 CTAs over the 148 SMs)
    const bool small = h->n <= 32 * 1024;
    const int rc = launch_obs_fmt<SNK_OBS_NONE, SNK_OBS_F32, SNK_OBS_I8, SNK_OBS_I64, SNK_OBS_PACKED2>(
        obs ? obs_fmt : SNK_OBS_NONE, [&](auto fmt) {
            constexpr int FMT = decltype(fmt)::value;
            if (small) k_rollout_ws<FMT, WS_EPB><<<nblocks(h->n, WS_EPB), WS_THREADS, 0, h->stream>>>(a);
            else k_rollout<FMT, RTPB><<<nblocks(h->n, RTPB), RTPB, 0, h->stream>>>(a);
        });
    if (rc == SNK_OK) h->step_counter += (u64)T;
    return rc;
}

int snk_host_alloc(void **p, size_t bytes) {
    SNK_REQUIRE(p != nullptr, "null out");
    SNK_CUDA(cudaMallocHost(p, bytes));
    return SNK_OK;
}
int snk_host_free(void *p) {
    if (p) SNK_CUDA(cudaFreeHost(p));
    return SNK_OK;
}

int snk_compression_supported(int device, int *yes) {
    SNK_REQUIRE(yes != nullptr, "null out");
    *yes = 0;
    int ndev = 0;
    SNK_CUDA(cudaGetDeviceCount(&ndev));
    SNK_REQUIRE(device >= 0 && device < ndev, "device index out of range");
    DeviceGuard guard(device);
    const Vmm *v = nullptr;
    if (vmm_api(&v) != SNK_OK) return SNK_OK;             // a driver without the virtual-memory entry points: no compression
    return vmm_compression_supported(*v, device, yes);
}

int snk_device_alloc(void **p, size_t bytes, int device, uint32_t flags, int *compressible) {
    SNK_REQUIRE(p != nullptr && bytes > 0, "bad argument");
    SNK_REQUIRE((flags & ~SNK_ALLOC_COMPRESSIBLE) == 0u, "unknown flag");
    *p = nullptr;
    if (compressible != nullptr) *compressible = 0;
    int ndev = 0;
    SNK_CUDA(cudaGetDeviceCount(&ndev));
    SNK_REQUIRE(device >= 0 && device < ndev, "device index out of range");
    DeviceGuard guard(device);
    DevAlloc a = {0, bytes, device, false};
    if (flags & SNK_ALLOC_COMPRESSIBLE) {
        int yes = 0;
        int rc = snk_compression_supported(device, &yes);
        if (rc != SNK_OK) return rc;
        if (yes) {
            const Vmm *v = nullptr;
            rc = vmm_api(&v);
            if (rc == SNK_OK) rc = vmm_alloc_compressible(*v, device, bytes, p, &a);
            if (rc != SNK_OK) return rc;
        }
    }
    if (*p == nullptr) SNK_CUDA(cudaMalloc(p, bytes));     // not requested, not supported, or the driver gave plain memory
    {
        std::lock_guard<std::mutex> lk(g_dev_allocs_mu);
        g_dev_allocs[*p] = a;
    }
    if (compressible != nullptr) *compressible = a.vmm ? 1 : 0;
    return SNK_OK;
}

int snk_device_free(void *p) {
    if (p == nullptr) return SNK_OK;
    DevAlloc a;
    {
        std::lock_guard<std::mutex> lk(g_dev_allocs_mu);
        auto it = g_dev_allocs.find(p);
        SNK_REQUIRE(it != g_dev_allocs.end(), "pointer was not returned by snk_device_alloc (or was freed already)");
        a = it->second;
    }
    // the entry is dropped only once the memory is given back: after a failed call (a device synchronise refused during a
    // stream capture, a sticky error) the pointer stays registered and the call can be repeated
    DeviceGuard guard(a.device);
    if (!a.vmm) {
        SNK_CUDA(cudaFree(p));
    } else {
        SNK_CUDA(cudaDeviceSynchronize());                // unmapping does not wait for kernels that may still write the range
        const Vmm *v = nullptr;
        int rc = vmm_api(&v);
        if (rc != SNK_OK) return rc;
        const CUdeviceptr d = (CUdeviceptr)p;
        CUresult r = v->unmap(d, a.size);
        if (r == CUDA_SUCCESS) r = v->address_free(d, a.size);
        if (r == CUDA_SUCCESS) r = v->release(a.handle);
        if (r != CUDA_SUCCESS) return fail(SNK_ERR_CUDA, "snk_device_free: CUresult %d", (int)r);
    }
    std::lock_guard<std::mutex> lk(g_dev_allocs_mu);
    g_dev_allocs.erase(p);
    return SNK_OK;
}

int snk_state(snk_handle h, void *obs, int obs_fmt) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(obs != nullptr, "null out");
    SNK_REQUIRE(((uintptr_t)obs & 15u) == 0, "obs must be 16-byte aligned");
    return launch_obs_fmt<SNK_OBS_F32, SNK_OBS_I8, SNK_OBS_I64, SNK_OBS_PACKED2, SNK_OBS_BITS>(obs_fmt, [&](auto fmt) {
        k_state<decltype(fmt)::value><<<nblocks(h->n, TPB), TPB, 0, h->stream>>>(h->s, h->n, obs);
    });
}

int snk_patch_reset_obs(snk_handle h, const uint8_t *done, void *obs, int obs_fmt) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(done != nullptr && obs != nullptr, "null argument");
    SNK_REQUIRE(((uintptr_t)obs & 15u) == 0, "obs must be 16-byte aligned");
    if (!(h->flags & SNK_AUTO_RESET)) return SNK_OK;          // frozen envs keep their terminal state
    return launch_obs_fmt<SNK_OBS_F32, SNK_OBS_I8, SNK_OBS_I64, SNK_OBS_PACKED2, SNK_OBS_BITS>(obs_fmt, [&](auto fmt) {
        k_patch_reset<decltype(fmt)::value><<<nblocks(h->n, TPB), TPB, 0, h->stream>>>(h->n, done, obs);
    });
}

int snk_losing_mask(snk_handle h, uint8_t *mask_3xN) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(mask_3xN != nullptr, "null out");
    k_losing_mask<<<nblocks(h->n, 256), 256, 0, h->stream>>>(h->s, h->n, mask_3xN, h->food);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

int snk_select_action(snk_handle h, const float *q_3xN, float eps, const float *u, const uint8_t *ridx,
                      uint8_t *act_idx_out) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(q_3xN != nullptr && act_idx_out != nullptr, "null argument");
    k_select<<<nblocks(h->n, 256), 256, 0, h->stream>>>(h->n, q_3xN, eps, u, ridx, h->seed, h->step_counter, act_idx_out);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

int snk_masked_target(const float *q_next_3xB, const uint8_t *mask_3xB, const float *r, const uint8_t *done, double gamma,
                      float fill, double *y_f64, float *y_f32, int64_t B, void *cuda_stream) {
    DeviceGuard guard__(device_of(q_next_3xB));
    SNK_REQUIRE(q_next_3xB && mask_3xB && r && done, "null input");
    SNK_REQUIRE(y_f64 || y_f32, "no output requested");
    SNK_REQUIRE(B >= 0, "negative batch");
    if (B == 0) return SNK_OK;
    k_masked_target<<<nblocks(B, 256), 256, 0, (cudaStream_t)cuda_stream>>>(q_next_3xB, mask_3xB, r, done, gamma, fill,
                                                                          y_f64, y_f32, B);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

static int scalars(snk_handle h, int which, void *out) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(out != nullptr, "null out");
    k_scalars<<<nblocks(h->n, 256), 256, 0, h->stream>>>(h->s, h->n, which, out);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}
int snk_get_score(snk_handle h, int32_t *score) { return scalars(h, 0, score); }
int snk_get_done(snk_handle h, uint8_t *done) { return scalars(h, 1, done); }
int snk_get_error_flags(snk_handle h, uint8_t *flags) { return scalars(h, 2, flags); }
int snk_get_steps(snk_handle h, int32_t *steps) { return scalars(h, 3, steps); }

int snk_count_errors_host(snk_handle h, int64_t *count) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(count != nullptr, "null out");
    SNK_CUDA(cudaMemsetAsync(h->d_count, 0, 8, h->stream));
    k_count_errors<<<nblocks(h->n, 256), 256, 0, h->stream>>>(h->s, h->n, h->d_count);
    SNK_CUDA(cudaGetLastError());
    unsigned long long c = 0;
    SNK_CUDA(cudaMemcpyAsync(&c, h->d_count, 8, cudaMemcpyDeviceToHost, h->stream));
    SNK_CUDA(cudaStreamSynchronize(h->stream));
    *count = (int64_t)c;
    return SNK_OK;
}


// ---- replay ring (ReplayBuffer, structs.jl:104-116; store!/sample/stack_exp, utils.jl:265-383) ----------
int snk_replay_create(snk_replay *out, int64_t capacity, int device) {
    SNK_REQUIRE(out != nullptr, "null out");
    SNK_REQUIRE(capacity >= 64, "batch_size (64) cannot be greater than the capacity of the buffer");   // structs.jl:113
    *out = nullptr;
    DeviceGuard guard(device);
    snk_replay_s *r = new (std::nothrow) snk_replay_s();
    if (r == nullptr) return fail(SNK_ERR_INVALID, "out of host memory");
    memset(r, 0, sizeof(*r));
    r->capacity = capacity; r->device = device;
    cudaError_t e = cudaMalloc((void **)&r->ring, (size_t)capacity * 128);
    if (e == cudaSuccess) e = cudaMalloc((void **)&r->d_bad, sizeof(int));
    if (e == cudaSuccess) e = cudaMemset(r->d_bad, 0, sizeof(int));
    if (e != cudaSuccess) {
        if (r->ring) cudaFree(r->ring);
        delete r;
        return fail(SNK_ERR_CUDA, "snk_replay_create: %s", cudaGetErrorString(e));
    }
    *out = r;
    return SNK_OK;
}
int snk_replay_destroy(snk_replay r) {
    if (r == nullptr) return SNK_OK;
    DeviceGuard guard(r->device);
    cudaFree(r->ring);
    cudaFree(r->d_bad);
    if (r->stage) cudaFree(r->stage);
    delete r;
    return SNK_OK;
}
int snk_replay_clear(snk_replay r) {                      // empty_buffer!, utils.jl:311-314
    SNK_REQUIRE(r != nullptr, "null replay");
    r->total = 0;
    return SNK_OK;
}
int snk_replay_length(snk_replay r, int64_t *length, int64_t *position) {
    SNK_REQUIRE(r != nullptr, "null replay");
    if (length) *length = r->total < r->capacity ? r->total : r->capacity;
    // rpb.position (1-based) only advances once the buffer is full (utils.jl:268-276)
    if (position) *position = r->total < r->capacity ? 1 : ((r->total - r->capacity) % r->capacity) + 1;
    return SNK_OK;
}

int snk_step_fused_store(snk_handle h, snk_replay r, const float *q, float eps, const float *u, const uint8_t *ridx,
                         uint8_t *act_idx, float *reward, uint8_t *done, void *obs, int obs_fmt, uint8_t *mask,
                         float *ep_return, int32_t *ep_score) {
    SNK_REQUIRE(r != nullptr, "null replay");
    return step_fused_impl(__func__, h, r, q, eps, u, ridx, act_idx, reward, done, obs, obs_fmt, mask, ep_return, ep_score);
}

int snk_replay_gather(snk_replay r, const int64_t *idx, int64_t B, float *states, float *next_states, uint8_t *actions,
                      float *rewards, uint8_t *dones, uint8_t *mask, float *ep_return, int32_t *score, void *cuda_stream) {
    SNK_REQUIRE(r != nullptr && idx != nullptr && B >= 0, "bad argument");
    SNK_REQUIRE((((uintptr_t)states | (uintptr_t)next_states) & 15u) == 0, "state buffers must be 16-byte aligned");
    if (B == 0) return SNK_OK;
    DeviceGuard guard(r->device);
    k_replay_gather<<<nblocks(B, GATHER_S), 128, 0, (cudaStream_t)cuda_stream>>>(
        r->ring, r->capacity, (const long long *)idx, B, states, next_states, actions, rewards, dones, mask, ep_return,
        score, r->d_bad);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

int snk_replay_sample_indices(snk_replay r, uint64_t seed, int64_t B, int64_t *idx_out, void *cuda_stream) {
    SNK_REQUIRE(r != nullptr && idx_out != nullptr, "bad argument");
    const long long n = r->total < r->capacity ? r->total : r->capacity;
    // sample(rpb): min(batch, length) distinct transitions (utils.jl:280-287)
    SNK_REQUIRE(B >= 0 && B <= n, "cannot sample more distinct transitions than the buffer holds");
    if (B == 0) return SNK_OK;
    DeviceGuard guard(r->device);
    const u64 key = splitmix64(seed ^ splitmix64(r->draws++));
    k_replay_sample<<<nblocks(B, 256), 256, 0, (cudaStream_t)cuda_stream>>>(n, B, key, (long long *)idx_out);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

int snk_replay_bad_index_host(snk_replay r, int *flag) {
    SNK_REQUIRE(r != nullptr && flag != nullptr, "bad argument");
    DeviceGuard guard(r->device);
    SNK_CUDA(cudaMemcpy(flag, r->d_bad, sizeof(int), cudaMemcpyDeviceToHost));
    return SNK_OK;
}

// ---- host-buffer forms ------------------------------------------------------------------------------------
// The fused step with HOST buffers: env chunks are pipelined three deep — the inputs of chunk c+1 go up on one copy
// stream while the kernel of chunk c runs and the outputs of chunk c-1 come down on the other (PCIe is full duplex).
// With a replay ring the same kernels also store! every transition into it (utils.jl:267-277).
static int step_fused_host_impl(snk_handle h, snk_replay_s *r, const float *q, float eps, const float *u, const uint8_t *ridx,
                                uint8_t *act_idx, float *reward, uint8_t *done, void *obs, int obs_fmt, uint8_t *mask,
                                float *ep_return, int32_t *ep_score) {
    SNK_CHECK_HANDLE(h);
    int rc = check_step_inputs(__func__, q, act_idx, obs, obs_fmt);
    if (rc == SNK_OK && r != nullptr) rc = check_replay(__func__, h, r, "storing transitions");
    if (rc != SNK_OK) return rc;
    const size_t n = (size_t)h->n;
    const size_t opb = obs ? obs_bytes(obs_fmt) : 0;
    if (obs && opb == 0) return fail(SNK_ERR_INVALID, "unknown obs_fmt %d", obs_fmt);
    // device staging
    SNK_CUDA(ensure(&h->d_act, n));
    if (q) { SNK_CUDA(ensure(&h->d_q, 12 * n)); }
    if (u) { SNK_CUDA(ensure(&h->d_u, 4 * n)); }
    if (ridx) { SNK_CUDA(ensure(&h->d_ridx, n)); }
    if (reward) { SNK_CUDA(ensure(&h->d_reward, 4 * n)); }
    if (done) { SNK_CUDA(ensure(&h->d_done, n)); }
    if (mask) { SNK_CUDA(ensure(&h->d_mask, 3 * n)); }
    if (ep_return) { SNK_CUDA(ensure(&h->d_ep_return, 4 * n)); }
    if (ep_score) { SNK_CUDA(ensure(&h->d_ep_score, 4 * n)); }
    if (opb && (rc = ensure_obs_staging(h, opb * n)) != SNK_OK) return rc;
    if ((rc = staging_guard(h)) != SNK_OK) return rc;
    cudaStream_t st = h->stream, down = h->copy_stream[0], up = h->copy_stream[1];
    StepArgs a = step_args(h, q ? h->d_q : nullptr, eps, u ? h->d_u : nullptr, ridx ? h->d_ridx : nullptr, act_idx ? h->d_act : nullptr,
                           {reward ? h->d_reward : nullptr, done ? h->d_done : nullptr, opb ? h->d_obs : nullptr,
                            mask ? h->d_mask : nullptr, ep_return ? h->d_ep_return : nullptr, ep_score ? h->d_ep_score : nullptr},
                           r);
    // Chunking trades copy/kernel overlap (and the time before the first output copy can start) against per-copy overhead
    // (~8 us per cudaMemcpyAsync): about SNK_HOST_CHUNK_MB of traffic per chunk, at most 16 chunks; only the observation is copied per chunk, the small per-env outputs go down once at the end.
    // (A first chunk of 1/8 size, so that the output copies start earlier, was A/B-measured on one box: 1.365 against 1.363 ms
    // per step — the step is bound by the device->host transfer itself, 62 MB at ~47 GB/s with the uploads running beside it.)
    const long long align = TPB * 8;
    const size_t traffic = (opb + 26) * n;
    int n_chunks = (int)((traffic + (SNK_HOST_CHUNK_MB << 20) - 1) / (SNK_HOST_CHUNK_MB << 20));
    if (n_chunks < 1) n_chunks = 1;
    if (n_chunks > 16) n_chunks = 16;
    const long long per = ((h->n + n_chunks - 1) / n_chunks + align - 1) / align * align;
    // the staging buffers may still be read by earlier work on the handle's stream
    SNK_CUDA(cudaEventRecord(h->ev_in, st));
    SNK_CUDA(cudaStreamWaitEvent(up, h->ev_in, 0));
    int ci = 0;
    for (long long b = 0; b < h->n; b += per, ci++) {
        const long long e = b + per < h->n ? b + per : h->n;
        const size_t nb = (size_t)(e - b);
        if (q) SNK_CUDA(cudaMemcpyAsync(h->d_q + 3 * b, q + 3 * b, 12 * nb, cudaMemcpyHostToDevice, up));
        if (u) SNK_CUDA(cudaMemcpyAsync(h->d_u + b, u + b, 4 * nb, cudaMemcpyHostToDevice, up));
        if (ridx) SNK_CUDA(cudaMemcpyAsync(h->d_ridx + b, ridx + b, nb, cudaMemcpyHostToDevice, up));
        if (!q) SNK_CUDA(cudaMemcpyAsync(h->d_act + b, act_idx + b, nb, cudaMemcpyHostToDevice, up));
        SNK_CUDA(cudaEventRecord(h->ev_up[ci], up));
        SNK_CUDA(cudaStreamWaitEvent(st, h->ev_up[ci], 0));
        if ((rc = launch_step(a, opb ? obs_fmt : SNK_OBS_NONE, q != nullptr, b, e, st)) != SNK_OK) return rc;
        SNK_CUDA(cudaEventRecord(h->ev_chunk[ci], st));
        SNK_CUDA(cudaStreamWaitEvent(down, h->ev_chunk[ci], 0));
        if (opb) SNK_CUDA(cudaMemcpyAsync((char *)obs + opb * b, (char *)h->d_obs + opb * b, opb * nb, cudaMemcpyDeviceToHost, down));
    }
    // `down` has waited for the last kernel: every per-env output is complete
    if (mask) SNK_CUDA(cudaMemcpyAsync(mask, h->d_mask, 3 * n, cudaMemcpyDeviceToHost, down));
    if (reward) SNK_CUDA(cudaMemcpyAsync(reward, h->d_reward, 4 * n, cudaMemcpyDeviceToHost, down));
    if (done) SNK_CUDA(cudaMemcpyAsync(done, h->d_done, n, cudaMemcpyDeviceToHost, down));
    if (ep_return) SNK_CUDA(cudaMemcpyAsync(ep_return, h->d_ep_return, 4 * n, cudaMemcpyDeviceToHost, down));
    if (ep_score) SNK_CUDA(cudaMemcpyAsync(ep_score, h->d_ep_score, 4 * n, cudaMemcpyDeviceToHost, down));
    if (q && act_idx) SNK_CUDA(cudaMemcpyAsync(act_idx, h->d_act, n, cudaMemcpyDeviceToHost, down));
    h->step_counter++;
    if (r != nullptr) r->total += h->n;
    // snk_sync() waits for these copies; the handle's stream itself does not (see staging_guard)
    SNK_CUDA(cudaEventRecord(h->ev_done, down));
    return SNK_OK;
}

int snk_step_fused_host(snk_handle h, const float *q, float eps, const float *u, const uint8_t *ridx, uint8_t *act_idx,
                        float *reward, uint8_t *done, void *obs, int obs_fmt, uint8_t *mask, float *ep_return,
                        int32_t *ep_score) {
    return step_fused_host_impl(h, nullptr, q, eps, u, ridx, act_idx, reward, done, obs, obs_fmt, mask, ep_return, ep_score);
}

int snk_step_fused_store_host(snk_handle h, snk_replay r, const float *q, float eps, const float *u, const uint8_t *ridx,
                              uint8_t *act_idx, float *reward, uint8_t *done, void *obs, int obs_fmt, uint8_t *mask,
                              float *ep_return, int32_t *ep_score) {
    SNK_REQUIRE(r != nullptr, "null replay");
    return step_fused_host_impl(h, r, q, eps, u, ridx, act_idx, reward, done, obs, obs_fmt, mask, ep_return, ep_score);
}

// Per-call getters with HOST outputs (any host memory; pinned is faster).  Unlike the enqueue-and-return entry points these
// return when the data has arrived: they are what a Julia host calls where the reference reads a field of `game`.
int snk_state_host(snk_handle h, void *obs_host, int obs_fmt) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(obs_host != nullptr, "null out");
    const size_t opb = obs_bytes(obs_fmt);
    if (opb == 0) return fail(SNK_ERR_INVALID, "unknown obs_fmt %d", obs_fmt);
    return get_host(h, obs_host, opb * (size_t)h->n, [&](void *d) { return snk_state(h, d, obs_fmt); });
}

int snk_losing_mask_host(snk_handle h, uint8_t *mask_3xN_host) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(mask_3xN_host != nullptr, "null out");
    return get_host(h, mask_3xN_host, 3 * (size_t)h->n, [&](void *d) { return snk_losing_mask(h, (uint8_t *)d); });
}

int snk_available_actions_host(snk_handle h, uint8_t *dirs_3xN_host) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(dirs_3xN_host != nullptr, "null out");
    return get_host(h, dirs_3xN_host, 3 * (size_t)h->n, [&](void *d) { return snk_available_actions(h, (uint8_t *)d); });
}

static int scalars_host(snk_handle h, int which, void *out_host, size_t elem) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(out_host != nullptr, "null out");
    return get_host(h, out_host, elem * (size_t)h->n, [&](void *d) { return scalars(h, which, d); });
}
int snk_get_score_host(snk_handle h, int32_t *score_host) { return scalars_host(h, 0, score_host, 4); }
int snk_get_done_host(snk_handle h, uint8_t *done_host) { return scalars_host(h, 1, done_host, 1); }
int snk_get_error_flags_host(snk_handle h, uint8_t *flags_host) { return scalars_host(h, 2, flags_host, 1); }
int snk_get_steps_host(snk_handle h, int32_t *steps_host) { return scalars_host(h, 3, steps_host, 4); }

// stack_exp (utils.jl:343-383) with HOST outputs for idx_host[0..B) (0-based slots): the sampled transitions are expanded to
// Float32 on the device and copied down (2 x 800 B + 13 B per sample); returns when the data has arrived.
int snk_replay_gather_host(snk_replay r, const int64_t *idx_host, int64_t B, float *states, float *next_states, uint8_t *actions,
                           float *rewards, uint8_t *dones, uint8_t *mask, void *cuda_stream) {
    SNK_REQUIRE(r != nullptr && idx_host != nullptr && B >= 0, "bad argument");
    if (B == 0) return SNK_OK;
    DeviceGuard guard(r->device);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const size_t need = (size_t)B * 1632 + 256;     // 2 x 800 B of states + 8 idx + 4 + 1 + 1 + 3 per sample
    if (r->stage_bytes < need) {
        if (r->stage) { SNK_CUDA(cudaStreamSynchronize(st)); SNK_CUDA(cudaFree(r->stage)); r->stage = nullptr; r->stage_bytes = 0; }
        SNK_CUDA(cudaMalloc((void **)&r->stage, need));
        r->stage_bytes = need;
    }
    // staging layout: states | next_states | idx | rewards | actions | dones | mask
    uint8_t *base = r->stage;
    float *d_s = (float *)base, *d_ns = d_s + 200 * B;
    int64_t *d_idx = (int64_t *)(d_ns + 200 * B);
    float *d_rw = (float *)(d_idx + B);
    uint8_t *d_act = (uint8_t *)(d_rw + B), *d_dn = d_act + B, *d_mk = d_dn + B;
    SNK_CUDA(cudaMemcpyAsync(d_idx, idx_host, 8 * (size_t)B, cudaMemcpyHostToDevice, st));
    int rc = snk_replay_gather(r, d_idx, B, states ? d_s : nullptr, next_states ? d_ns : nullptr, actions ? d_act : nullptr,
                               rewards ? d_rw : nullptr, dones ? d_dn : nullptr, mask ? d_mk : nullptr, nullptr, nullptr, cuda_stream);
    if (rc != SNK_OK) return rc;
    if (states) SNK_CUDA(cudaMemcpyAsync(states, d_s, 800 * (size_t)B, cudaMemcpyDeviceToHost, st));
    if (next_states) SNK_CUDA(cudaMemcpyAsync(next_states, d_ns, 800 * (size_t)B, cudaMemcpyDeviceToHost, st));
    if (rewards) SNK_CUDA(cudaMemcpyAsync(rewards, d_rw, 4 * (size_t)B, cudaMemcpyDeviceToHost, st));
    if (actions) SNK_CUDA(cudaMemcpyAsync(actions, d_act, (size_t)B, cudaMemcpyDeviceToHost, st));
    if (dones) SNK_CUDA(cudaMemcpyAsync(dones, d_dn, (size_t)B, cudaMemcpyDeviceToHost, st));
    if (mask) SNK_CUDA(cudaMemcpyAsync(mask, d_mk, 3 * (size_t)B, cudaMemcpyDeviceToHost, st));
    SNK_CUDA(cudaStreamSynchronize(st));
    return SNK_OK;
}

// ---- checkpoints: save_trainer / load_trainer (utils.jl:408-418), save_buffer / load_buffer (utils.jl:316-340) -----------
int snk_env_checkpoint_bytes(snk_handle h, size_t *bytes) {
    if (h == nullptr || bytes == nullptr) return fail(SNK_ERR_INVALID, "%s: null argument", __func__);
    *bytes = sizeof(EnvCkptHeader) + ENV_STATE_BYTES * (size_t)h->n;
    return SNK_OK;
}

int snk_env_save_host(snk_handle h, void *blob_host, size_t bytes) {
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(blob_host != nullptr, "null blob");
    size_t need = 0;
    snk_env_checkpoint_bytes(h, &need);
    if (bytes != need) return fail(SNK_ERR_INVALID, "%s: blob of %zu bytes, the checkpoint has %zu", __func__, bytes, need);
    EnvCkptHeader hd;
    memset(&hd, 0, sizeof(hd));
    memcpy(hd.magic, kEnvMagic, 8);
    hd.version = CKPT_VERSION; hd.flags = h->flags; hd.n = h->n; hd.seed = h->seed; hd.step_counter = h->step_counter;
    hd.food_n = h->food.n;
    for (int i = 0; i < h->food.n; i++) {
        hd.food_rc[2 * i] = (uint8_t)((h->food.bit[i] & 7) + 2);
        hd.food_rc[2 * i + 1] = (uint8_t)((h->food.bit[i] >> 3) + 2);
    }
    memcpy(blob_host, &hd, sizeof(hd));
    void *p[7];
    size_t b[7];
    env_arrays(h->s, p, b);
    uint8_t *dst = (uint8_t *)blob_host + sizeof(hd);
    for (int k = 0; k < 7; k++) {
        SNK_CUDA(cudaMemcpyAsync(dst, p[k], b[k] * (size_t)h->n, cudaMemcpyDeviceToHost, h->stream));
        dst += b[k] * (size_t)h->n;
    }
    SNK_CUDA(cudaStreamSynchronize(h->stream));
    return SNK_OK;
}

int snk_env_load_host(snk_handle h, const void *blob_host, size_t bytes, int64_t *first_bad_env) {
    if (first_bad_env != nullptr) *first_bad_env = -1;
    SNK_CHECK_HANDLE(h);
    SNK_REQUIRE(blob_host != nullptr, "null blob");
    EnvCkptHeader hd;
    if (bytes < sizeof(hd))
        return fail(SNK_ERR_INVALID, "%s: truncated blob: %zu bytes, the header alone has %zu", __func__, bytes, sizeof(hd));
    memcpy(&hd, blob_host, sizeof(hd));
    if (memcmp(hd.magic, kEnvMagic, 8) != 0) return fail(SNK_ERR_INVALID, "%s: not an env checkpoint (wrong magic)", __func__);
    if (hd.version != CKPT_VERSION)
        return fail(SNK_ERR_INVALID, "%s: checkpoint format version %u, this library reads %u", __func__, hd.version, CKPT_VERSION);
    if (hd.n != h->n) return fail(SNK_ERR_INVALID, "%s: checkpoint of %lld envs, the handle has %lld", __func__, (long long)hd.n, h->n);
    if ((hd.flags ^ h->flags) & SNK_AUTO_RESET)
        return fail(SNK_ERR_INVALID, "%s: checkpoint %s SNK_AUTO_RESET, the handle %s", __func__, (hd.flags & SNK_AUTO_RESET) ? "has" : "lacks",
                    (h->flags & SNK_AUTO_RESET) ? "has it" : "does not");
    const size_t arrays = ENV_STATE_BYTES * (size_t)h->n;
    if (bytes != sizeof(hd) + arrays)
        return fail(SNK_ERR_INVALID, "%s: blob of %zu bytes, a checkpoint of %lld envs has %zu", __func__, bytes, h->n, sizeof(hd) + arrays);
    FoodTable ft;
    if (set_food(ft, hd.food_rc, hd.food_n) != SNK_OK) {
        char why[512];
        snprintf(why, sizeof(why), "%s", err_buf());
        return fail(SNK_ERR_INVALID, "%s: the checkpoint's food list: %s", __func__, why);
    }
    // the blob's arrays into device scratch, validated there; the live state is touched only if every env passes
    LoadScratch sc;
    int rc = load_scratch(sc, (const uint8_t *)blob_host + sizeof(hd), arrays, h->stream);
    if (rc != SNK_OK) return rc;
    EnvState s;
    void *p[7], *q[7];
    size_t b[7];
    uint8_t *src = sc.data();
    for (int k = 0; k < 7; k++) { q[k] = src; src += (k < 6 ? 8 : 4) * (size_t)h->n; }
    s.occ = (u64 *)q[0]; s.pocc = (u64 *)q[1]; s.clo = (u64 *)q[2]; s.chi = (u64 *)q[3]; s.cons = (u64 *)q[4]; s.misc = (u64 *)q[5];
    s.ret = (float *)q[6];
    k_env_validate<<<nblocks(h->n, 256), 256, 0, h->stream>>>(s, h->n, ft.mask(), sc.first());
    long long bad = -1;
    int rule = 0;
    if ((rc = load_verdict(sc, h->stream, &bad, &rule)) != SNK_OK) return rc;
    if (bad >= 0) {
        if (first_bad_env != nullptr) *first_bad_env = bad;
        return fail(SNK_ERR_INVALID, "%s: env %lld of the checkpoint: %s", __func__, bad,
                    rule < (int)(sizeof(kEnvRuleText) / sizeof(kEnvRuleText[0])) ? kEnvRuleText[rule] : "?");
    }
    env_arrays(h->s, p, b);
    for (int k = 0; k < 7; k++) SNK_CUDA(cudaMemcpyAsync(p[k], q[k], b[k] * (size_t)h->n, cudaMemcpyDeviceToDevice, h->stream));
    SNK_CUDA(cudaStreamSynchronize(h->stream));
    h->seed = hd.seed;
    h->step_counter = hd.step_counter;
    h->food = ft;
    return SNK_OK;
}

int snk_replay_checkpoint_bytes(snk_replay r, size_t *bytes) {
    if (r == nullptr || bytes == nullptr) return fail(SNK_ERR_INVALID, "%s: null argument", __func__);
    const long long filled = r->total < r->capacity ? r->total : r->capacity;
    *bytes = sizeof(ReplayCkptHeader) + (size_t)filled * 128;
    return SNK_OK;
}

int snk_replay_save_host(snk_replay r, void *blob_host, size_t bytes) {
    SNK_REQUIRE(r != nullptr && blob_host != nullptr, "null argument");
    size_t need = 0;
    snk_replay_checkpoint_bytes(r, &need);
    if (bytes != need) return fail(SNK_ERR_INVALID, "%s: blob of %zu bytes, the checkpoint has %zu", __func__, bytes, need);
    DeviceGuard guard(r->device);
    ReplayCkptHeader hd;
    memset(&hd, 0, sizeof(hd));
    memcpy(hd.magic, kReplayMagic, 8);
    hd.version = CKPT_VERSION; hd.record_bytes = 128; hd.capacity = r->capacity; hd.total = r->total; hd.draws = r->draws;
    memcpy(blob_host, &hd, sizeof(hd));
    SNK_CUDA(cudaDeviceSynchronize());                     // the steps that store into the ring run on the env's stream
    if (bytes > sizeof(hd)) SNK_CUDA(cudaMemcpy((uint8_t *)blob_host + sizeof(hd), r->ring, bytes - sizeof(hd), cudaMemcpyDeviceToHost));
    return SNK_OK;
}

int snk_replay_load_host(snk_replay r, const void *blob_host, size_t bytes, int64_t *first_bad_slot) {
    if (first_bad_slot != nullptr) *first_bad_slot = -1;
    SNK_REQUIRE(r != nullptr && blob_host != nullptr, "null argument");
    ReplayCkptHeader hd;
    if (bytes < sizeof(hd))
        return fail(SNK_ERR_INVALID, "%s: truncated blob: %zu bytes, the header alone has %zu", __func__, bytes, sizeof(hd));
    memcpy(&hd, blob_host, sizeof(hd));
    if (memcmp(hd.magic, kReplayMagic, 8) != 0) return fail(SNK_ERR_INVALID, "%s: not a replay checkpoint (wrong magic)", __func__);
    if (hd.version != CKPT_VERSION || hd.record_bytes != 128)
        return fail(SNK_ERR_INVALID, "%s: checkpoint format version %u (records of %u bytes), this library reads %u (128)", __func__,
                    hd.version, hd.record_bytes, CKPT_VERSION);
    if (hd.capacity != r->capacity)
        return fail(SNK_ERR_INVALID, "%s: checkpoint of a ring of %lld, this ring holds %lld", __func__, (long long)hd.capacity, r->capacity);
    if (hd.total < 0) return fail(SNK_ERR_INVALID, "%s: negative count of stored transitions", __func__);
    const long long filled = hd.total < hd.capacity ? hd.total : hd.capacity;
    const size_t recs = (size_t)filled * 128;
    if (bytes != sizeof(hd) + recs)
        return fail(SNK_ERR_INVALID, "%s: blob of %zu bytes, a checkpoint of %lld records has %zu", __func__, bytes, filled, sizeof(hd) + recs);
    DeviceGuard guard(r->device);
    LoadScratch sc;
    int rc = load_scratch(sc, (const uint8_t *)blob_host + sizeof(hd), recs, nullptr);
    if (rc != SNK_OK) return rc;
    const uint4 *ring = reinterpret_cast<const uint4 *>(sc.data());
    if (filled > 0) k_replay_validate<<<nblocks(filled, 256), 256>>>(ring, filled, sc.first());
    long long bad = -1;
    int rule = 0;
    if ((rc = load_verdict(sc, nullptr, &bad, &rule)) != SNK_OK) return rc;
    if (bad >= 0) {
        if (first_bad_slot != nullptr) *first_bad_slot = bad;
        return fail(SNK_ERR_INVALID, "%s: record %lld of the checkpoint: %s", __func__, bad,
                    rule < (int)(sizeof(kReplayRuleText) / sizeof(kReplayRuleText[0])) ? kReplayRuleText[rule] : "?");
    }
    SNK_CUDA(cudaDeviceSynchronize());                     // nothing in flight reads or writes the ring any more
    if (recs) SNK_CUDA(cudaMemcpy(r->ring, sc.data(), recs, cudaMemcpyDeviceToDevice));
    r->total = hd.total;
    r->draws = hd.draws;
    return SNK_OK;
}

}  // extern "C"
