// gram_shard.cu — the row-sharded multi-GPU Gram behind the C ABI (SURVEY §8b/§8e, BASELINE config 5b): one
// snk_gram_shard per rank (= per process, one GPU each), ONE call per rank and Gram (snk_gram_shard_run).
//
// Rank g owns rows_g of A (K_total x P).  G[rows_g, :] needs every other rank's rows — the one real exchange on the path:
//   1. pack: my rows -> bf16 planes (hi, lo) in cudaIpc-exportable memory (or written there directly by a producer,
//      snk_qnet_sample_grads);
//   2. planes ring: at step i my rows are multiplied against the planes of rank (g+i) % R while the planes of rank
//      (g+i+1) % R are copied from that peer's memory over NVLink into the other half of a double buffer on a copy
//      stream — the all-gather never exists as a separate phase, it hides under the tcgen05 main loop;
//         Y[rows_g, rows_p] = hi_g hi_p^T + hi_g lo_p^T + lo_g hi_p^T        (a finished block of G)
//      G is symmetric, so the ring stops half way: i = 0 (my own block, upper-triangle tiles only) .. R/2; the step
//      R/2 of an even R is shared between the two ranks of the pair (snk_gram_shard_schedule);
//   3. mirror: the blocks I did not compute are the transposes of blocks my peers did — the transpose kernel reads
//      Y[rows_p, rows_g] straight out of rank p's memory (peer loads over NVLink), the transpose all-to-all is fused
//      into that kernel.
// The three phases are separated by a DEVICE-side barrier over peer memory (k_peer_barrier: every rank stores its epoch
// into a slot of every peer's flag array and spins on its own array), so a run is a pure stream of kernels and copies:
// no host synchronisation, no communicator.  The host language only has to move 192 bytes of IPC handles per rank once
// (any transport: MPI, Distributed.jl, torch.distributed, a file).
#include <string.h>

#include <new>
#include <vector>

#include "common.h"
#include "peer.h"

namespace snk {
namespace gram_shard {

struct PeerFlags {
    unsigned long long *p[MAX_WORLD];
};

// thread r: publish my arrival at `epoch` in slot [rank] of rank r's flag array, then wait for rank r's arrival in my
// slot [r] (peer.h).  Everything this stream did before the barrier is visible to a peer that has passed it.
__global__ void k_peer_barrier(PeerFlags peers, unsigned long long *mine, int world, int rank, unsigned long long epoch,
                               int *timed_out) {
    const int r = threadIdx.x;
    if (r >= world) return;
    peer_signal(peers.p[r] + rank, epoch);
    peer_wait(mine + r, epoch, timed_out);
}

// the ring schedule of one rank (see snk_gram_shard_schedule in the header)
struct Step { long long a0, a1, b0, b1; };
// where the two ranks of a pair divide the lower rank's rows.  Rounding to the 256-row tile would not shorten the longer side
// (6,250 rows: 13 x 25 tiles against 25 x 13 either way), so the split is simply even.
static long long split_point(long long rows) { return rows / 2; }
static int schedule(const long long *rows_all, int world, int rank, Step *out) {
    const int steps = world / 2 + 1;
    for (int i = 0; i < steps; i++) {
        const int p = (rank + i) % world;
        Step s = {0, rows_all[rank], 0, rows_all[p]};
        if (i > 0 && world % 2 == 0 && i == world / 2) {
            if (rank < p) s.a1 = split_point(rows_all[rank]);
            else s.b0 = split_point(rows_all[p]);
        }
        out[i] = s;
    }
    return steps;
}

}  // namespace gram_shard
}  // namespace snk

using namespace snk;
using namespace snk::gram_shard;

struct snk_gram_shard_s {
    int world, rank, device, splits;
    long long P, rows, K, max_rows, pitch;
    size_t plane_bytes;
    std::vector<long long> rows_all, col0;
    uint8_t *planes;                 // [hi | lo] of my rows (exported)
    uint8_t *stage[2];               // peers' planes, double buffered
    float *Y;                        // my row block of Y: rows x K (exported)
    void *scratch;
    unsigned long long *flags;       // MAX_WORLD epoch slots written by the peers (exported)
    int *d_timed_out;
    uint8_t *peer_planes[MAX_WORLD];
    float *peer_Y[MAX_WORLD];
    PeerFlags peer_flags;
    std::vector<void *> opened;      // cudaIpcOpenMemHandle mappings to close
    bool connected;
    unsigned long long epoch;
    cudaStream_t copy;
    cudaEvent_t ev_copied[MAX_WORLD], ev_used[MAX_WORLD], ev_go;
};

static void shard_free(snk_gram_shard_s *g) {
    for (void *p : g->opened) cudaIpcCloseMemHandle(p);
    void *ptrs[] = {g->planes, g->stage[0], g->stage[1], g->Y, g->scratch, g->flags, g->d_timed_out};
    for (void *p : ptrs) if (p) cudaFree(p);
    for (int i = 0; i < MAX_WORLD; i++) {
        if (g->ev_copied[i]) cudaEventDestroy(g->ev_copied[i]);
        if (g->ev_used[i]) cudaEventDestroy(g->ev_used[i]);
    }
    if (g->ev_go) cudaEventDestroy(g->ev_go);
    if (g->copy) cudaStreamDestroy(g->copy);
    delete g;
}

extern "C" {

int snk_gram_shard_create(snk_gram_shard *out, const int64_t *rows_all, int world, int rank, int64_t P, int splits, int device) {
    SNK_REQUIRE(out != nullptr && rows_all != nullptr, "null argument");
    SNK_REQUIRE(world >= 1 && world <= MAX_WORLD && rank >= 0 && rank < world && P > 0 && splits >= 0, "bad argument");
    *out = nullptr;
    for (int r = 0; r < world; r++) SNK_REQUIRE(rows_all[r] > 0, "every rank must own at least one row");
    DeviceGuard guard(device);
    snk_gram_shard_s *g = new (std::nothrow) snk_gram_shard_s();
    if (g == nullptr) return fail(SNK_ERR_INVALID, "out of host memory");
    g->world = world; g->rank = rank; g->device = device; g->splits = splits; g->P = P;
    g->rows_all.assign(rows_all, rows_all + world);
    g->col0.resize(world);
    long long acc = 0, mx = 0;
    for (int r = 0; r < world; r++) { g->col0[r] = acc; acc += rows_all[r]; if (rows_all[r] > mx) mx = rows_all[r]; }
    g->K = acc; g->rows = rows_all[rank]; g->max_rows = mx;
    int64_t pitch = 0;
    snk_gram_planes_layout(mx, P, &g->plane_bytes, &pitch);
    g->pitch = pitch;
    size_t sb = 0;                                   // the largest split-K scratch any block of my schedule needs
    {
        Step sch[MAX_WORLD];
        const int steps = schedule(g->rows_all.data(), world, rank, sch);
        for (int i = 0; i < steps; i++) {
            size_t need = 0;
            if (sch[i].a1 > sch[i].a0 && sch[i].b1 > sch[i].b0)
                snk_gram_block_scratch_bytes(sch[i].a1 - sch[i].a0, sch[i].b1 - sch[i].b0, P, splits, &need);
            if (need > sb) sb = need;
        }
    }
    cudaError_t e = cudaSuccess;
    auto A = [&](void **p, size_t bytes) { if (e == cudaSuccess) e = cudaMalloc(p, bytes < 256 ? 256 : bytes); };
    A((void **)&g->planes, 2 * g->plane_bytes);
    if (world > 1) { A((void **)&g->stage[0], 2 * g->plane_bytes); A((void **)&g->stage[1], 2 * g->plane_bytes); }
    A((void **)&g->Y, (size_t)g->rows * g->K * 4);
    A(&g->scratch, sb);
    A((void **)&g->flags, MAX_WORLD * 8);
    A((void **)&g->d_timed_out, 4);
    if (e == cudaSuccess) e = cudaMemset(g->flags, 0, MAX_WORLD * 8);
    if (e == cudaSuccess) e = cudaMemset(g->d_timed_out, 0, 4);
    // the padding columns of the planes (P..pitch) and the rows of a smaller shard must read as zero
    if (e == cudaSuccess) e = cudaMemset(g->planes, 0, 2 * g->plane_bytes);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&g->copy, cudaStreamNonBlocking);
    for (int i = 0; i < MAX_WORLD && e == cudaSuccess; i++) {
        e = cudaEventCreateWithFlags(&g->ev_copied[i], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g->ev_used[i], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&g->ev_go, cudaEventDisableTiming);
    if (e != cudaSuccess) {
        int rc = fail(SNK_ERR_CUDA, "snk_gram_shard_create: %s", cudaGetErrorString(e));
        shard_free(g);
        return rc;
    }
    g->peer_planes[rank] = g->planes; g->peer_Y[rank] = g->Y; g->peer_flags.p[rank] = g->flags;
    g->connected = world == 1;
    *out = g;
    return SNK_OK;
}

int snk_gram_shard_destroy(snk_gram_shard g) {
    if (g == nullptr) return SNK_OK;
    DeviceGuard guard(g->device);
    cudaDeviceSynchronize();
    shard_free(g);
    return SNK_OK;
}

int snk_gram_shard_export_host(snk_gram_shard g, uint8_t *handle192) {
    SNK_REQUIRE(g != nullptr && handle192 != nullptr, "null argument");
    DeviceGuard guard(g->device);
    int rc;
    if ((rc = snk_ipc_export(g->planes, handle192)) != SNK_OK) return rc;
    if ((rc = snk_ipc_export(g->Y, handle192 + 64)) != SNK_OK) return rc;
    return snk_ipc_export(g->flags, handle192 + 128);
}

int snk_gram_shard_connect_host(snk_gram_shard g, const uint8_t *handles) {
    SNK_REQUIRE(g != nullptr && handles != nullptr, "null argument");
    SNK_REQUIRE(!g->connected, "already connected");
    DeviceGuard guard(g->device);
    for (int r = 0; r < g->world; r++) {
        if (r == g->rank) continue;
        void *p[3] = {nullptr, nullptr, nullptr};
        for (int k = 0; k < 3; k++) {
            int rc = snk_ipc_import(handles + (size_t)r * SNK_GRAM_SHARD_HANDLE_BYTES + 64 * k, &p[k]);
            if (rc != SNK_OK) return rc;
            g->opened.push_back(p[k]);
        }
        g->peer_planes[r] = (uint8_t *)p[0]; g->peer_Y[r] = (float *)p[1]; g->peer_flags.p[r] = (unsigned long long *)p[2];
    }
    g->connected = true;
    return SNK_OK;
}

int snk_gram_shard_connect_local(snk_gram_shard g, const snk_gram_shard *peers) {
    SNK_REQUIRE(g != nullptr && peers != nullptr, "null argument");
    for (int r = 0; r < g->world; r++) {
        SNK_REQUIRE(peers[r] != nullptr && peers[r]->rank == r && peers[r]->world == g->world && peers[r]->K == g->K, "peer list does not match");
        g->peer_planes[r] = peers[r]->planes; g->peer_Y[r] = peers[r]->Y; g->peer_flags.p[r] = peers[r]->flags;
    }
    g->connected = true;
    return SNK_OK;
}

int snk_gram_shard_planes(snk_gram_shard g, void **hi, void **lo, int64_t *pitch_elems) {
    SNK_REQUIRE(g != nullptr, "null shard");
    if (hi) *hi = g->planes;
    if (lo) *lo = g->planes + g->plane_bytes;
    if (pitch_elems) *pitch_elems = g->pitch;
    return SNK_OK;
}

int snk_gram_shard_pack(snk_gram_shard g, const void *A_rows, int a_dtype, void *cuda_stream) {
    SNK_REQUIRE(g != nullptr && A_rows != nullptr, "null argument");
    DeviceGuard guard(g->device);
    return snk_gram_pack_planes(A_rows, a_dtype, g->P, g->rows, g->planes, g->planes + g->plane_bytes, cuda_stream);
}

int snk_gram_shard_barrier(snk_gram_shard g, void *cuda_stream) {
    SNK_REQUIRE(g != nullptr && g->connected, "shard not connected");
    DeviceGuard guard(g->device);
    g->epoch++;
    k_peer_barrier<<<1, 32, 0, (cudaStream_t)cuda_stream>>>(g->peer_flags, g->flags, g->world, g->rank, g->epoch, g->d_timed_out);
    SNK_CUDA(cudaGetLastError());
    return SNK_OK;
}

int snk_gram_shard_schedule(const int64_t *rows_all, int world, int rank, int *steps, int64_t *a0, int64_t *a1, int64_t *b0,
                            int64_t *b1) {
    SNK_REQUIRE(rows_all && steps && a0 && a1 && b0 && b1, "null argument");
    SNK_REQUIRE(world >= 1 && world <= MAX_WORLD && rank >= 0 && rank < world, "bad argument");
    long long rows[MAX_WORLD];
    for (int r = 0; r < world; r++) rows[r] = rows_all[r];
    Step st[MAX_WORLD];
    *steps = schedule(rows, world, rank, st);
    for (int i = 0; i < *steps; i++) { a0[i] = st[i].a0; a1[i] = st[i].a1; b0[i] = st[i].b0; b1[i] = st[i].b1; }
    return SNK_OK;
}

int snk_gram_shard_ring(snk_gram_shard g, int terms, int block_k, void *cuda_stream) {
    SNK_REQUIRE(g != nullptr && g->connected, "shard not connected");
    SNK_REQUIRE(terms == 1 || terms == 3, "terms must be 1 (bf16) or 3 (bf16 hi/lo split)");
    DeviceGuard guard(g->device);
    cudaStream_t st = (cudaStream_t)cuda_stream, cs = g->copy;
    const int W = g->world;
    Step sch[MAX_WORLD];
    const int steps = schedule(g->rows_all.data(), W, g->rank, sch);
    const size_t row_bytes = (size_t)g->pitch * 2;
    SNK_CUDA(cudaEventRecord(g->ev_go, st));                      // the peers' planes are ready when the stream gets here
    SNK_CUDA(cudaStreamWaitEvent(cs, g->ev_go, 0));
    for (int i = 0; i < steps; i++) {
        const int p = (g->rank + i) % W;
        if (i + 1 < steps) {                                      // prefetch the NEXT peer's planes while this step computes
            const int nxt = (g->rank + i + 1) % W;
            const Step &n = sch[i + 1];
            if (i >= 1) SNK_CUDA(cudaStreamWaitEvent(cs, g->ev_used[i - 1], 0));   // that buffer was the B operand of step i-1
            uint8_t *dst = g->stage[(i + 1) % 2];
            const size_t off = (size_t)n.b0 * row_bytes, used = (size_t)(n.b1 - n.b0) * row_bytes;   // only the rows this step reads
            if (used > 0) {
                SNK_CUDA(cudaMemcpyAsync(dst + off, g->peer_planes[nxt] + off, used, cudaMemcpyDefault, cs));
                if (terms > 1)
                    SNK_CUDA(cudaMemcpyAsync(dst + g->plane_bytes + off, g->peer_planes[nxt] + g->plane_bytes + off, used,
                                             cudaMemcpyDefault, cs));
            }
            SNK_CUDA(cudaEventRecord(g->ev_copied[i + 1], cs));
        }
        const uint8_t *b_hi = g->planes;
        if (i > 0) {
            SNK_CUDA(cudaStreamWaitEvent(st, g->ev_copied[i], 0));
            b_hi = g->stage[i % 2];
        }
        const Step &s = sch[i];
        if (s.a1 > s.a0 && s.b1 > s.b0) {
            const uint8_t *a_hi = g->planes + (size_t)s.a0 * row_bytes;
            const uint8_t *bb = b_hi + (size_t)s.b0 * row_bytes;
            int rc = snk_gram_block(a_hi, a_hi + g->plane_bytes, s.a1 - s.a0, bb, bb + g->plane_bytes, s.b1 - s.b0, g->P, terms,
                                    i == 0 ? 1 : 0, block_k, g->splits, g->scratch,
                                    g->Y + (size_t)s.a0 * g->K + g->col0[p] + s.b0, g->K, cuda_stream);
            if (rc != SNK_OK) return rc;
        }
        SNK_CUDA(cudaEventRecord(g->ev_used[i], st));
    }
    return SNK_OK;
}

int snk_gram_shard_mirror(snk_gram_shard g, float *G_rows, int64_t ldG, void *cuda_stream) {
    SNK_REQUIRE(g != nullptr && g->connected && G_rows != nullptr && ldG >= g->K, "bad argument");
    DeviceGuard guard(g->device);
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const int W = g->world;
    Step mine[MAX_WORLD], theirs[MAX_WORLD];
    const int steps = schedule(g->rows_all.data(), W, g->rank, mine);
    for (int i = 0; i < steps; i++) {                             // the blocks I computed: out of my Y
        const int p = (g->rank + i) % W;
        const Step &s = mine[i];
        if (s.a1 == s.a0 || s.b1 == s.b0) continue;
        SNK_CUDA(cudaMemcpy2DAsync(G_rows + (size_t)s.a0 * ldG + g->col0[p] + s.b0, (size_t)ldG * 4,
                                   g->Y + (size_t)s.a0 * g->K + g->col0[p] + s.b0, (size_t)g->K * 4, (size_t)(s.b1 - s.b0) * 4,
                                   (size_t)(s.a1 - s.a0), cudaMemcpyDeviceToDevice, st));
    }
    for (int i = 1; i < steps; i++) {                             // the blocks rank q = g - i computed against my rows: transposed
        const int q = (g->rank - i + W) % W;
        schedule(g->rows_all.data(), W, q, theirs);
        const Step &s = theirs[i];                                // q's rows [a0,a1) x my rows [b0,b1), in q's Y
        if (s.a1 == s.a0 || s.b1 == s.b0) continue;
        int rc = snk_gram_transpose_block(g->peer_Y[q] + (size_t)s.a0 * g->K + g->col0[g->rank] + s.b0, g->K, s.b1 - s.b0, s.a1 - s.a0,
                                          G_rows + (size_t)s.b0 * ldG + g->col0[q] + s.a0, ldG, cuda_stream);
        if (rc != SNK_OK) return rc;
    }
    return SNK_OK;
}

int snk_gram_shard_run(snk_gram_shard g, const void *A_rows, int a_dtype, int terms, int block_k, float *G_rows, int64_t ldG,
                       void *cuda_stream) {
    SNK_REQUIRE(g != nullptr && g->connected, "shard not connected");
    SNK_REQUIRE(terms == 1 || terms == 3, "terms must be 1 (bf16) or 3 (bf16 hi/lo split)");
    int rc;
    if (A_rows != nullptr && (rc = snk_gram_shard_pack(g, A_rows, a_dtype, cuda_stream)) != SNK_OK) return rc;   // NULL: planes already written
    if ((rc = snk_gram_shard_barrier(g, cuda_stream)) != SNK_OK) return rc;      // every rank's planes are packed
    if ((rc = snk_gram_shard_ring(g, terms, block_k, cuda_stream)) != SNK_OK) return rc;
    if ((rc = snk_gram_shard_barrier(g, cuda_stream)) != SNK_OK) return rc;      // every rank's blocks of Y are complete
    if ((rc = snk_gram_shard_mirror(g, G_rows, ldG, cuda_stream)) != SNK_OK) return rc;
    return snk_gram_shard_barrier(g, cuda_stream);                                // nobody still reads my Y / planes
}

int snk_gram_shard_status_host(snk_gram_shard g, int *timed_out) {
    SNK_REQUIRE(g != nullptr && timed_out != nullptr, "null argument");
    DeviceGuard guard(g->device);
    SNK_CUDA(cudaMemcpy(timed_out, g->d_timed_out, 4, cudaMemcpyDeviceToHost));
    if (*timed_out) return fail(SNK_ERR_TIMEOUT, "snk_gram_shard: a peer did not reach a barrier within ~20 s");
    return SNK_OK;
}

}  // extern "C"
