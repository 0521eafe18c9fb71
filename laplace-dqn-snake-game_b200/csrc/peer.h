// peer.h — the one definition of the epoch flags through which ranks of a box order their work on the device (the barrier
// of the row-sharded Gram, gram_shard.cu; the reduction chain of the data-parallel learner, qnet.cu).
//
// A flag is a monotonically increasing 64-bit epoch in device memory that peers may map (snk_ipc_*).  A rank announces
// "everything my stream did before this point is done" by storing the epoch into a peer's flag slot; a waiter spins on its
// own slot until it holds at least that epoch.  Release at system scope before the store, acquire on the load: whatever the
// signalling stream wrote before is visible to every kernel the waiting stream runs after the wait.
#pragma once
#include <stdint.h>

namespace snk {

constexpr int MAX_WORLD = 16;                 // ranks of one box

__device__ __forceinline__ void peer_signal(unsigned long long *slot, unsigned long long epoch) {
    __threadfence_system();
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(slot), "l"(epoch) : "memory");
}

// Bounded spin: a missing peer sets *timed_out and returns after ~20 s (at 2 GHz) instead of hanging the stream.
__device__ __forceinline__ void peer_wait(const unsigned long long *slot, unsigned long long epoch, int *timed_out) {
    const long long t0 = clock64();
    for (;;) {
        unsigned long long v;
        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(slot) : "memory");
        if (v >= epoch) break;
        if (clock64() - t0 > 40000000000ll) {
            *timed_out = 1;
            break;
        }
        __nanosleep(200);
    }
    __threadfence_system();
}

}  // namespace snk
