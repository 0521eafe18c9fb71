// qnet_theta.h — where each parameter of the Q-net lives in the device copy of theta (qnet_grads.cu reads it, qnet.cu writes it)
#pragma once

namespace snk {
namespace qgrad {

// Flux.destructure offsets (SURVEY 8c)
constexpr int O_W1 = 0, O_B1 = 288, O_W2 = 304, O_B2 = 4912, O_W3 = 4944, O_B3 = 78672, O_W4 = 78736, O_B4 = 181136,
              O_W5 = 181200, O_B5 = 181392, NP = 181395;
// the device copy of theta carries two re-ordered copies of W3 behind it (written by qnet.cu's scatter_param)
constexpr int O_W3OF = 181440;                 // [c][a2][a1][o]: W3of[((c*6 + a2)*6 + a1)*64 + o] = W3[a1 + 6 (a2 + 6 (c + 32 o))]
constexpr int O_W3CF = O_W3OF + 73728;         // [o][a2][a1][c]: W3cf[((o*6 + a2)*6 + a1)*32 + c]
constexpr int THETA_EXT = O_W3CF + 73728;

}  // namespace qgrad
}  // namespace snk
