// mlp_layout.cuh -- offsets of the layers inside the flat float32 parameter blocks.
// Keras order [W1 (in x out row-major), b1, W2, b2, ...]:
//   actor  ns -> 256 -> 256 -> na         (NeuralNetwork.py:51-63, LeakyReLU(0.3) between)
//   critic ns -> 64 -> 64 -> 128 -> 128 -> 1  (NeuralNetwork.py:95-108, sin after the first four)
// The transposed block used by the backward sweeps has the same offsets with every W stored (out x in).
#pragma once
#include <stdint.h>

namespace cacto {

constexpr int ACTOR_H = 256;
constexpr int CR_H1 = 64, CR_H2 = 64, CR_H3 = 128, CR_H4 = 128;
constexpr float LEAKY_ALPHA = 0.3f;   // keras.layers.LeakyReLU() default

// hidden widths h1 / h2: ACTOR_H for the fused kernels, any 1..CACTO_ACTOR_MAX_WIDTH for the width-generic ones (actor_width.cu)
struct ActorLayout {
  int ns, na, h1, h2;
  int64_t W1, b1, W2, b2, W3, b3, total;
  __host__ __device__ ActorLayout(int ns_, int na_, int h1_ = ACTOR_H, int h2_ = ACTOR_H) : ns(ns_), na(na_), h1(h1_), h2(h2_) {
    W1 = 0; b1 = W1 + (int64_t)ns * h1;
    W2 = b1 + h1; b2 = W2 + (int64_t)h1 * h2;
    W3 = b2 + h2; b3 = W3 + (int64_t)h2 * na;
    total = b3 + na;
  }
};

struct CriticLayout {
  int ns;
  int64_t W[5], b[5], total;
  int in[5], out[5];
  __host__ __device__ explicit CriticLayout(int ns_) : ns(ns_) {
    const int dims[6] = {ns_, CR_H1, CR_H2, CR_H3, CR_H4, 1};
    int64_t o = 0;
    for (int l = 0; l < 5; ++l) {
      in[l] = dims[l]; out[l] = dims[l + 1];
      W[l] = o; o += (int64_t)dims[l] * dims[l + 1];
      b[l] = o; o += dims[l + 1];
    }
    total = o;
  }
};

}  // namespace cacto
