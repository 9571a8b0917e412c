// TEST VEHICLE (tests/ only) -- compiles the product's restatement of numpy's default_rng stream
// (ppo-2dgrid_b200/csrc/np_random.cuh) for the HOST so the CPU test tier can compare the exact code the seeded layout
// kernel runs with numpy itself.  It is not part of the product and is not shipped or loaded by it.
#include <stdint.h>

#include "np_random.cuh"

using namespace merlin;

extern "C" {

// SeedSequence(seed).generate_state(4, uint64) for every seed: out u64[n][4]
void nr_seed_state(const uint64_t* seeds, int n, uint64_t* out) {
  for (int i = 0; i < n; ++i) {
    uint64_t w[4];
    seed_sequence_state(seeds[i], w);
    for (int k = 0; k < 4; ++k) out[4 * i + k] = w[k];
  }
}

// PCG64(seed).random_raw(count) for every seed: out u64[n][count]
void nr_raw(const uint64_t* seeds, int n, int count, uint64_t* out) {
  for (int i = 0; i < n; ++i) {
    NpRandom g;
    g.seed(seeds[i]);
    for (int k = 0; k < count; ++k) out[(int64_t)i * count + k] = g.next64();
  }
}

// One fresh default_rng(seed) per seed, driven by the same script of calls:
//   ops[3*o] == 0: integers(ops[3*o+1], ops[3*o+2])                        -> one value
//   ops[3*o] == 1: choice(ops[3*o+1], size=ops[3*o+2], replace=False)      -> ops[3*o+2] values
// out: int64[n][n_out], n_out = the number of values the script yields.
void nr_script(const uint64_t* seeds, int n, const int64_t* ops, int n_ops, int n_out, int64_t* out) {
  for (int i = 0; i < n; ++i) {
    NpRandom g;
    g.seed(seeds[i]);
    int64_t* o = out + (int64_t)i * n_out;
    for (int p = 0; p < n_ops; ++p) {
      if (ops[3 * p] == 0) {
        *o++ = g.integers(ops[3 * p + 1], ops[3 * p + 2]);
      } else {
        int picks[NpRandom::kMaxChoice];
        const int k = (int)ops[3 * p + 2];
        g.choice((int)ops[3 * p + 1], k, picks);
        for (int t = 0; t < k; ++t) *o++ = picks[t];
      }
    }
  }
}

}  // extern "C"
