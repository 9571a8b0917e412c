// np_random.cuh -- the random stream of `np.random.default_rng(seed)` restated as host+device inline code, so that the
// seeded layout generator (layout_kernels.cu) builds on the GPU exactly the layouts `env.reset(seed=s)` builds in the
// reference.  The host test vehicle tests/csrc/np_random_model.cpp compiles the SAME code with g++ and the CPU test tier
// compares it with numpy itself (tests/test_np_random_cpu.py).
//
// What is restated (numpy sources: random/bit_generator.pyx, random/_pcg64.pyx, random/src/pcg64/pcg64.h,
// random/src/distributions/distributions.c, random/_generator.pyx):
//   SeedSequence(seed)        entropy = the seed as little-endian uint32 words (one word below 2^32, two up to 2^64-1),
//                             no spawn key; mix_entropy into a pool of 4 words (hashmix INIT_A / MULT_A, then mix
//                             MIX_MULT_L / MIX_MULT_R, XSHIFT 16); generate_state(4, uint64) with INIT_B / MULT_B
//   PCG64(seed_seq)           pcg64_set_seed: state = words 0||1, inc = (words 2||3 << 1) | 1, two-step seeding;
//                             128-bit LCG, XSL-RR output taken after the step
//   next_uint32               the low half of a 64-bit output; the high half is buffered for the next call (has_uint32)
//   integers(lo, hi)          int64 default dtype: random_bounded_uint64(off = lo, rng = hi - 1 - lo, use_masked = 0).
//                             rng == 0 returns lo and draws nothing; rng == 2^32 - 1 is one next_uint32; otherwise
//                             Lemire's bounded method on next_uint32.  Ranges wider than 2^32 are not restated.
//   choice(pop, k, replace=False)  pop <= 10000: Floyd's algorithm (val = bounded [0, j] for j in [pop-k, pop), no draw
//                             for j == 0; val if not yet taken, else j), then _shuffle_int of the k picks (for
//                             i = k-1 .. 1 swap with a Lemire-bounded draw in [0, i]).
// Pinned to numpy 2.3.5.  Older numpy shuffles the picks with the masked `random_interval`: the same set, a different
// stream, and every later draw diverges.  The CPU tests print the numpy version they compared against.
#pragma once
#include <stdint.h>

#ifndef MERLIN_HD
#if defined(__CUDACC__)
#define MERLIN_HD __host__ __device__ __forceinline__
#else
#define MERLIN_HD inline
#endif
#endif

namespace merlin {

// SeedSequence(seed).generate_state(4, np.uint64)
MERLIN_HD void seed_sequence_state(uint64_t seed, uint64_t (&out)[4]) {
  constexpr uint32_t kInitA = 0x43b0d7e5u, kMultA = 0x931e8875u, kInitB = 0x8b51f9ddu, kMultB = 0x58f38dedu;
  constexpr uint32_t kMixL = 0xca01f9ddu, kMixR = 0x4973f715u;
  const uint32_t words[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
  const int n_words = (seed >> 32) ? 2 : 1;
  uint32_t hash_const = kInitA;
  auto hashmix = [&hash_const](uint32_t v) {
    v ^= hash_const;
    hash_const *= kMultA;
    v *= hash_const;
    return v ^ (v >> 16);
  };
  auto mix = [](uint32_t x, uint32_t y) {
    const uint32_t r = kMixL * x - kMixR * y;
    return r ^ (r >> 16);
  };
  uint32_t pool[4];
  for (int i = 0; i < 4; ++i) pool[i] = hashmix(i < n_words ? words[i] : 0u);
  for (int s = 0; s < 4; ++s)
    for (int d = 0; d < 4; ++d)
      if (s != d) pool[d] = mix(pool[d], hashmix(pool[s]));
  uint32_t h = kInitB;
  uint32_t state[8];
  for (int i = 0; i < 8; ++i) {
    uint32_t v = pool[i & 3] ^ h;
    h *= kMultB;
    v *= h;
    state[i] = v ^ (v >> 16);
  }
  for (int i = 0; i < 4; ++i) out[i] = (uint64_t)state[2 * i] | ((uint64_t)state[2 * i + 1] << 32);
}

MERLIN_HD uint64_t mulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
  return __umul64hi(a, b);
#else
  return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

// numpy's Generator(PCG64(SeedSequence(seed))): the draws the layout routines make
struct NpRandom {
  static constexpr uint64_t kMulHi = 2549297995355413924ull, kMulLo = 4865540595714422341ull;
  static constexpr int kMaxChoice = 8;  // largest k of choice(): hard draws at most 5 gap rows
  uint64_t hi, lo, inc_hi, inc_lo;
  uint32_t buffered;
  bool has_buffered;

  MERLIN_HD void step() {  // state = state * mult + inc (mod 2^128)
    const uint64_t m_lo = lo * kMulLo;
    const uint64_t m_hi = mulhi64(lo, kMulLo) + lo * kMulHi + hi * kMulLo;
    lo = m_lo + inc_lo;
    hi = m_hi + inc_hi + (lo < m_lo ? 1u : 0u);
  }
  MERLIN_HD void seed(uint64_t s) {  // pcg64_set_seed(seed_sequence words 0..1, words 2..3)
    uint64_t w[4];
    seed_sequence_state(s, w);
    inc_hi = (w[2] << 1) | (w[3] >> 63);
    inc_lo = (w[3] << 1) | 1u;
    hi = lo = 0;
    step();
    const uint64_t add_lo = lo + w[1];
    hi = hi + w[0] + (add_lo < lo ? 1u : 0u);
    lo = add_lo;
    step();
    has_buffered = false;
    buffered = 0;
  }
  MERLIN_HD uint64_t next64() {  // XSL-RR of the stepped state
    step();
    const uint64_t x = hi ^ lo;
    const unsigned r = (unsigned)(hi >> 58);
    return (x >> r) | (x << ((64u - r) & 63u));
  }
  MERLIN_HD uint32_t next32() {
    if (has_buffered) {
      has_buffered = false;
      return buffered;
    }
    const uint64_t v = next64();
    has_buffered = true;
    buffered = (uint32_t)(v >> 32);
    return (uint32_t)v;
  }
  // random_bounded_uint64(off = 0, rng, use_masked = 0) for rng < 2^32: uniform in [0, rng]
  MERLIN_HD uint32_t bounded(uint32_t rng) {
    if (rng == 0) return 0;
    if (rng == 0xffffffffu) return next32();
    const uint32_t rng_excl = rng + 1;
    uint64_t m = (uint64_t)next32() * rng_excl;
    uint32_t left = (uint32_t)m;
    if (left < rng_excl) {
      const uint32_t threshold = (0xffffffffu - rng) % rng_excl;
      while (left < threshold) {
        m = (uint64_t)next32() * rng_excl;
        left = (uint32_t)m;
      }
    }
    return (uint32_t)(m >> 32);
  }
  // integers(lo, hi) for lo < hi <= lo + 2^32
  MERLIN_HD long long integers(long long lo_, long long hi_) { return lo_ + (long long)bounded((uint32_t)(hi_ - 1 - lo_)); }
  // choice(pop, size=k, replace=False) for 1 <= k <= min(pop, kMaxChoice), pop <= 10000: indices in [0, pop)
  MERLIN_HD void choice(int pop, int k, int* out) {
    for (int j = pop - k; j < pop; ++j) {
      const int val = (int)bounded((uint32_t)j);
      bool taken = false;
      for (int t = 0; t < j - (pop - k); ++t) taken |= out[t] == val;
      out[j - (pop - k)] = taken ? j : val;
    }
    for (int i = k - 1; i >= 1; --i) {
      const int t = (int)bounded((uint32_t)i);
      const int tmp = out[t];
      out[t] = out[i];
      out[i] = tmp;
    }
  }
};

}  // namespace merlin
