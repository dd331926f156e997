// shuffle_rng.cuh -- the counter-based generator of the shuffle significance test (mirfold_shuffle_test).
//
// A shuffle is a pure function of (seed, record r, replicate k): its generator state is derived from those three
// numbers alone, so results do not depend on device count, chunking or rounds.  splitmix64 (Steele, Lea, Flood 2014):
// state += golden gamma, output = the mix64 finaliser of the state.  A draw in [0, m) is the high word of draw * m
// (no rejection: the bias is below m / 2^64).  tests/test_shuffle_significance.py mirrors this file in Python; the
// two must change together.
#pragma once
#include <cstdint>

#define MF_SHUF_GAMMA 0x9E3779B97F4A7C15ULL
#define MF_SHUF_MAX_SYMBOLS 16   /* distinct bytes per record in dinucleotide mode */

__host__ __device__ __forceinline__ uint64_t mf_mix64(uint64_t z)
{
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

// initial state of replicate k of record r
__host__ __device__ __forceinline__ uint64_t mf_shuf_state(uint64_t seed, uint32_t r, uint32_t k)
{
    return mf_mix64(mf_mix64(seed + MF_SHUF_GAMMA) ^ (((uint64_t)r << 32) | (uint64_t)k));
}

__host__ __device__ __forceinline__ uint64_t mf_shuf_next(uint64_t &s)
{
    s += MF_SHUF_GAMMA;
    return mf_mix64(s);
}

// uniform draw in [0, m), m >= 1
__host__ __device__ __forceinline__ uint32_t mf_shuf_below(uint64_t &s, uint32_t m)
{
#ifdef __CUDA_ARCH__
    return (uint32_t)__umul64hi(mf_shuf_next(s), (uint64_t)m);
#else
    return (uint32_t)(((unsigned __int128)mf_shuf_next(s) * m) >> 64);
#endif
}
