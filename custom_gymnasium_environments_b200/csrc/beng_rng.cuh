// Counter-based device RNG of the engine: Philox4x32-10 keyed by (seed), positioned by
// (draw index, global env id, stream).  The contract (draw -> value maps) is stated in
// oracle/philox.py and include/beng.h; this file is its one device statement, and every kernel's
// word source uses the keying and the maps defined here.  The reference's draw SITES that consume it are cited
// at each call (e.g. _place_food, snake_env_classic/snake_env.py:121-129).
#pragma once
#include <cstdint>

namespace beng {

struct Philox4 {
    uint32_t v[4];
};

__device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                 uint32_t k1) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    return Philox4{{c0, c1, c2, c3}};
}

// Where an env's stream sits in Philox's input: counter = (block, env_lo, env_hi, stream), key = the 64-bit seed.
struct StreamKey {
    uint32_t env_lo, env_hi, stream, k0, k1;
};
__device__ __forceinline__ StreamKey stream_key(uint64_t env, uint32_t stream, uint64_t seed) {
    return StreamKey{(uint32_t)env, (uint32_t)(env >> 32), stream, (uint32_t)seed, (uint32_t)(seed >> 32)};
}
// Block `blk` of a stream: its draws 4 blk .. 4 blk + 3.
__device__ __forceinline__ Philox4 philox_block(uint32_t blk, const StreamKey &s) {
    return philox4x32_10(blk, s.env_lo, s.env_hi, s.stream, s.k0, s.k1);
}

// random() from the top 27 bits of one draw and the top 26 of the next, CPython's random.random() construction
__device__ __forceinline__ double bits53(uint32_t a27, uint32_t b26) {
    return ((double)a27 * 67108864.0 + (double)b26) * (1.0 / 9007199254740992.0);
}

// Box-Muller: the standard-normal deviate of two random() values (the contract's np.random.normal stand-in)
__device__ __forceinline__ double box_muller(double u1, double u2) {
    return sqrt(-2.0 * log(1.0 - u1)) * cos(2.0 * 3.141592653589793 * u2);
}

// The draw -> value maps of the contract over any word source `Src` that provides u32(), the env stream's next draw.
template <class Src>
struct Draws {
    __device__ __forceinline__ uint32_t draw() { return static_cast<Src *>(this)->u32(); }
    // randint(a, b) inclusive: one draw, multiply-high range map
    __device__ __forceinline__ int randint(int a, int b) { return a + (int)__umulhi(draw(), (uint32_t)(b - a + 1)); }
    // random(): two draws, 53 bits.  Each draw is shifted as it is taken; to_random53() of the two draws computes the
    // same value but gives the climate and crypto kernels another register assignment.
    __device__ __forceinline__ double random53() {
        const uint32_t a = draw() >> 5, b = draw() >> 6;
        return bits53(a, b);
    }
    __device__ __forceinline__ double uniform(double a, double b) { return a + (b - a) * random53(); }
    // normal(mu, sd): Box-Muller on two random53() draws (four u32)
    __device__ __forceinline__ double normal(double mu, double sd) {
        const double u1 = random53(), u2 = random53();
        return mu + sd * box_muller(u1, u2);
    }
};

// Sequential view of one env's stream.  `ctr` is the index of the next u32 draw and is what gets
// persisted in the env state; a Philox block (4 draws) is computed lazily and reused.
struct EnvStream : Draws<EnvStream> {
    uint32_t ctr;
    StreamKey key;
    uint32_t cached_blk;
    Philox4 cache;

    __device__ __forceinline__ EnvStream(uint64_t seed, uint64_t env, uint32_t stream, uint32_t ctr_)
        : ctr(ctr_), key(stream_key(env, stream, seed)), cached_blk(0xFFFFFFFFu) {}

    __device__ __forceinline__ uint32_t u32() {
        const uint32_t blk = ctr >> 2;
        if (blk != cached_blk) {
            cache = philox_block(blk, key);
            cached_blk = blk;
        }
        const uint32_t lane = ctr & 3u;
        ++ctr;
        // select without dynamic register indexing
        return lane == 0 ? cache.v[0] : lane == 1 ? cache.v[1] : lane == 2 ? cache.v[2] : cache.v[3];
    }
    // The next N <= 9 draws at once, for callers that know how many they will consume (a fixed-shape step): the two or
    // three blocks they span are computed up front and each draw is one 4-way select on the starting offset, instead
    // of a block check, an offset select and a counter update per draw.  Same values as N calls of u32().
    template <int N>
    __device__ __forceinline__ void take(uint32_t (&out)[N]) {
        static_assert(N >= 1 && N <= 9, "at most three blocks");
        const uint32_t blk = ctr >> 2, o = ctr & 3u;
        const Philox4 A = philox_block(blk, key);
        Philox4 B = A, C = A;
        if (N > 1) B = philox_block(blk + 1, key);
        if (N > 5 && o + N > 8) C = philox_block(blk + 2, key);
        const uint32_t v[12] = {A.v[0], A.v[1], A.v[2], A.v[3], B.v[0], B.v[1], B.v[2], B.v[3], C.v[0], C.v[1], C.v[2], C.v[3]};
#pragma unroll
        for (int j = 0; j < N; ++j) out[j] = o == 0 ? v[j] : o == 1 ? v[j + 1] : o == 2 ? v[j + 2] : v[j + 3];
        ctr += N;
        cached_blk = 0xFFFFFFFFu;  // (the lazy cache is not kept in step with this path)
    }
    // random() from two given draws (the construction of random53())
    static __device__ __forceinline__ double to_random53(uint32_t d0, uint32_t d1) { return bits53(d0 >> 5, d1 >> 6); }
    // normal(mu, sd) from four given draws (the construction of normal())
    static __device__ __forceinline__ double to_normal(double mu, double sd, uint32_t d0, uint32_t d1, uint32_t d2, uint32_t d3) {
        const double u1 = to_random53(d0, d1), u2 = to_random53(d2, d3);
        return mu + sd * box_muller(u1, u2);
    }
};

}  // namespace beng
