// Microbenchmark (dev tool, not product): the price of a partly written 32-byte sector against a whole one, in the
// store pattern of the in-place snake step (csrc/snake.cu, snake_patch_kernel).  A 419 MB buffer of 1,048,576 rows of
// 400 B, one thread per row, and per launch one store into a random 32-byte sector that lies inside the thread's row,
// plus a second one into another random in-row sector for every fifth row (1.2 stores per row):
//   none   the same launch, index math and hashing, no store
//   byte   one 1-byte store into the sector
//   v8     the whole sector in one 256-bit store (st.global.v8.b32, SASS STG.E.ENL2.256)
//   2xv4   the whole sector as two 16-byte stores by the same thread
// The sectors move every launch (the hash is salted with the launch index), so back-to-back launches mostly miss L2
// (419 MB against 126 MB).  Modes run in rounds, the order rotating every round; each entry is one round of REPS
// back-to-back launches between two CUDA events.
//
// `./sector_store walk` asks instead whether the order in which a launch visits the rows lets the L2 keep the sectors
// the next launch writes again.  Each row holds a random-walk "head" on a 20 x 20 board (one step up, down, left or
// right per launch, kept on the board, as a length-1 snake moves); a launch writes the whole 32-byte sector (two 16-byte
// stores) of the old cell and, when it differs, of the new one, so a row's sector at launch i + 1 is the one of launch
// i or a neighbour.  The cell lives in a 2-byte-per-row array.  Modes:
//   fwd / alt          rows in ascending CTA order every launch / CTA order reversed every other launch
//   +rmw               beside the stores, a coalesced 46 B/row stream: 16 B record read and written, 8 B read from
//                      one of 32 rotating 8 MB "action" buffers (256 MB, so they do not stay in L2), 6 B written
//   +rmw+ef            the same with an L2 evict-first policy on the action load and streaming (.cs) result stores
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o sector_store sector_store.cu && ./sector_store [walk]
#include <cuda_runtime.h>
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#define CK(x) do { cudaError_t e = (x); if (e != cudaSuccess) { printf("CUDA error %s at %d\n", cudaGetErrorString(e), __LINE__); return 1; } } while (0)

constexpr int ROW = 400, REPS = 50, ROUNDS = 7;
constexpr long long ROWS = 1 << 20;

__device__ __forceinline__ uint32_t mix(uint32_t x) {  // lowbias32
    x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
    return x;
}

enum Mode { NONE, BYTE, V8, V4X2, N_MODES };
const char *const NAMES[N_MODES] = {"none", "byte", "v8", "2xv4"};

template <Mode M>
__device__ __forceinline__ void put(uint8_t *sec, uint32_t h) {
    if constexpr (M == BYTE) {
        sec[h & 31] = (uint8_t)h;
    } else if constexpr (M == V8) {
        asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(sec), "r"(h), "r"(0), "r"(0), "r"(0),
                     "r"(0), "r"(0), "r"(0), "r"(h >> 1) : "memory");
    } else if constexpr (M == V4X2) {
        reinterpret_cast<uint4 *>(sec)[0] = make_uint4(h, 0, 0, 0);
        reinterpret_cast<uint4 *>(sec)[1] = make_uint4(0, 0, 0, h >> 1);
    }
}

template <Mode M>
__global__ void __launch_bounds__(256) sector_store(uint8_t *buf, uint32_t salt, int *sink) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= ROWS) return;
    // the 12 whole sectors of a 400-byte row start at its first 32-byte boundary (+0 on even rows, +16 on odd ones)
    uint8_t *first = buf + ((r * ROW + 31) & ~31LL);
    const uint32_t h = mix((uint32_t)r * 0x9E3779B9u ^ salt);
    const int k0 = (int)((h >> 8) % 12u);
    put<M>(first + 32 * k0, h);
    if ((h & 0xFF) < 51) {  // ~20 % of the rows: a second, different sector
        const int k1 = (k0 + 1 + (int)((h >> 16) % 11u)) % 12;
        put<M>(first + 32 * k1, h);
    }
    if constexpr (M == NONE) {
        if (h == 0x12345678u) *sink = k0;  // keeps the index math alive
    }
}

template <bool RMW, bool EF>
__global__ void __launch_bounds__(256) walk_store(uint8_t *buf, uint16_t *pos, uint32_t salt, uint32_t reverse,
                                                  uint4 *rec, const long long *act, float *rew, uint8_t *t1,
                                                  uint8_t *t2) {
    const unsigned tile = reverse ? gridDim.x - 1 - blockIdx.x : blockIdx.x;
    const long long r = (long long)tile * blockDim.x + threadIdx.x;
    if (r >= ROWS) return;
    long long a = 0;
    uint4 s = make_uint4(0, 0, 0, 0);
    if constexpr (RMW) {
        s = rec[r];
        if constexpr (EF) {
            uint64_t policy;
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
            asm volatile("ld.global.L1::no_allocate.L2::cache_hint.s64 %0, [%1], %2;" : "=l"(a) : "l"(act + r), "l"(policy));
        } else {
            a = act[r];
        }
    }
    const int p = pos[r];
    const uint32_t h = mix((uint32_t)r * 0x9E3779B9u ^ salt);
    int y = p / 20, x = p % 20;
    switch (h & 3) {
        case 0: y = y > 0 ? y - 1 : y; break;
        case 1: x = x < 19 ? x + 1 : x; break;
        case 2: y = y < 19 ? y + 1 : y; break;
        default: x = x > 0 ? x - 1 : x; break;
    }
    const int q = y * 20 + x;
    uint8_t *row = buf + r * ROW;
    uint8_t *s0 = (uint8_t *)((uintptr_t)(row + p) & ~(uintptr_t)31), *s1 = (uint8_t *)((uintptr_t)(row + q) & ~(uintptr_t)31);
    put<V4X2>(s0, h);
    if (s1 != s0) put<V4X2>(s1, h);
    pos[r] = (uint16_t)q;
    if constexpr (RMW) {
        s.x += (uint32_t)a;
        rec[r] = s;
        if constexpr (EF) {
            __stcs(rew + r, (float)a); __stcs(t1 + r, (uint8_t)(a & 1)); __stcs(t2 + r, (uint8_t)(a & 2));
        } else {
            rew[r] = (float)a; t1[r] = (uint8_t)(a & 1); t2[r] = (uint8_t)(a & 2);
        }
    }
}

int walk_main() {
    const size_t total = (size_t)ROWS * ROW;
    constexpr int N_ACT = 32, WM = 6;
    uint8_t *buf, *t1, *t2; uint16_t *pos; uint4 *rec; long long *act; float *rew;
    CK(cudaMalloc(&buf, total)); CK(cudaMemset(buf, 0, total));
    CK(cudaMalloc(&pos, ROWS * 2)); CK(cudaMemset(pos, 0, ROWS * 2));
    CK(cudaMalloc(&rec, ROWS * 16)); CK(cudaMemset(rec, 0, ROWS * 16));
    CK(cudaMalloc(&act, ROWS * 8 * N_ACT)); CK(cudaMemset(act, 1, ROWS * 8 * N_ACT));
    CK(cudaMalloc(&rew, ROWS * 4)); CK(cudaMalloc(&t1, ROWS)); CK(cudaMalloc(&t2, ROWS));
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, 0));
    const char *names[WM] = {"fwd", "alt", "fwd+rmw", "alt+rmw", "fwd+rmw+ef", "alt+rmw+ef"};
    printf("%s, %d SMs, walk: %lld rows of %d B, one random-walk cell per row, whole sectors (2 x 16 B) of the old and "
           "new cell, %d launches per entry\n", prop.name, prop.multiProcessorCount, ROWS, ROW, REPS);
    const unsigned grid = (unsigned)((ROWS + 255) / 256);
    uint32_t salt = 1;
    auto launch = [&](int m, int i) {
        ++salt;
        const uint32_t rev = (m & 1) ? (uint32_t)(i & 1) : 0u;
        const long long *a = act + (size_t)(salt % N_ACT) * ROWS;
        switch (m >> 1) {
            case 0: walk_store<false, false><<<grid, 256>>>(buf, pos, salt, rev, rec, a, rew, t1, t2); break;
            case 1: walk_store<true, false><<<grid, 256>>>(buf, pos, salt, rev, rec, a, rew, t1, t2); break;
            default: walk_store<true, true><<<grid, 256>>>(buf, pos, salt, rev, rec, a, rew, t1, t2); break;
        }
    };
    for (int i = 0; i < 400; ++i) launch(i % WM, i);  // spreads the heads over the board
    CK(cudaDeviceSynchronize());
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    std::vector<float> us[WM];
    for (int round = 0; round < ROUNDS; ++round)
        for (int j = 0; j < WM; ++j) {
            const int m = (j + round) % WM;
            CK(cudaEventRecord(e0));
            for (int i = 0; i < REPS; ++i) launch(m, i);
            CK(cudaEventRecord(e1)); CK(cudaEventSynchronize(e1));
            float ms; CK(cudaEventElapsedTime(&ms, e0, e1));
            us[m].push_back(ms * 1e3f / REPS);
        }
    CK(cudaGetLastError());
    for (int m = 0; m < WM; ++m) {
        std::vector<float> v = us[m];
        std::sort(v.begin(), v.end());
        printf("%-10s : median %6.2f us per launch (min %6.2f, max %6.2f)\n", names[m], v[v.size() / 2], v.front(), v.back());
    }
    return 0;
}

int main(int argc, char **argv) {
    if (argc > 1 && std::string(argv[1]) == "walk") return walk_main();
    const size_t total = (size_t)ROWS * ROW;
    uint8_t *buf; int *sink;
    CK(cudaMalloc(&buf, total)); CK(cudaMalloc(&sink, 4)); CK(cudaMemset(buf, 0, total));
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, 0));
    printf("%s, %d SMs, buffer %.1f MB, %lld rows of %d B, 1.2 stores per row per launch, %d launches per entry\n",
           prop.name, prop.multiProcessorCount, total / 1e6, ROWS, ROW, REPS);
    const unsigned grid = (unsigned)((ROWS + 255) / 256);
    uint32_t salt = 1;
    auto launch = [&](int m) {
        ++salt;
        switch (m) {
            case NONE: sector_store<NONE><<<grid, 256>>>(buf, salt, sink); break;
            case BYTE: sector_store<BYTE><<<grid, 256>>>(buf, salt, sink); break;
            case V8: sector_store<V8><<<grid, 256>>>(buf, salt, sink); break;
            default: sector_store<V4X2><<<grid, 256>>>(buf, salt, sink); break;
        }
    };
    cudaEvent_t a, b; CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b));
    for (int m = 0; m < N_MODES; ++m) for (int i = 0; i < 20; ++i) launch(m);
    CK(cudaDeviceSynchronize());
    std::vector<float> us[N_MODES];
    for (int round = 0; round < ROUNDS; ++round)
        for (int j = 0; j < N_MODES; ++j) {
            const int m = (j + round) % N_MODES;
            CK(cudaEventRecord(a));
            for (int i = 0; i < REPS; ++i) launch(m);
            CK(cudaEventRecord(b)); CK(cudaEventSynchronize(b));
            float ms; CK(cudaEventElapsedTime(&ms, a, b));
            us[m].push_back(ms * 1e3f / REPS);
        }
    CK(cudaGetLastError());
    for (int m = 0; m < N_MODES; ++m) {
        std::vector<float> v = us[m];
        std::sort(v.begin(), v.end());
        printf("%-5s : median %6.2f us per launch (min %6.2f, max %6.2f)\n", NAMES[m], v[v.size() / 2], v.front(), v.back());
    }
    return 0;
}
