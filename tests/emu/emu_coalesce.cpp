// tests/emu/emu_coalesce.cpp -- TEST HARNESS ONLY: the device code of the coalesced per-call operations (harmony_b200/csrc/hbls.cu
// co_launch) run on the host, the same way as tests/emu/emu_kernels.cpp: k_hm_gather, and the struct-layout epilogue of
// k_g2_decode_pair / k_g1_decode_jac against the one-thread g2_deserialize / g1_deserialize that blsSignatureDeserialize /
// blsPublicKeyDeserialize ran before, byte for byte.  Never linked into libhbls.so.
#define HB_HOST_EMU 1
#include <cstring>
#include <cstdint>
#include <cstddef>
#include <vector>
struct hb_dim3 { unsigned x, y, z; };
static thread_local hb_dim3 threadIdx = {0, 0, 0}, blockIdx = {0, 0, 0}, blockDim = {1, 1, 1}, gridDim = {1, 1, 1};
#define __global__
#define __shared__ static
#define __restrict__
#define __launch_bounds__(...)
struct uint4 { unsigned x, y, z, w; };
static inline void __syncwarp() {}
static inline unsigned __funnelshift_l(unsigned lo, unsigned hi, unsigned sh) { sh &= 31; return sh ? (hi << sh) | (lo >> (32 - sh)) : hi; }
static inline unsigned __ballot_sync(unsigned, bool p) { return p ? 1u : 0u; }
#include "../../harmony_b200/csrc/pairing.cuh"
static inline void __syncthreads() { if (blockDim.x == 2) hb::hb_emu_exchange(0); }
static inline unsigned atomicAdd(unsigned* p, unsigned v) { unsigned o = *p; *p += v; return o; }
static inline long long clock64() { return 0; }
template <class T> static inline T __shfl_down_sync(unsigned, T v, int) { return v; }
#include "../../harmony_b200/csrc/kernels.cuh"
using namespace hb;

template <class F> static void run_seq(unsigned grid, unsigned block, F f) {
    gridDim = {grid, 1, 1}; blockDim = {block, 1, 1};
    for (unsigned b = 0; b < grid; b++) for (unsigned t = 0; t < block; t++) { blockIdx = {b, 0, 0}; threadIdx = {t, 0, 0}; f(); }
    gridDim = {1, 1, 1}; blockDim = {1, 1, 1}; blockIdx = {0, 0, 0}; threadIdx = {0, 0, 0};
}
template <class F> static void run_pair(F f) {
    hb_emu_pair_reset();
    auto lane = [&](unsigned t) {
        gridDim = {1, 1, 1}; blockDim = {2, 1, 1}; blockIdx = {0, 0, 0}; threadIdx = {t, 0, 0};
        hb_emu.role = (int)t; hb_emu.seq = 0;
        f();
        blockDim = {1, 1, 1}; threadIdx = {0, 0, 0}; hb_emu.role = 0;
    };
    std::thread th(lane, 1u); lane(0u); th.join();
}

// k_hm_gather over n items: item i gets H(distinct message idx[i]) and its ok flag; the distinct points come from the thread-per-item
// hash kernel over m messages of msg_len bytes.  1 = every item holds exactly its distinct message's point and flag.
extern "C" int emu_hm_gather(size_t m, const uint8_t* msgs, uint32_t msg_len, size_t n, const uint32_t* idx) {
    std::vector<g2a> dh(m), hm(n); std::vector<uint8_t> dok(m), ok(n, 0xee);
    run_seq(1, (unsigned)m, [&] { k_hash_to_g2(m, msgs, msg_len, dh.data(), dok.data()); });
    memset(hm.data(), 0xa5, n * sizeof(g2a));
    run_seq((unsigned)((n + 2) / 3), 3, [&] { k_hm_gather(n, idx, dh.data(), dok.data(), hm.data(), ok.data()); });
    for (size_t i = 0; i < n; i++)
        if (idx[i] >= m || ok[i] != dok[idx[i]] || memcmp(&hm[i], &dh[idx[i]], sizeof(g2a)) != 0) return 0;
    return 1;
}

// per item, class[i]: 1 decoded, struct == g2_deserialize's point byte for byte; 2 rejected, on the curve but outside the subgroup;
// 3 rejected, not a point (non-canonical / no square root); 0 the batched decode disagrees with g2_deserialize or touched the struct
extern "C" int emu_decode_struct_g2(size_t n, const uint8_t* sigs96, uint8_t* cls) {
    int agree = 0;
    for (size_t i = 0; i < n; i++) {
        g2 want, sentinel, got; memset(&sentinel, 0x5a, sizeof sentinel); got = sentinel;
        const bool good = g2_deserialize(want, sigs96 + 96 * i, true);
        g2 tmp; const bool on_curve = g2_deserialize(tmp, sigs96 + 96 * i, false);
        uint8_t ok = 0xee;
        run_pair([&] { k_g2_decode_pair(1, sigs96 + 96 * i, (g2a*)nullptr, &ok, 1, &got); });
        bool same;
        if (good) same = ok == 1 && memcmp(&got, &want, sizeof(g2)) == 0;
        else same = ok == 0 && memcmp(&got, &sentinel, sizeof(g2)) == 0;
        cls[i] = !same ? 0 : good ? 1 : on_curve ? 2 : 3;
        agree += same;
    }
    return agree;
}
extern "C" int emu_decode_struct_g1(size_t n, const uint8_t* pks48, uint8_t* cls) {
    int agree = 0;
    for (size_t i = 0; i < n; i++) {
        g1 want, got; uint8_t ok = 0xee;
        const bool good = g1_deserialize(want, pks48 + 48 * i, true);
        g1 tmp; const bool on_curve = g1_deserialize(tmp, pks48 + 48 * i, false);
        run_seq(1, 1, [&] { k_g1_decode_jac(1, pks48 + 48 * i, &got, &ok, 1); });
        const bool same = good ? (ok == 1 && memcmp(&got, &want, sizeof(g1)) == 0) : ok == 0;      // (hbls.cu copies out only ok items)
        cls[i] = !same ? 0 : good ? 1 : on_curve ? 2 : 3;
        agree += same;
    }
    return agree;
}
