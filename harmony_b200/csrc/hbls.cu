// harmony_b200/csrc/hbls.cu -- libhbls.so: C ABI (include/hbls.h) over the sm_100a kernels.
// Host side = plumbing only (buffers, streams, launches); every group/field operation runs on the GPU.
// No CPU fallback exists: without a usable CUDA device blsInit fails and every entry point returns HBLS_ERR_CUDA.
#include <cuda_runtime.h>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <unordered_map>
#include <vector>
#include "../../include/hbls.h"
#include "coalesce.hpp"
#include "kernels.cuh"

using namespace hb;

namespace {

// per-stream scratch: a bump arena + the timing events and the pinned counters of the last batch issued on that stream.
// Calls on one stream are stream-ordered, so re-using its arena from offset 0 is safe; different streams never share one.
struct Scratch {
    uint8_t* base = nullptr; size_t cap = 0;
    cudaEvent_t ev[8] = {}; bool ev_ok = false, ev7_set = false;
    unsigned* h_counts = nullptr;            // pinned: [0] rounds re-verified exactly, [1] groups failed
    cudaEvent_t done = nullptr;
    cudaEvent_t fork = nullptr, join[2] = {}; bool forked = false;      // small batches: decode / hash on two auxiliary streams
    cudaEvent_t mid = nullptr, join2 = nullptr;                          // H(m) cached: "signature decoded" / "subgroup test done"
};
struct Ctx {
    bool ready = false;
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    cudaStream_t aux[2] = {nullptr, nullptr};               // latency path: signature decode and hash-to-G2 run beside the mask aggregation
    std::mutex mu;
    std::map<cudaStream_t, Scratch> scratch;
    std::atomic<uint64_t> launches{0};
    bool stage_timing = false; Scratch* stage_sc = nullptr;
    int batch_mode = 1;                                     // 1: random-linear-combination groups + exact pass over failed groups, 0: exact per round
    // tuning (hbls_set_param)
    long long rlc_min = 12288, rlc_g = 0, tpsm = 384, tpsm_split = 512, tpsm_light = 1024, coop_max = 4096, overlap = 1, coop_wpsm = 14, hash_coop_max = 592, mask_sort = 1, hash_split = 2, tpsm_sw = 512, hash_fallback = 0, rlc_two_phase = 2, tpsm_lines = 512, tpsm_accum = 512, tpsm_cof = 512, tpsm_dec = 512, tpsm_scale = 384, tpsm_scale_g1 = 384, scale_split = 1, decode_split = 1, exact_two_phase = 1;
    // coefficient stream: ChaCha20 keyed from /dev/urandom, block counter = call number
    uint32_t chacha_key[8] = {}; uint64_t rlc_calls = 0;
    // last batch
    hbls_batch_info info = {}; Scratch* info_sc = nullptr; bool info_valid = false;
    // last error of a call that cannot return one
    int last_err = 0; char last_err_msg[160] = {};
    // H(m) cache (device-resident, LRU): the messages a node hashes again and again -- the block hash / commit payload it SIGNS
    // itself (consensus/validator.go: prepare / commit votes) and then VERIFIES in PREPARED / COMMITTED (validator.go:219-236,
    // engine.go:630-640), the one message of a leader's vote collection (leader.go:127-290).  Keyed by the 48 zero-padded bytes
    // hash_to_fp reads (A.3: longer inputs are truncated).  Mirrors the reference's own caches on this path (BLSPubKeyCache LRU,
    // crypto/bls/mask.go:35-55; epochCtx committee cache, engine.go:727-761).
    struct HmEntry { uint8_t key[48] = {}; uint64_t stamp = 0; bool used = false, has_reader = false; cudaEvent_t filled = nullptr, read_done = nullptr; };
    static constexpr int HM_N = 64;
    g2a* hm_slots = nullptr; uint8_t* hm_ok = nullptr; HmEntry hm[HM_N];
    uint64_t hm_clock = 0, hm_hits = 0, hm_misses = 0;
    long long hm_cache = 1;                                 // hbls_set_param("hm_cache", 0) turns it off (cold-path measurements)
    // pinned host staging of the per-call operations (device -> host copies of a coalesced batch, hbls.cu co_run)
    uint8_t* pin = nullptr; size_t pin_cap = 0;
};
Ctx g;

void note_error(cudaError_t e, const char* what, const char* file, int line) {
    fprintf(stderr, "[hbls] CUDA error %s at %s:%d: %s\n", what, file, line, cudaGetErrorString(e));
    g.last_err = (int)e;
    snprintf(g.last_err_msg, sizeof g.last_err_msg, "%s: %s", what, cudaGetErrorString(e));
}
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { note_error(e_, #call, __FILE__, __LINE__); return HBLS_ERR_CUDA; } } while (0)

int ensure_init() {
    if (g.ready) return 0;
    fprintf(stderr, "[hbls] not initialised: call blsInit / hbls_init_device first (no CPU fallback)\n");
    return HBLS_ERR_CUDA;
}

struct Arena {
    uint8_t* base; size_t off = 0, cap;
    template <class T> T* take(size_t n) {
        off = (off + 255) & ~(size_t)255;
        T* p = reinterpret_cast<T*>(base + off); off += n * sizeof(T);
        return p;
    }
};
// scratch of stream s, grown to `bytes` (growing frees the old block: cudaFree waits for the device, so no kernel still reads it)
int reserve(cudaStream_t s, size_t bytes, Scratch** out) {
    Scratch& sc = g.scratch[s];
    bytes += 4096;
    if (bytes > sc.cap) {
        if (sc.base) CK(cudaFree(sc.base));
        sc.base = nullptr; sc.cap = 0;
        size_t cap = bytes + bytes / 4;
        CK(cudaMalloc(&sc.base, cap));
        sc.cap = cap;
    }
    if (!sc.h_counts) {
        CK(cudaMallocHost(&sc.h_counts, 64)); sc.h_counts[0] = sc.h_counts[1] = 0;
        CK(cudaEventCreateWithFlags(&sc.done, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&sc.fork, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&sc.join[0], cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&sc.join[1], cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&sc.mid, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&sc.join2, cudaEventDisableTiming));
    }
    sc.forked = false; sc.ev7_set = false;
    *out = &sc;
    return 0;
}
inline unsigned blocks_for(size_t n, unsigned tpb) { return (unsigned)((n + tpb - 1) / tpb); }
// pinned host staging of at least `bytes` (growing frees the old block: callers hold g.mu and have synchronised their copies)
int reserve_pinned(size_t bytes, uint8_t** out) {
    if (bytes > g.pin_cap) {
        if (g.pin) CK(cudaFreeHost(g.pin));
        g.pin = nullptr; g.pin_cap = 0;
        const size_t cap = bytes + bytes / 4 + 4096;
        CK(cudaMallocHost(&g.pin, cap));
        g.pin_cap = cap;
    }
    *out = g.pin;
    return 0;
}

// ------------------------------------------------------------------ H(m) cache.  Caller holds g.mu.  Entries are filled and read on
// whatever stream the call runs on; `filled` orders readers after the fill, `read_done` orders a later overwrite after the readers.
void hm_key(uint8_t key[48], const void* msg, size_t len) { memset(key, 0, 48); if (len) memcpy(key, msg, len > 48 ? 48 : len); }
bool hm_enabled() { return g.hm_cache != 0 && g.hm_slots != nullptr; }
// hit: stream st copies the cached point into dst / dst_ok and true is returned
bool hm_fetch(const uint8_t key[48], g2a* dst, uint8_t* dst_ok, cudaStream_t st) {
    for (int i = 0; i < Ctx::HM_N; i++) {
        Ctx::HmEntry& e = g.hm[i];
        if (!e.used || memcmp(e.key, key, 48) != 0) continue;
        cudaStreamWaitEvent(st, e.filled, 0);
        cudaMemcpyAsync(dst, g.hm_slots + i, sizeof(g2a), cudaMemcpyDeviceToDevice, st);
        cudaMemcpyAsync(dst_ok, g.hm_ok + i, 1, cudaMemcpyDeviceToDevice, st);
        cudaEventRecord(e.read_done, st); e.has_reader = true;
        e.stamp = ++g.hm_clock; g.hm_hits++;
        return true;
    }
    g.hm_misses++;
    return false;
}
// after stream st has produced H(key) in src / src_ok: keep a copy in the least recently used slot
void hm_store(const uint8_t key[48], const g2a* src, const uint8_t* src_ok, cudaStream_t st) {
    int victim = 0;
    for (int i = 0; i < Ctx::HM_N; i++) {
        if (!g.hm[i].used) { victim = i; break; }
        if (g.hm[i].stamp < g.hm[victim].stamp) victim = i;
    }
    Ctx::HmEntry& e = g.hm[victim];
    if (e.used) { cudaStreamWaitEvent(st, e.filled, 0); if (e.has_reader) cudaStreamWaitEvent(st, e.read_done, 0); }
    cudaMemcpyAsync(g.hm_slots + victim, src, sizeof(g2a), cudaMemcpyDeviceToDevice, st);
    cudaMemcpyAsync(g.hm_ok + victim, src_ok, 1, cudaMemcpyDeviceToDevice, st);
    cudaEventRecord(e.filled, st);
    memcpy(e.key, key, 48); e.used = true; e.has_reader = false; e.stamp = ++g.hm_clock;
}
#define LAUNCH(kern, grid, block, strm, ...) do { kern<<<(grid), (block), 0, (strm)>>>(__VA_ARGS__); g.launches++; } while (0)
#define LAUNCH_SMEM(kern, grid, block, smem, strm, ...) do { kern<<<(grid), (block), (smem), (strm)>>>(__VA_ARGS__); g.launches++; } while (0)

constexpr unsigned TPB = 64;      // heavy kernels: 64-thread CTAs
// persistent launch geometry for the grid-stride kernels: at most `tpsm` resident threads per SM (default 384: measured 256: 267 ms,
// 384: 263 ms, 512: 280 ms per 303 104 rounds) so the per-thread stack (Fp12 temporaries) stays in L1/L2
unsigned capped_blocks(size_t n, long long tpsm, unsigned tpb) {
    size_t cap = (size_t)g.sm_count * (size_t)((tpsm < (long long)tpb ? tpb : tpsm) / tpb);
    size_t need = (n + tpb - 1) / tpb;
    return (unsigned)(need < cap ? need : cap);
}
unsigned heavy_blocks(size_t n) { return capped_blocks(n, g.tpsm, TPB); }
unsigned light_blocks(size_t n) { return capped_blocks(n, g.tpsm_light, TPB); }       // small-state kernels: the register count decides
unsigned split_blocks(size_t nthreads) { return capped_blocks(nthreads, g.tpsm_split, HB_TPB_SPLIT); }

// hash-to-G2 of a small batch (latency path): one WARP per message while that still leaves every warp its own scheduler's worth of
// an SM (the cofactor clearing runs as VM step programs: 2.7 instead of 3.7 ms for one message), else one message per lane pair
void launch_hash_small(cudaStream_t st, size_t n, const uint8_t* d_msgs, uint32_t msg_len, g2a* hm, uint8_t* ok_hm) {
    if ((long long)n <= g.hash_coop_max) LAUNCH(k_hash_to_g2_coop, (unsigned)n, 32, st, n, d_msgs, msg_len, hm, ok_hm, (int)g.hash_fallback);
    else LAUNCH(k_hash_to_g2_pair, blocks_for(2 * n, 32), 32, st, n, d_msgs, msg_len, hm, ok_hm);
}

// ------------------------------------------------------------------ coefficient stream (host): ChaCha20 block function, RFC 8439
void chacha20_block(const uint32_t key[8], uint64_t counter, uint32_t out[16], uint32_t block = 0) {
    uint32_t st[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u, key[0], key[1], key[2], key[3], key[4], key[5], key[6], key[7],
                       (uint32_t)counter, (uint32_t)(counter >> 32), 0x68626c73u /* "hbls" */, block};
    uint32_t x[16]; memcpy(x, st, sizeof x);
    auto rotl = [](uint32_t v, int c) { return (v << c) | (v >> (32 - c)); };
    auto qr = [&](int a, int b, int c, int d) {
        x[a] += x[b]; x[d] ^= x[a]; x[d] = rotl(x[d], 16); x[c] += x[d]; x[b] ^= x[c]; x[b] = rotl(x[b], 12);
        x[a] += x[b]; x[d] ^= x[a]; x[d] = rotl(x[d], 8);  x[c] += x[d]; x[b] ^= x[c]; x[b] = rotl(x[b], 7);
    };
    for (int r = 0; r < 10; r++) { qr(0, 4, 8, 12); qr(1, 5, 9, 13); qr(2, 6, 10, 14); qr(3, 7, 11, 15); qr(0, 5, 10, 15); qr(1, 6, 11, 12); qr(2, 7, 8, 13); qr(3, 4, 9, 14); }
    for (int i = 0; i < 16; i++) out[i] = x[i] + st[i];
}
// one fresh draw per position inside a group, per call (kernels.cuh: rlc_coeffs); the low bit of each half-scalar pair is forced
// odd on the device (rlc_scale_pair), leaving 63 random bits per coefficient
rlc_coeffs rlc_draw() {
    uint32_t blk[16]; chacha20_block(g.chacha_key, ++g.rlc_calls, blk);
    rlc_coeffs co;
    for (int k = 0; k < HB_RLC_GMAX; k++) co.c[k] = ((uint64_t)blk[2 * k + 1] << 32) | blk[2 * k];
    return co;
}

// one independent draw per item (the single combined check of hbls_rlc_partial / hbls_rlc_fold)
std::vector<uint64_t> rlc_draw_items(size_t k) {
    std::vector<uint64_t> c(k); const uint64_t call = ++g.rlc_calls; uint32_t blk[16];
    for (size_t j = 0; j < k; j++) {
        if ((j & 7) == 0) chacha20_block(g.chacha_key, call, blk, (uint32_t)(j >> 3) + 1);
        c[j] = ((uint64_t)blk[2 * (j & 7) + 1] << 32) | blk[2 * (j & 7)];
    }
    return c;
}

// ------------------------------------------------------------------ one verification pass over device-resident inputs.
// batched form: groups of 8 once that still gives every SM a full CTA of lane pairs (fewer Miller-loop pairs and final exponentiations
// per round), else 4
size_t rlc_group_size(size_t B) {
    return (g.rlc_g == 4 || g.rlc_g == 8) ? (size_t)g.rlc_g : (2 * (B / 8) >= (size_t)g.sm_count * HB_TPB_SPLIT ? 8 : 4);
}
constexpr size_t RLC_CHUNK_GROUPS = 37888;             // two-phase form: groups per pass (148 SMs x 256 lane pairs)
static bool rlc_applies(size_t B);
static bool exact_two_phase(size_t B);
size_t rlc_lines_bytes(size_t B) {
    if (!g.rlc_two_phase) return 0;
    if (!rlc_applies(B)) {      // exact form through the same kernels: "groups" of one round, two pairs each
        if (!exact_two_phase(B)) return 0;
        const size_t ngc = B < RLC_CHUNK_GROUPS ? B : RLC_CHUNK_GROUPS;
        return (size_t)HB_ML_STEPS * 3 * 2 * ngc * 2 * sizeof(fp) + 256;
    }
    const size_t G = rlc_group_size(B), ng = B / G, ngc = ng < RLC_CHUNK_GROUPS ? ng : RLC_CHUNK_GROUPS;
    const size_t rlc_bytes = (size_t)HB_ML_STEPS * 3 * (G + 1) * ngc * 2 * sizeof(fp);
    // the exact pass over the rounds of failed groups runs through the same buffer ("groups" of one round, <= all rounds of the batch)
    const size_t nlc = B < RLC_CHUNK_GROUPS ? B : RLC_CHUNK_GROUPS;
    const size_t list_bytes = g.exact_two_phase ? (size_t)HB_ML_STEPS * 3 * 2 * nlc * 2 * sizeof(fp) + B * sizeof(g2a) + 256 : 0;
    return (rlc_bytes > list_bytes ? rlc_bytes : list_bytes) + 256;
}
size_t verify_scratch_bytes(size_t B) {
    return B * (sizeof(g2a) * 2 + sizeof(g1a) * 2 + sizeof(g1) + sizeof(g2) + 16 + 4 + 7) + HB_MASK_BINS * 4 + (B / HB_RLC_G + 1) * (sizeof(g2a) + 8) + 44 * 256
           + (B <= 8192 ? B * (12 * sizeof(fp2) + 3) + 1024 : 0)                // latency path: Miller values of (B, sigma) and (-apk, H(m))
           + rlc_lines_bytes(B);                                                 // two-kernel pairing: the line functions of one chunk
}
struct VerifyBufs { g2a* sig; g2a* hm; g1a* pkneg; g1* apk; uint8_t* ok_sig; uint8_t* ok_hm; uint8_t* ok_pk;
                    g1a* pk_scaled; g2* S; uint8_t* bad; g2a* Sg; uint8_t* group_ok; uint32_t* fail_list; unsigned* counts;
                    fp2* f1; uint8_t* irr1; fp2* f2; uint8_t* irr2; uint8_t* ok_sub;
                    uint16_t* mask_cost; unsigned* mask_hist; uint32_t* mask_order; fp* lines; uint8_t* verdict; };
VerifyBufs carve_verify(Arena& ar, size_t B) {
    VerifyBufs v;
    v.sig = ar.take<g2a>(B); v.hm = ar.take<g2a>(B); v.pkneg = ar.take<g1a>(B); v.apk = ar.take<g1>(B);
    v.ok_sig = ar.take<uint8_t>(B); v.ok_hm = ar.take<uint8_t>(B); v.ok_pk = ar.take<uint8_t>(B);
    v.pk_scaled = ar.take<g1a>(B); v.S = ar.take<g2>(B); v.bad = ar.take<uint8_t>(B);
    v.Sg = ar.take<g2a>(B / HB_RLC_G + 1); v.group_ok = ar.take<uint8_t>(B / HB_RLC_G + 1);
    v.fail_list = ar.take<uint32_t>(B); v.counts = ar.take<unsigned>(2);
    v.mask_cost = ar.take<uint16_t>(B); v.mask_hist = ar.take<unsigned>(HB_MASK_BINS); v.mask_order = ar.take<uint32_t>(B);
    v.verdict = ar.take<uint8_t>(B);
    v.lines = nullptr;
    if (rlc_lines_bytes(B)) v.lines = reinterpret_cast<fp*>(ar.take<uint8_t>(rlc_lines_bytes(B)));
    v.f1 = v.f2 = nullptr; v.irr1 = v.irr2 = v.ok_sub = nullptr;
    if (B <= 8192) { v.f1 = ar.take<fp2>(6 * B); v.irr1 = ar.take<uint8_t>(B); v.f2 = ar.take<fp2>(6 * B); v.irr2 = ar.take<uint8_t>(B); v.ok_sub = ar.take<uint8_t>(B); }
    return v;
}
// Small batches (latency path): the inputs are on the device from here on -- signature decode and hash-to-G2 may start on the
// auxiliary streams while the caller's stream still aggregates the public keys (launch_verify_tail joins them before the pairing).
static bool latency_path(size_t B);
void fork_point(size_t B, Scratch* sc, cudaStream_t s) {
    if (!latency_path(B) || !g.overlap || g.stage_timing) return;
    if (cudaEventRecord(sc->fork, s) == cudaSuccess) sc->forked = true;
}
// batched (random-linear-combination) form applies: default mode and a batch large enough
static bool rlc_applies(size_t B) { return g.batch_mode == 1 && (long long)B >= g.rlc_min && B >= 2 * HB_RLC_GMAX; }
static bool latency_path(size_t B) { return !rlc_applies(B) && (long long)B <= g.coop_max; }
// exact checks of batches beyond the warp-per-round range run as line kernel + accumulator kernel too (twice the lane pairs in the
// first one; the second no longer carries the running points)
static bool exact_two_phase(size_t B) { return g.rlc_two_phase >= 2 && g.exact_two_phase && !rlc_applies(B) && (long long)B > g.coop_max; }
// exact check of n rounds (contiguous arrays) as "groups" of one round through k_rlc_lines_split<1> / k_rlc_accum_split<1>
void launch_exact_two_phase(size_t n, const g2a* sig, const g1a* pkneg, const g2a* hm, const uint8_t* ok_a, const uint8_t* ok_b, const uint8_t* ok_c,
                            uint8_t* bad, uint8_t* verdict, fp* lines, uint8_t* d_results, cudaStream_t s);
#define STAGE_EV(i, sc, strm) do { if (g.stage_timing && (sc)->ev_ok) cudaEventRecord((sc)->ev[i], (strm)); } while (0)
// v.apk holds the Jacobian (aggregate) public key of every round; ok_pk (nullable) = per-round "key decoded" flags of the triple form
// h_msg (nullable): host copy of THE message when the call has a single one (one round, or a same-message batch) -- the key of the
// H(m) cache
void launch_verify_tail(size_t B, const VerifyBufs& v, Scratch* sc, const uint8_t* d_sig96, const uint8_t* d_msgs, uint32_t msg_len,
                        const uint8_t* ok_pk, uint8_t* d_results, cudaStream_t s, bool same_msg, const uint8_t* h_msg = nullptr) {
    STAGE_EV(1, sc, s);
    const bool rlc = rlc_applies(B);
    // the batched check consumes the Jacobian sums directly; -apk in affine form is then only needed for the rounds of failed groups
    // small batches (latency path): one item per lane pair, binary-GCD inversions; large ones: one item per thread, persistent
    const bool pairs = latency_path(B);
    if (!rlc) {
        if (pairs) LAUNCH(k_g1_normalize_lat, blocks_for(B, 32), 32, s, B, v.apk, v.pkneg, 1);
        else LAUNCH(k_g1_normalize, blocks_for(B, TPB), TPB, s, B, v.apk, v.pkneg, 1, (const int*)nullptr);
    }
    STAGE_EV(2, sc, s);
    const bool forked = pairs && sc->forked;              // decode on aux[0], hash on aux[1], concurrently with the work above
    cudaStream_t sd = forked ? g.aux[0] : s, sh = forked ? g.aux[1] : s;
    if (forked) { cudaStreamWaitEvent(sd, sc->fork, 0); cudaStreamWaitEvent(sh, sc->fork, 0); }
    const size_t coop_cap = (size_t)g.sm_count * (size_t)(g.coop_wpsm > 0 ? g.coop_wpsm : 1);      // resident warps (one round each)
    const unsigned coop_grid = (unsigned)(B < coop_cap ? B : coop_cap);
    const bool split_ml = forked && v.f1 != nullptr;       // Miller value of (B, sigma) on the decode stream, beside hash-to-G2
    // one message (one round, or a same-message batch): H(m) once -- from the cache when this node has hashed it before (it signed
    // it, verified it, or prefetched it)
    const bool one_msg = (same_msg && B > 1) || (B == 1 && h_msg);
    const bool use_cache = one_msg && h_msg != nullptr && hm_enabled();
    uint8_t key[48]; bool hit = false;
    if (use_cache) { hm_key(key, h_msg, msg_len); hit = hm_fetch(key, v.hm, v.ok_hm, sh); }
    // H(m) known up front: the two Miller values do not depend on each other -- (-apk, H(m)) starts right after the key aggregation
    // on the caller's stream, (B, sigma) after the decode on the decode stream with the signature's subgroup test beside it
    const bool warm = hit && split_ml;
    if (pairs) LAUNCH(k_g2_decode_pair, blocks_for(2 * B, 32), 32, sd, B, d_sig96, v.sig, v.ok_sig, warm ? 0 : 1);
    else if (g.decode_split) {
        LAUNCH(k_g2_decode, capped_blocks(B, g.tpsm_dec, TPB), TPB, s, B, d_sig96, v.sig, v.ok_sig, 0);
        LAUNCH(k_g2_subgroup, capped_blocks(B, g.tpsm_dec, TPB), TPB, s, B, v.sig, v.ok_sig);
    } else LAUNCH(k_g2_decode, capped_blocks(B, g.tpsm_dec, TPB), TPB, s, B, d_sig96, v.sig, v.ok_sig, 1);
    if (warm) {
        cudaEventRecord(sc->mid, sd);
        LAUNCH(k_miller_pq_coop, coop_grid, 32, sd, B, (const g1a*)nullptr, v.sig, v.ok_sig, v.f1, v.irr1);
    } else if (split_ml) LAUNCH(k_miller1_coop, coop_grid, 32, sd, B, v.sig, v.ok_sig, v.f1, v.irr1);
    STAGE_EV(3, sc, s);
    if (one_msg) {
        if (!hit) {
            if (pairs) launch_hash_small(sh, 1, d_msgs, msg_len, v.hm, v.ok_hm);
            else LAUNCH(k_hash_to_g2, 1, TPB, sh, (size_t)1, d_msgs, msg_len, v.hm, v.ok_hm);
            if (use_cache) hm_store(key, v.hm, v.ok_hm, sh);
        }
        if (B > 1) LAUNCH(k_broadcast_hm, blocks_for(B, 256), 256, sh, B, v.hm, v.ok_hm);
    } else if (pairs)
        launch_hash_small(sh, B, d_msgs, msg_len, v.hm, v.ok_hm);
    else if (g.hash_split && HB_BATCH_INV) {
        LAUNCH(k_hash_sw, capped_blocks(B, g.tpsm_sw, TPB), TPB, s, B, d_msgs, msg_len, v.hm, v.ok_hm);
        if (g.hash_split >= 2) {        // three kernels: map | cofactor clearing (Jacobian, into the S buffer the scaling stage fills later) | affine
            LAUNCH(k_hash_cofactor_jac, capped_blocks(B, g.tpsm_cof, TPB), TPB, s, B, (const g2a*)v.hm, (const uint8_t*)v.ok_hm, v.S);
            LAUNCH(k_g2_normalize_batch, heavy_blocks(B), TPB, s, B, (const g2*)v.S, v.hm);
        } else
            LAUNCH(k_hash_cofactor, heavy_blocks(B), TPB, s, B, v.hm, (const uint8_t*)v.ok_hm);
    } else
        LAUNCH(k_hash_to_g2, heavy_blocks(B), TPB, s, B, d_msgs, msg_len, v.hm, v.ok_hm);
    if (warm) {
        cudaEventRecord(sc->join[1], sh); cudaStreamWaitEvent(s, sc->join[1], 0);
        LAUNCH(k_miller_pq_coop, coop_grid, 32, s, B, (const g1a*)v.pkneg, v.hm, (const uint8_t*)v.ok_hm, v.f2, v.irr2);
        cudaStreamWaitEvent(sh, sc->mid, 0);
        LAUNCH(k_g2_subgroup_pair, blocks_for(2 * B, 32), 32, sh, B, v.sig, v.ok_sig, v.ok_sub);
        cudaEventRecord(sc->join2, sh); cudaEventRecord(sc->join[0], sd);
        cudaStreamWaitEvent(s, sc->join[0], 0); cudaStreamWaitEvent(s, sc->join2, 0);
        cudaMemcpyAsync(v.ok_sig, v.ok_sub, B, cudaMemcpyDeviceToDevice, s);          // decode flag := decoded AND in the subgroup
    } else if (forked) {
        cudaEventRecord(sc->join[0], sd); cudaEventRecord(sc->join[1], sh);
        cudaStreamWaitEvent(s, sc->join[0], 0); cudaStreamWaitEvent(s, sc->join[1], 0);
    }
    STAGE_EV(4, sc, s);
    hbls_batch_info& bi = g.info;
    bi = hbls_batch_info{}; bi.rounds = B; bi.mode = rlc ? 1 : 0;
    cudaMemsetAsync(v.counts, 0, 2 * sizeof(unsigned), s);
    if (rlc) {
        // batched form (north-star "batched Miller loop + shared final exponentiation"): strided groups of G rounds; G = 8 once
        // that still gives every SM a full CTA of lane pairs (fewer Miller-loop pairs and final exponentiations per round), else 4
        const size_t G = rlc_group_size(B);
        const size_t ng = B / G, nr = ng * G, tail = B - nr;
        const rlc_coeffs co = rlc_draw();
        if (g.scale_split && HB_BATCH_INV) {
            LAUNCH(k_rlc_scale_g1, capped_blocks(nr, g.tpsm_scale_g1, TPB), TPB, s, nr, ng, v.apk, co, v.pk_scaled);
            LAUNCH(k_rlc_scale_g2, capped_blocks(nr, g.tpsm_scale, TPB), TPB, s, nr, ng, v.apk, v.sig, v.hm, v.ok_sig, v.ok_hm, ok_pk, co, v.S, v.bad);
        } else
        LAUNCH(k_rlc_scale, capped_blocks(nr, g.tpsm_scale, TPB), TPB, s, nr, ng, v.apk, v.sig, v.hm, v.ok_sig, v.ok_hm, ok_pk, co, (const uint64_t*)nullptr, v.pk_scaled, v.S, v.bad);
        const bool full = 2 * ng >= (size_t)g.sm_count * HB_TPB_SPLIT;
        const unsigned pb = full ? split_blocks(2 * ng) : blocks_for(2 * ng, 64), pt = full ? HB_TPB_SPLIT : 64;
        const bool two_phase = g.rlc_two_phase && v.lines != nullptr && (full || g.rlc_two_phase >= 2);
        if (G == 8) LAUNCH(k_rlc_group_sum<8>, heavy_blocks(ng), TPB, s, ng, v.S, v.Sg);
        else LAUNCH(k_rlc_group_sum<4>, heavy_blocks(ng), TPB, s, ng, v.S, v.Sg);
        STAGE_EV(5, sc, s);
        if (two_phase) {
            // running points in their own kernel (lines to HBM, read once), accumulator + final exponentiation in the second
            for (size_t g0 = 0; g0 < ng; g0 += RLC_CHUNK_GROUPS) {
                const size_t ngc = ng - g0 < RLC_CHUNK_GROUPS ? ng - g0 : RLC_CHUNK_GROUPS;
                // one lock-stepped CTA per SM, its size = the resident threads wanted for that kernel (multiple of 64, <= 512)
                auto cta = [](long long t) { t = t < 64 ? 64 : (t > HB_TPB_SPLIT ? HB_TPB_SPLIT : t); return (unsigned)(t & ~63ll); };
                // a batch that does not fill the chip: 64-thread CTAs spread over the SMs (the line kernel has G + 1 times the lane pairs)
                const unsigned lt = full ? cta(g.tpsm_lines) : 64, at = full ? cta(g.tpsm_accum) : 64;
                const unsigned lb = full ? capped_blocks(2 * (G + 1) * ngc, lt, lt) : blocks_for(2 * (G + 1) * ngc, 64);
                const unsigned ab = full ? capped_blocks(2 * ngc, at, at) : blocks_for(2 * ngc, 64);
                if (G == 8) LAUNCH(k_rlc_lines_split<8>, lb, lt, s, ng, g0, ngc, v.pk_scaled, v.hm, v.Sg, v.lines);
                else LAUNCH(k_rlc_lines_split<4>, lb, lt, s, ng, g0, ngc, v.pk_scaled, v.hm, v.Sg, v.lines);
                if (g0 == 0) { STAGE_EV(7, sc, s); sc->ev7_set = g.stage_timing && sc->ev_ok; }       // line kernel | accumulator kernel (first chunk)
                if (G == 8) LAUNCH(k_rlc_accum_split<8>, ab, at, s, ng, g0, ngc, (const fp*)v.lines, v.bad, v.group_ok);
                else LAUNCH(k_rlc_accum_split<4>, ab, at, s, ng, g0, ngc, (const fp*)v.lines, v.bad, v.group_ok);
            }
        } else if (G == 8)
            LAUNCH_SMEM(k_rlc_pairing_split<8>, pb, pt, HB_SMEM_F ? pt * HB_SMEM_F_WORDS * 4 : 0, s, ng, v.pk_scaled, v.hm, v.Sg, v.bad, v.group_ok);
        else
            LAUNCH_SMEM(k_rlc_pairing_split<4>, pb, pt, HB_SMEM_F ? pt * HB_SMEM_F_WORDS * 4 : 0, s, ng, v.pk_scaled, v.hm, v.Sg, v.bad, v.group_ok);
        // exact pass over the rounds of failed groups only (compacted on the device; the launches are sized for the worst case and
        // return at once when the list is short or empty)
        LAUNCH(k_rlc_finish, blocks_for(nr, 256), 256, s, nr, ng, v.group_ok, d_results, v.fail_list, v.counts);
        LAUNCH(k_g1_normalize_list, heavy_blocks(nr), TPB, s, v.counts, v.fail_list, v.apk, v.pkneg, 1);
        if (two_phase && g.exact_two_phase) {
            // the listed rounds, gathered into contiguous arrays, through the line / accumulator kernels as "groups" of one round; the
            // launches are sized for the worst case and return at once beyond the device-side count
            const size_t nlc = nr < RLC_CHUNK_GROUPS ? nr : RLC_CHUNK_GROUPS;
            g2a* hm_c = reinterpret_cast<g2a*>(v.lines + (size_t)HB_ML_STEPS * 3 * 2 * nlc * 2);      // behind the chunk's lines
            g2a* sig_c = reinterpret_cast<g2a*>(v.S); g1a* pk_c = v.pk_scaled;                        // both free after the group pass
            const unsigned* cnt = v.counts;
            LAUNCH(k_exact_prepare, blocks_for(nr, 256), 256, s, nr, (const uint32_t*)v.fail_list, (const g2a*)v.sig, (const g1a*)v.pkneg, (const g2a*)v.hm,
                   (const uint8_t*)v.ok_sig, (const uint8_t*)v.ok_hm, ok_pk, pk_c, hm_c, sig_c, v.bad, d_results, cnt);
            const bool lfull = 2 * nr >= (size_t)g.sm_count * HB_TPB_SPLIT;
            const unsigned bt = lfull ? HB_TPB_SPLIT : 64;
            for (size_t g0 = 0; g0 < nr; g0 += RLC_CHUNK_GROUPS) {
                const size_t nc = nr - g0 < RLC_CHUNK_GROUPS ? nr - g0 : RLC_CHUNK_GROUPS;
                const unsigned lb = lfull ? split_blocks(4 * nc) : blocks_for(4 * nc, 64), ab = lfull ? split_blocks(2 * nc) : blocks_for(2 * nc, 64);
                LAUNCH(k_rlc_lines_split<1>, lb, bt, s, nr, g0, nc, (const g1a*)pk_c, (const g2a*)hm_c, (const g2a*)sig_c, v.lines, cnt);
                LAUNCH(k_rlc_accum_split<1>, ab, bt, s, nr, g0, nc, (const fp*)v.lines, (const uint8_t*)v.bad, v.verdict, cnt);
            }
            LAUNCH(k_exact_publish, blocks_for(nr, 256), 256, s, nr, (const uint32_t*)v.fail_list, (const uint8_t*)v.verdict, d_results, cnt);
        } else if (2 * nr >= (size_t)g.sm_count * HB_TPB_SPLIT)
            LAUNCH(k_pairing_verify_split_list, split_blocks(2 * nr), HB_TPB_SPLIT, s, v.counts, v.fail_list, v.sig, v.pkneg, v.hm, v.ok_sig, v.ok_hm, ok_pk, d_results);
        else
            LAUNCH(k_pairing_verify_split_list, blocks_for(2 * nr, 64), 64, s, v.counts, v.fail_list, v.sig, v.pkneg, v.hm, v.ok_sig, v.ok_hm, ok_pk, d_results);
        LAUNCH(k_pairing_fixup_list, heavy_blocks(nr), TPB, s, v.counts, v.fail_list, v.sig, v.pkneg, v.hm, v.ok_sig, v.ok_hm, ok_pk, d_results);
        if (tail) {       // the < G rounds that do not fill a group are always verified exactly
            LAUNCH(k_g1_normalize, 1, TPB, s, tail, v.apk + nr, v.pkneg + nr, 1, (const int*)nullptr);
            LAUNCH(k_pairing_verify_split, blocks_for(2 * tail, 64), 64, s, tail, v.sig + nr, v.pkneg + nr, v.hm + nr, v.ok_sig + nr, v.ok_hm + nr,
                   ok_pk ? ok_pk + nr : (const uint8_t*)nullptr, d_results + nr, (const int*)nullptr);
            LAUNCH(k_pairing_fixup, 1, TPB, s, tail, v.sig + nr, v.pkneg + nr, v.hm + nr, v.ok_sig + nr, v.ok_hm + nr,
                   ok_pk ? ok_pk + nr : (const uint8_t*)nullptr, d_results + nr, (const int*)nullptr);
        }
        bi.group_size = (int32_t)G; bi.groups = ng; bi.tail_rounds = (uint32_t)tail; bi.cta_threads = pt;
    } else {
        // exact form at every batch size: a lane pair per round.  Large batches use 512-thread lock-stepped CTAs (one per SM),
        // small ones 64-thread CTAs spread over the SMs.
        STAGE_EV(5, sc, s);
        const bool full = 2 * B >= (size_t)g.sm_count * HB_TPB_SPLIT;
        const bool coop = (long long)B <= g.coop_max;        // latency form: one warp per round (vm.cuh), up to 14 resident rounds per SM (15 KB of slots each)
        if (coop && warm)
            LAUNCH(k_fe2_coop, coop_grid, 32, s, B, v.f1, v.irr1, v.f2, v.irr2, v.ok_sig, v.ok_hm, ok_pk, (const uint8_t*)nullptr, d_results);
        else if (coop && split_ml)
            LAUNCH(k_pairing_coop2, coop_grid, 32, s, B, v.f1, v.irr1, v.pkneg, v.hm, v.ok_sig, v.ok_hm, ok_pk, d_results);
        else if (coop)
            LAUNCH(k_pairing_coop, coop_grid, 32, s, B, v.sig, v.pkneg, v.hm, v.ok_sig, v.ok_hm, ok_pk, d_results);
        else if (exact_two_phase(B) && v.lines)
            launch_exact_two_phase(B, v.sig, v.pkneg, v.hm, v.ok_sig, v.ok_hm, ok_pk, v.bad, v.verdict, v.lines, d_results, s);
        else if (full)
            LAUNCH(k_pairing_verify_split, split_blocks(2 * B), HB_TPB_SPLIT, s, B, v.sig, v.pkneg, v.hm, v.ok_sig, v.ok_hm, ok_pk, d_results, (const int*)nullptr);
        else
            LAUNCH(k_pairing_verify_split, blocks_for(2 * B, 64), 64, s, B, v.sig, v.pkneg, v.hm, v.ok_sig, v.ok_hm, ok_pk, d_results, (const int*)nullptr);
        LAUNCH(k_pairing_fixup, heavy_blocks(B), TPB, s, B, v.sig, v.pkneg, v.hm, v.ok_sig, v.ok_hm, ok_pk, d_results, (const int*)nullptr);
        bi.cta_threads = coop ? 32 : (full ? HB_TPB_SPLIT : 64);
    }
    STAGE_EV(6, sc, s);
    cudaMemcpyAsync(sc->h_counts, v.counts, 2 * sizeof(unsigned), cudaMemcpyDeviceToHost, s);
    cudaEventRecord(sc->done, s);
    g.info_sc = sc; g.info_valid = true;
    if (g.stage_timing && sc->ev_ok) g.stage_sc = sc;
}

void launch_exact_two_phase(size_t n, const g2a* sig, const g1a* pkneg, const g2a* hm, const uint8_t* ok_a, const uint8_t* ok_b, const uint8_t* ok_c,
                            uint8_t* bad, uint8_t* verdict, fp* lines, uint8_t* d_results, cudaStream_t s) {
    LAUNCH(k_exact_prepare, blocks_for(n, 256), 256, s, n, (const uint32_t*)nullptr, sig, pkneg, hm, ok_a, ok_b, ok_c,
           (g1a*)nullptr, (g2a*)nullptr, (g2a*)nullptr, bad, d_results);
    const bool full = 2 * n >= (size_t)g.sm_count * HB_TPB_SPLIT;
    for (size_t g0 = 0; g0 < n; g0 += RLC_CHUNK_GROUPS) {
        const size_t nc = n - g0 < RLC_CHUNK_GROUPS ? n - g0 : RLC_CHUNK_GROUPS;
        const unsigned bt = full ? HB_TPB_SPLIT : 64;
        const unsigned lb = full ? split_blocks(4 * nc) : blocks_for(4 * nc, 64), ab = full ? split_blocks(2 * nc) : blocks_for(2 * nc, 64);
        LAUNCH(k_rlc_lines_split<1>, lb, bt, s, n, g0, nc, pkneg, hm, sig, lines);
        LAUNCH(k_rlc_accum_split<1>, ab, bt, s, n, g0, nc, (const fp*)lines, (const uint8_t*)bad, verdict);
    }
    LAUNCH(k_exact_publish, blocks_for(n, 256), 256, s, n, (const uint32_t*)nullptr, (const uint8_t*)verdict, d_results);
}

int single_op(int op, const void* a, size_t an, const void* b, size_t bn, void* out, size_t on, int* rc_out, uint32_t len = 0) {
    if (int e = ensure_init()) return e;
    std::lock_guard<std::mutex> lk(g.mu);
    Scratch* sc; if (int e = reserve(g.stream, an + bn + on + 4096, &sc)) return e;
    Arena ar{sc->base, 0, sc->cap};
    uint8_t* da = ar.take<uint8_t>(an ? an : 1); uint8_t* db = ar.take<uint8_t>(bn ? bn : 1);
    uint8_t* dout = ar.take<uint8_t>(on ? on : 1); int* drc = ar.take<int>(1);
    if (an) CK(cudaMemcpyAsync(da, a, an, cudaMemcpyHostToDevice, g.stream));
    if (bn) CK(cudaMemcpyAsync(db, b, bn, cudaMemcpyHostToDevice, g.stream));
    LAUNCH(k_single, 1, 32, g.stream, op, da, db, dout, drc, len);
    int rc = 0;
    CK(cudaMemcpyAsync(&rc, drc, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
    CK(cudaStreamSynchronize(g.stream));
    if (on && rc >= 0 && !(op == OP_MAP_SER && rc != 0))
        CK(cudaMemcpy(out, dout, on, cudaMemcpyDeviceToHost));
    *rc_out = rc;
    return 0;
}

// sk (little-endian u64 x 4, < r < Z^4) -> its four base-Z digits, Z = |z| = 0xd201000000010000 (plain long division on the host)
bool sk_digits_base_z(const uint64_t sk[4], uint64_t dig[4]) {
    const uint64_t Z = 0xd201000000010000ull;
    uint64_t v[4] = {sk[0], sk[1], sk[2], sk[3]};
    for (int k = 0; k < 3; k++) {
        unsigned __int128 rem = 0;
        for (int i = 3; i >= 0; i--) { const unsigned __int128 cur = (rem << 64) | v[i]; v[i] = (uint64_t)(cur / Z); rem = cur % Z; }
        dig[k] = (uint64_t)rem;
    }
    dig[3] = v[0];
    return (v[1] | v[2] | v[3]) == 0;                 // always for sk < r < Z^4; a hand-filled struct >= Z^4 takes the plain ladder
}

// r (BLS12-381 group order), little-endian u64
const uint64_t R_ORDER[4] = {0xffffffff00000001ull, 0x53bda402fffe5bfeull, 0x3339d80809a1d805ull, 0x73eda753299d7d48ull};
bool scalar_lt_r(const uint64_t k[4]) {
    for (int i = 3; i >= 0; i--) { if (k[i] < R_ORDER[i]) return true; if (k[i] > R_ORDER[i]) return false; }
    return false;
}

// SHA-256 (host; GetAddress = first 20 bytes of SHA-256 of the serialized key)
struct Sha256 {
    static uint32_t rotr(uint32_t x, int n) { return (x >> n) | (x << (32 - n)); }
    static void digest(const uint8_t* msg, size_t len, uint8_t out[32]) {
        static const uint32_t K[64] = {
            0x428a2f98,0x71374491,0xb5c0fbcf,0xe9b5dba5,0x3956c25b,0x59f111f1,0x923f82a4,0xab1c5ed5,0xd807aa98,0x12835b01,0x243185be,0x550c7dc3,0x72be5d74,0x80deb1fe,0x9bdc06a7,0xc19bf174,
            0xe49b69c1,0xefbe4786,0x0fc19dc6,0x240ca1cc,0x2de92c6f,0x4a7484aa,0x5cb0a9dc,0x76f988da,0x983e5152,0xa831c66d,0xb00327c8,0xbf597fc7,0xc6e00bf3,0xd5a79147,0x06ca6351,0x14292967,
            0x27b70a85,0x2e1b2138,0x4d2c6dfc,0x53380d13,0x650a7354,0x766a0abb,0x81c2c92e,0x92722c85,0xa2bfe8a1,0xa81a664b,0xc24b8b70,0xc76c51a3,0xd192e819,0xd6990624,0xf40e3585,0x106aa070,
            0x19a4c116,0x1e376c08,0x2748774c,0x34b0bcb5,0x391c0cb3,0x4ed8aa4a,0x5b9cca4f,0x682e6ff3,0x748f82ee,0x78a5636f,0x84c87814,0x8cc70208,0x90befffa,0xa4506ceb,0xbef9a3f7,0xc67178f2};
        uint32_t h[8] = {0x6a09e667,0xbb67ae85,0x3c6ef372,0xa54ff53a,0x510e527f,0x9b05688c,0x1f83d9ab,0x5be0cd19};
        std::vector<uint8_t> m(msg, msg + len);
        m.push_back(0x80);
        while (m.size() % 64 != 56) m.push_back(0);
        uint64_t bits = (uint64_t)len * 8;
        for (int i = 7; i >= 0; i--) m.push_back((uint8_t)(bits >> (8 * i)));
        for (size_t off = 0; off < m.size(); off += 64) {
            uint32_t w[64];
            for (int i = 0; i < 16; i++) w[i] = ((uint32_t)m[off + 4 * i] << 24) | ((uint32_t)m[off + 4 * i + 1] << 16) | ((uint32_t)m[off + 4 * i + 2] << 8) | m[off + 4 * i + 3];
            for (int i = 16; i < 64; i++) {
                uint32_t s0 = rotr(w[i - 15], 7) ^ rotr(w[i - 15], 18) ^ (w[i - 15] >> 3), s1 = rotr(w[i - 2], 17) ^ rotr(w[i - 2], 19) ^ (w[i - 2] >> 10);
                w[i] = w[i - 16] + s0 + w[i - 7] + s1;
            }
            uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], gg = h[6], hh = h[7];
            for (int i = 0; i < 64; i++) {
                uint32_t S1 = rotr(e, 6) ^ rotr(e, 11) ^ rotr(e, 25), ch = (e & f) ^ (~e & gg), t1 = hh + S1 + ch + K[i] + w[i];
                uint32_t S0 = rotr(a, 2) ^ rotr(a, 13) ^ rotr(a, 22), mj = (a & b) ^ (a & c) ^ (b & c), t2 = S0 + mj;
                hh = gg; gg = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
            }
            h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += gg; h[7] += hh;
        }
        for (int i = 0; i < 8; i++) for (int j = 0; j < 4; j++) out[4 * i + j] = (uint8_t)(h[i] >> (24 - 8 * j));
    }
};

// SHA-512 (host; only for the test-only blsSign/blsVerify string API: mcl Fp::setHashOf, SURVEY A.7)
struct Sha512 {
    static uint64_t rotr(uint64_t x, int n) { return (x >> n) | (x << (64 - n)); }
    static void digest(const uint8_t* msg, size_t len, uint8_t out[64]) {
        static const uint64_t K[80] = {
            0x428a2f98d728ae22ull,0x7137449123ef65cdull,0xb5c0fbcfec4d3b2full,0xe9b5dba58189dbbcull,0x3956c25bf348b538ull,0x59f111f1b605d019ull,0x923f82a4af194f9bull,0xab1c5ed5da6d8118ull,
            0xd807aa98a3030242ull,0x12835b0145706fbeull,0x243185be4ee4b28cull,0x550c7dc3d5ffb4e2ull,0x72be5d74f27b896full,0x80deb1fe3b1696b1ull,0x9bdc06a725c71235ull,0xc19bf174cf692694ull,
            0xe49b69c19ef14ad2ull,0xefbe4786384f25e3ull,0x0fc19dc68b8cd5b5ull,0x240ca1cc77ac9c65ull,0x2de92c6f592b0275ull,0x4a7484aa6ea6e483ull,0x5cb0a9dcbd41fbd4ull,0x76f988da831153b5ull,
            0x983e5152ee66dfabull,0xa831c66d2db43210ull,0xb00327c898fb213full,0xbf597fc7beef0ee4ull,0xc6e00bf33da88fc2ull,0xd5a79147930aa725ull,0x06ca6351e003826full,0x142929670a0e6e70ull,
            0x27b70a8546d22ffcull,0x2e1b21385c26c926ull,0x4d2c6dfc5ac42aedull,0x53380d139d95b3dfull,0x650a73548baf63deull,0x766a0abb3c77b2a8ull,0x81c2c92e47edaee6ull,0x92722c851482353bull,
            0xa2bfe8a14cf10364ull,0xa81a664bbc423001ull,0xc24b8b70d0f89791ull,0xc76c51a30654be30ull,0xd192e819d6ef5218ull,0xd69906245565a910ull,0xf40e35855771202aull,0x106aa07032bbd1b8ull,
            0x19a4c116b8d2d0c8ull,0x1e376c085141ab53ull,0x2748774cdf8eeb99ull,0x34b0bcb5e19b48a8ull,0x391c0cb3c5c95a63ull,0x4ed8aa4ae3418acbull,0x5b9cca4f7763e373ull,0x682e6ff3d6b2b8a3ull,
            0x748f82ee5defb2fcull,0x78a5636f43172f60ull,0x84c87814a1f0ab72ull,0x8cc702081a6439ecull,0x90befffa23631e28ull,0xa4506cebde82bde9ull,0xbef9a3f7b2c67915ull,0xc67178f2e372532bull,
            0xca273eceea26619cull,0xd186b8c721c0c207ull,0xeada7dd6cde0eb1eull,0xf57d4f7fee6ed178ull,0x06f067aa72176fbaull,0x0a637dc5a2c898a6ull,0x113f9804bef90daeull,0x1b710b35131c471bull,
            0x28db77f523047d84ull,0x32caab7b40c72493ull,0x3c9ebe0a15c9bebcull,0x431d67c49c100d4cull,0x4cc5d4becb3e42b6ull,0x597f299cfc657e2aull,0x5fcb6fab3ad6faecull,0x6c44198c4a475817ull};
        uint64_t h[8] = {0x6a09e667f3bcc908ull,0xbb67ae8584caa73bull,0x3c6ef372fe94f82bull,0xa54ff53a5f1d36f1ull,0x510e527fade682d1ull,0x9b05688c2b3e6c1full,0x1f83d9abfb41bd6bull,0x5be0cd19137e2179ull};
        std::vector<uint8_t> m(msg, msg + len);
        m.push_back(0x80);
        while (m.size() % 128 != 112) m.push_back(0);
        for (int i = 0; i < 8; i++) m.push_back(0);
        uint64_t bits = (uint64_t)len * 8;
        for (int i = 7; i >= 0; i--) m.push_back((uint8_t)(bits >> (8 * i)));
        for (size_t off = 0; off < m.size(); off += 128) {
            uint64_t w[80];
            for (int i = 0; i < 16; i++) { w[i] = 0; for (int j = 0; j < 8; j++) w[i] = (w[i] << 8) | m[off + 8 * i + j]; }
            for (int i = 16; i < 80; i++) {
                uint64_t s0 = rotr(w[i - 15], 1) ^ rotr(w[i - 15], 8) ^ (w[i - 15] >> 7);
                uint64_t s1 = rotr(w[i - 2], 19) ^ rotr(w[i - 2], 61) ^ (w[i - 2] >> 6);
                w[i] = w[i - 16] + s0 + w[i - 7] + s1;
            }
            uint64_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], gg = h[6], hh = h[7];
            for (int i = 0; i < 80; i++) {
                uint64_t S1 = rotr(e, 14) ^ rotr(e, 18) ^ rotr(e, 41), ch = (e & f) ^ (~e & gg);
                uint64_t t1 = hh + S1 + ch + K[i] + w[i];
                uint64_t S0 = rotr(a, 28) ^ rotr(a, 34) ^ rotr(a, 39), mj = (a & b) ^ (a & c) ^ (b & c);
                uint64_t t2 = S0 + mj;
                hh = gg; gg = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
            }
            h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += gg; h[7] += hh;
        }
        for (int i = 0; i < 8; i++) for (int j = 0; j < 8; j++) out[8 * i + j] = (uint8_t)(h[i] >> (56 - 8 * j));
    }
};

}  // namespace

struct hbls_committee {
    size_t n = 0;
    g1a* table = nullptr;       // device, affine, Montgomery
    g1* total = nullptr;        // device, sum of all rows (lets dense bitmaps be aggregated from their complement)
    ~hbls_committee() { if (table) cudaFree(table); if (total) cudaFree(total); }
};
struct hbls_mask {
    const hbls_committee* c = nullptr;
    std::vector<uint8_t> bitmap;        // Mask.Bitmap (host)
    g1* d_acc = nullptr;                // Mask.AggregatePublic (device, Jacobian)
    ~hbls_mask() { if (d_acc) cudaFree(d_acc); }
};
struct hbls_ballot_box {
    const hbls_committee* c = nullptr;
    std::vector<uint8_t> collected;     // signers already counted
    g2* d_sum = nullptr;                // running aggregate signature (device, Jacobian)
    ~hbls_ballot_box() { if (d_sum) cudaFree(d_sum); }
};

namespace {
int popcount_slots(const uint8_t* bm, size_t n) {          // set bits among slots i < n only (padding bits of the last byte never count)
    int c = 0;
    for (size_t i = 0; i < (n >> 3); i++) c += __builtin_popcount(bm[i]);
    if (n & 7) c += __builtin_popcount(bm[n >> 3] & ((1u << (n & 7)) - 1u));
    return c;
}
bool all_messages_equal(const uint8_t* msgs, size_t n, size_t msg_len) {
    for (size_t i = 1; i < n; i++) if (memcmp(msgs, msgs + i * msg_len, msg_len) != 0) return false;
    return n > 1;
}
// rounds against one committee, everything device-resident
int agg_verify_device_locked(const hbls_committee* c, size_t B, const uint8_t* d_bitmaps, size_t blen, const uint8_t* d_sigs,
                             const uint8_t* d_msgs, size_t msg_len, uint8_t* d_results, cudaStream_t s, Scratch* sc, Arena& ar, bool same_msg,
                             VerifyBufs* v_out = nullptr, const uint8_t* h_msg = nullptr) {
    VerifyBufs v = carve_verify(ar, B);
    fork_point(B, sc, s);
    STAGE_EV(0, sc, s);
    if (B >= (size_t)g.sm_count * 256)
    {
        // rounds sorted by the number of point additions they need (device counting sort), so that the lanes of a warp finish together
        const uint32_t* order = nullptr;
        if (g.mask_sort && B <= 0xffffffffull) {
            cudaMemsetAsync(v.mask_hist, 0, HB_MASK_BINS * sizeof(unsigned), s);
            LAUNCH(k_mask_count, blocks_for(B, 256), 256, s, B, c->n, d_bitmaps, blen, v.mask_cost, v.mask_hist);
            LAUNCH(k_mask_scan, 1, 32, s, v.mask_hist);
            LAUNCH(k_mask_scatter, blocks_for(B, 256), 256, s, B, v.mask_cost, v.mask_hist, v.mask_order);
            order = v.mask_order;
        }
        LAUNCH(k_mask_aggregate_serial, light_blocks(B), TPB, s, B, c->n, c->table, c->total, d_bitmaps, blen, v.apk, order);
    }
    else
        LAUNCH(k_mask_aggregate, blocks_for(B * 32, 128), 128, s, B, c->n, c->table, d_bitmaps, blen, v.apk);
    launch_verify_tail(B, v, sc, d_sigs, d_msgs, (uint32_t)msg_len, nullptr, d_results, s, same_msg, h_msg);
    if (v_out) *v_out = v;
    return 0;
}
void ensure_stage_events(Scratch* sc) {
    if (g.stage_timing && !sc->ev_ok) { for (int i = 0; i < 8; i++) cudaEventCreate(&sc->ev[i]); sc->ev_ok = true; }
}
}  // namespace

extern "C" {

int hbls_init_device(int device) {
    std::lock_guard<std::mutex> lk(g.mu);
    if (g.ready) return 0;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        fprintf(stderr, "[hbls] no CUDA device (%s): this backend has no CPU fallback\n", e == cudaSuccess ? "count = 0" : cudaGetErrorString(e));
        return HBLS_ERR_CUDA;
    }
    if (device < 0 || device >= count) device = 0;
    CK(cudaSetDevice(device));
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, device));
    g.device = device; g.sm_count = prop.multiProcessorCount;
    CK(cudaStreamCreateWithFlags(&g.stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&g.aux[0], cudaStreamNonBlocking)); CK(cudaStreamCreateWithFlags(&g.aux[1], cudaStreamNonBlocking));
    { FILE* f = fopen("/dev/urandom", "rb"); if (!f || fread(g.chacha_key, 1, 32, f) != 32) { if (f) fclose(f); fprintf(stderr, "[hbls] cannot read /dev/urandom\n"); return HBLS_ERR_CUDA; } fclose(f); }
    auto envll = [](const char* name, long long dflt) { const char* e = getenv(name); return e ? atoll(e) : dflt; };
    g.rlc_min = envll("HBLS_RLC_MIN", 12288); g.rlc_g = envll("HBLS_RLC_G", 0); g.coop_max = envll("HBLS_COOP_MAX", 4096);
    g.tpsm = envll("HBLS_TPSM", 384); g.tpsm_split = envll("HBLS_TPSM_SPLIT", 512); g.tpsm_light = envll("HBLS_TPSM_LIGHT", 1024);
    // the heavy kernels keep their Fp12 temporaries in per-thread local memory: give L1 the whole 228 KB
#if HB_SMEM_F
    cudaFuncSetAttribute(k_rlc_pairing_split<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, HB_TPB_SPLIT * HB_SMEM_F_WORDS * 4);
    cudaFuncSetAttribute(k_rlc_pairing_split<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, HB_TPB_SPLIT * HB_SMEM_F_WORDS * 4);
#else
    cudaFuncSetAttribute(k_rlc_pairing_split<4>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_rlc_pairing_split<8>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
#endif
    cudaFuncSetAttribute(k_rlc_lines_split<1>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_rlc_accum_split<1>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_rlc_lines_split<4>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_rlc_lines_split<8>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_rlc_accum_split<4>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_rlc_accum_split<8>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_pairing_verify_split, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_pairing_verify_split_list, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_hash_to_g2, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_g2_decode, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_rlc_scale, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_mask_aggregate_serial, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_mask_aggregate, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    CK(cudaMalloc(&g.hm_slots, Ctx::HM_N * sizeof(g2a))); CK(cudaMalloc(&g.hm_ok, Ctx::HM_N));
    for (int i = 0; i < Ctx::HM_N; i++) {
        CK(cudaEventCreateWithFlags(&g.hm[i].filled, cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&g.hm[i].read_done, cudaEventDisableTiming));
    }
    g.hm_cache = envll("HBLS_HM_CACHE", 1); g.mask_sort = envll("HBLS_MASK_SORT", 1); g.hash_coop_max = envll("HBLS_HASH_COOP_MAX", 592);
    g.rlc_two_phase = envll("HBLS_RLC_2P", 2); g.tpsm_lines = envll("HBLS_TPSM_LINES", 512); g.tpsm_accum = envll("HBLS_TPSM_ACCUM", 512); g.tpsm_cof = envll("HBLS_TPSM_COF", 512); g.tpsm_dec = envll("HBLS_TPSM_DEC", 512); g.tpsm_scale = envll("HBLS_TPSM_SCALE", 384); g.tpsm_scale_g1 = envll("HBLS_TPSM_SCALE_G1", 384); g.scale_split = envll("HBLS_SCALE_SPLIT", 1); g.decode_split = envll("HBLS_DECODE_SPLIT", 1); g.exact_two_phase = envll("HBLS_EXACT_2P", 1);
    g.hash_split = envll("HBLS_HASH_SPLIT", 2); g.tpsm_sw = envll("HBLS_TPSM_SW", 512);
    cudaFuncSetAttribute(k_hash_sw, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_hash_cofactor, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_hash_cofactor_jac, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    cudaFuncSetAttribute(k_g2_normalize_batch, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    g.ready = true;
    return 0;
}
int blsInit(int curve, int compiledTimeVar) {
    if (curve != HBLS_BLS12_381 || compiledTimeVar != HBLS_COMPILED_TIME_VAR) return -1;
    const char* d = getenv("HBLS_DEVICE");
    if (!d) d = getenv("LOCAL_RANK");
    return hbls_init_device(d ? atoi(d) : 0);
}
uint64_t hbls_kernel_launch_count(void) { return g.launches.load(); }
int hbls_build_info(void) { return (HB_BATCH_INV ? 1 : 0) | (HB_BATCH_K << 8); }
void hbls_set_batch_mode(int mode) { std::lock_guard<std::mutex> lk(g.mu); g.batch_mode = mode ? 1 : 0; }
int hbls_get_batch_mode(void) { std::lock_guard<std::mutex> lk(g.mu); return g.batch_mode; }
static long long* param_slot(const char* name) {
    if (!name) return nullptr;
    if (!strcmp(name, "rlc_min")) return &g.rlc_min;
    if (!strcmp(name, "rlc_g")) return &g.rlc_g;
    if (!strcmp(name, "tpsm")) return &g.tpsm;
    if (!strcmp(name, "tpsm_split")) return &g.tpsm_split;
    if (!strcmp(name, "tpsm_light")) return &g.tpsm_light;
    if (!strcmp(name, "coop_max")) return &g.coop_max;
    if (!strcmp(name, "overlap")) return &g.overlap;
    if (!strcmp(name, "coop_wpsm")) return &g.coop_wpsm;
    if (!strcmp(name, "hm_cache")) return &g.hm_cache;
    if (!strcmp(name, "hash_coop_max")) return &g.hash_coop_max;
    if (!strcmp(name, "mask_sort")) return &g.mask_sort;
    if (!strcmp(name, "hash_split")) return &g.hash_split;
    if (!strcmp(name, "hash_fallback")) return &g.hash_fallback;
    if (!strcmp(name, "rlc_two_phase")) return &g.rlc_two_phase;
    if (!strcmp(name, "tpsm_cof")) return &g.tpsm_cof;
    if (!strcmp(name, "tpsm_dec")) return &g.tpsm_dec;
    if (!strcmp(name, "tpsm_scale")) return &g.tpsm_scale;
    if (!strcmp(name, "tpsm_scale_g1")) return &g.tpsm_scale_g1;
    if (!strcmp(name, "scale_split")) return &g.scale_split;
    if (!strcmp(name, "decode_split")) return &g.decode_split;
    if (!strcmp(name, "exact_two_phase")) return &g.exact_two_phase;
    if (!strcmp(name, "tpsm_lines")) return &g.tpsm_lines;
    if (!strcmp(name, "tpsm_accum")) return &g.tpsm_accum;
    if (!strcmp(name, "tpsm_sw")) return &g.tpsm_sw;
    return nullptr;
}
int hbls_set_param(const char* name, long long value) {
    std::lock_guard<std::mutex> lk(g.mu);
    long long* p = param_slot(name);
    if (!p || value < 0) return HBLS_ERR_ARG;
    if (p == &g.rlc_g && value != 0 && value != 4 && value != 8) return HBLS_ERR_ARG;
    *p = value; return 0;
}
long long hbls_get_param(const char* name) { std::lock_guard<std::mutex> lk(g.mu); long long* p = param_slot(name); return p ? *p : -1; }
int hbls_last_error(char* msg, size_t msg_cap) {
    std::lock_guard<std::mutex> lk(g.mu);
    int e = g.last_err;
    if (msg && msg_cap) { strncpy(msg, g.last_err_msg, msg_cap - 1); msg[msg_cap - 1] = 0; }
    g.last_err = 0; g.last_err_msg[0] = 0;
    return e;
}
int hbls_last_batch_info(hbls_batch_info* out) {
    std::lock_guard<std::mutex> lk(g.mu);
    if (!out || !g.info_valid || !g.info_sc) return HBLS_ERR_ARG;
    CK(cudaEventSynchronize(g.info_sc->done));
    *out = g.info;
    out->rounds_rechecked = g.info_sc->h_counts[0]; out->groups_failed = g.info_sc->h_counts[1];
    return 0;
}

// ------------------------------------------------------------------ secret keys (host bytes; no group arithmetic)
int blsSecretKeySetByCSPRNG(blsSecretKey* sec) {
    FILE* f = fopen("/dev/urandom", "rb");
    if (!f) return -1;
    size_t got = fread(sec->d, 1, 32, f); fclose(f);
    if (got != 32) return -1;
    sec->d[3] &= 0x3fffffffffffffffull;          // < 2^254 < r
    return 0;
}
size_t blsSecretKeySerialize(void* buf, size_t maxBufSize, const blsSecretKey* sec) { if (maxBufSize < 32) return 0; memcpy(buf, sec->d, 32); return 32; }
size_t blsSecretKeyDeserialize(blsSecretKey* sec, const void* buf, size_t bufSize) {
    if (bufSize < 32) return 0;
    uint64_t k[4]; memcpy(k, buf, 32);
    if (!scalar_lt_r(k)) return 0;
    memcpy(sec->d, k, 32); return 32;
}
int blsSecretKeyIsEqual(const blsSecretKey* l, const blsSecretKey* r) { return memcmp(l, r, 32) == 0; }

// ------------------------------------------------------------------ single-element group ops.  The herumi signatures of Add / Sub /
// GetPublicKey are void: on a CUDA failure the destination becomes the identity and the error is kept for hbls_last_error().
void blsPublicKeyAdd(blsPublicKey* pub, const blsPublicKey* rhs) { int rc; if (single_op(OP_G1_ADD, pub, 144, rhs, 144, pub, 144, &rc)) memset(pub, 0, sizeof *pub); }
void blsPublicKeySub(blsPublicKey* pub, const blsPublicKey* rhs) { int rc; if (single_op(OP_G1_SUB, pub, 144, rhs, 144, pub, 144, &rc)) memset(pub, 0, sizeof *pub); }
void blsSignatureAdd(blsSignature* sig, const blsSignature* rhs) { int rc; if (single_op(OP_G2_ADD, sig, 288, rhs, 288, sig, 288, &rc)) memset(sig, 0, sizeof *sig); }
int blsPublicKeyIsEqual(const blsPublicKey* l, const blsPublicKey* r) { int rc = 0; if (single_op(OP_G1_EQ, l, 144, r, 144, nullptr, 0, &rc)) return 0; return rc; }
int blsSignatureIsEqual(const blsSignature* l, const blsSignature* r) { int rc = 0; if (single_op(OP_G2_EQ, l, 288, r, 288, nullptr, 0, &rc)) return 0; return rc; }
size_t blsPublicKeySerialize(void* buf, size_t maxBufSize, const blsPublicKey* pub) {
    if (maxBufSize < 48) return 0; int rc = 0; if (single_op(OP_G1_SER, pub, 144, nullptr, 0, buf, 48, &rc)) return 0; return rc == 48 ? 48 : 0; }
size_t blsSignatureSerialize(void* buf, size_t maxBufSize, const blsSignature* sig) {
    if (maxBufSize < 96) return 0; int rc = 0; if (single_op(OP_G2_SER, sig, 288, nullptr, 0, buf, 96, &rc)) return 0; return rc == 96 ? 96 : 0; }
int hbls_map_to_g2(const void* msg, size_t msg_len, uint8_t out96[96]) {
    if (msg_len > 48) msg_len = 48;      // only the first 48 bytes matter (SURVEY A.3)
    int rc = -1; if (int e = single_op(OP_MAP_SER, msg, msg_len, nullptr, 0, out96, 96, &rc, (uint32_t)msg_len)) return e; return rc; }
// asynchronous: enqueues H(msg) on the hash stream and returns; a later SignHash / VerifyHash / aggregate-verify of that message
// finds the point in the cache (stream-ordered after the fill).  0 ok (also when already cached or the cache is off).
int hbls_hash_prefetch(const void* msg, size_t msg_len) {
    if (int e = ensure_init()) return e;
    std::lock_guard<std::mutex> lk(g.mu);
    if (!hm_enabled()) return 0;
    if (msg_len > 48) msg_len = 48;
    uint8_t key[48]; hm_key(key, msg, msg_len);
    for (int i = 0; i < Ctx::HM_N; i++) if (g.hm[i].used && memcmp(g.hm[i].key, key, 48) == 0) { g.hm[i].stamp = ++g.hm_clock; return 0; }
    cudaStream_t st = g.aux[1];
    Scratch* sc; if (int e = reserve(st, 4096, &sc)) return e;
    Arena ar{sc->base, 0, sc->cap};
    uint8_t* dmsg = ar.take<uint8_t>(64); g2a* dhm = ar.take<g2a>(1); uint8_t* dok = ar.take<uint8_t>(1);
    // the 48 key bytes ARE the bytes hash_to_fp reads (pageable source: the runtime stages it before cudaMemcpyAsync returns)
    CK(cudaMemcpyAsync(dmsg, key, 48, cudaMemcpyHostToDevice, st));
    launch_hash_small(st, 1, dmsg, 48, dhm, dok);
    hm_store(key, dhm, dok, st);
    CK(cudaGetLastError());
    return 0;
}
int hbls_hash_cache_stats(uint64_t* hits, uint64_t* misses) {
    std::lock_guard<std::mutex> lk(g.mu);
    if (hits) *hits = g.hm_hits;
    if (misses) *misses = g.hm_misses;
    return 0;
}
int hbls_get_address(const blsPublicKey* pub, uint8_t out20[20]) {
    uint8_t ser[48], dg[32];
    if (blsPublicKeySerialize(ser, 48, pub) != 48) return HBLS_ERR_CUDA;
    Sha256::digest(ser, 48, dg); memcpy(out20, dg, 20); return 0;
}

}  // extern "C"

// ------------------------------------------------------------------ per-call operations, coalesced (coalesce.hpp).  Concurrent
// VerifyHash / SignHash / Deserialize / GetPublicKey calls queue up; one caller at a time takes g.mu, drains the queue and runs ONE
// batched device pass per operation kind over everything drained, with one stream synchronise.  A batch of one is the single call.
namespace {

struct HashMsg { const void* h; size_t size; };
// device bytes of launch_hm_batch over k items (every take of the arena is 256-byte aligned)
size_t hm_batch_bytes(size_t k) { return k * (sizeof(g2a) + 1 + 48 + 4) + 8 * 256; }
// H(m) of k items into hm / ok, each DISTINCT message once: the distinct messages (keyed by the 48 zero-padded bytes hash_to_fp reads,
// hm_key) are looked up in the H(m) cache, the misses are hashed in one launch and stored, then k_hm_gather copies every item's point
// from the distinct array.  Cache hit / miss counters count distinct messages.  Caller holds g.mu; runs on g.stream.
int launch_hm_batch(Arena& ar, size_t k, const HashMsg* msgs, g2a* hm, uint8_t* ok) {
    const bool cache = hm_enabled();
    std::vector<uint8_t> ukey(48 * k); std::vector<uint32_t> item_u(k);
    std::unordered_map<std::string, uint32_t> seen; seen.reserve(2 * k);
    size_t nu = 0;
    for (size_t i = 0; i < k; i++) {
        uint8_t key[48]; hm_key(key, msgs[i].h, msgs[i].size);
        auto ins = seen.emplace(std::string((const char*)key, 48), (uint32_t)nu);
        if (ins.second) memcpy(&ukey[48 * nu++], key, 48);
        item_u[i] = ins.first->second;
    }
    g2a* dhm = ar.take<g2a>(nu); uint8_t* dok = ar.take<uint8_t>(nu); uint8_t* dkeys = ar.take<uint8_t>(48 * nu); uint32_t* didx = ar.take<uint32_t>(k);
    // slots of the distinct array: misses from the front (one contiguous hash launch), cache hits from the back
    std::vector<uint32_t> slot(nu); std::vector<uint8_t> mkeys; mkeys.reserve(48 * nu);
    size_t lo = 0, hi = nu;
    for (size_t u = 0; u < nu; u++) {
        if (cache && hm_fetch(&ukey[48 * u], dhm + hi - 1, dok + hi - 1, g.stream)) slot[u] = (uint32_t)--hi;
        else { slot[u] = (uint32_t)lo++; mkeys.insert(mkeys.end(), &ukey[48 * u], &ukey[48 * u] + 48); }
    }
    if (lo) {
        CK(cudaMemcpyAsync(dkeys, mkeys.data(), 48 * lo, cudaMemcpyHostToDevice, g.stream));
        launch_hash_small(g.stream, lo, dkeys, 48, dhm, dok);
        if (cache)                                   // only the last HM_N would survive anyway
            for (size_t j = lo > (size_t)Ctx::HM_N ? lo - Ctx::HM_N : 0; j < lo; j++) hm_store(&mkeys[48 * j], dhm + j, dok + j, g.stream);
    }
    std::vector<uint32_t> idx(k);
    for (size_t i = 0; i < k; i++) idx[i] = slot[item_u[i]];
    CK(cudaMemcpyAsync(didx, idx.data(), 4 * k, cudaMemcpyHostToDevice, g.stream));
    LAUNCH(k_hm_gather, blocks_for(k, 128), 128, g.stream, k, (const uint32_t*)didx, (const g2a*)dhm, (const uint8_t*)dok, hm, ok);
    return 0;
}

size_t verify_pass_bytes(size_t k) { return verify_scratch_bytes(k) + k * (sizeof(g2) + 1) + 96 + hm_batch_bytes(k) + 16 * 256; }
// VerifyHash of k items, enqueued on g.stream; res[j] (pinned host) is valid once the stream has synchronised.  Keys: host structs
// (pubs) or one device Jacobian key (d_apk, k = 1: hbls_mask_verify); signatures: host structs (sigs) or one serialized signature
// (sig96, k = 1), decoded and subgroup-checked on the device.  Caller holds g.mu and reserved verify_pass_bytes(k).
int verify_hash_locked(Arena& ar, size_t k, const blsSignature* const* sigs, const uint8_t* sig96, const blsPublicKey* const* pubs,
                       const g1* d_apk, const HashMsg* msgs, uint8_t* res) {
    VerifyBufs v = carve_verify(ar, k);
    g2* dsig = ar.take<g2>(k); uint8_t* dsig96 = ar.take<uint8_t>(96); uint8_t* dres = ar.take<uint8_t>(k);
    if (d_apk) CK(cudaMemcpyAsync(v.apk, d_apk, sizeof(g1), cudaMemcpyDeviceToDevice, g.stream));
    else {
        std::vector<g1> hp(k);
        for (size_t j = 0; j < k; j++) memcpy(&hp[j], pubs[j], sizeof(g1));
        CK(cudaMemcpyAsync(v.apk, hp.data(), k * sizeof(g1), cudaMemcpyHostToDevice, g.stream));
    }
    LAUNCH(k_g1_normalize_lat, blocks_for(k, 32), 32, g.stream, k, v.apk, v.pkneg, 1);
    const uint8_t* ok_sig = nullptr;
    if (sig96) {          // serialized signature: decode (+ subgroup check) on the device
        CK(cudaMemcpyAsync(dsig96, sig96, 96, cudaMemcpyHostToDevice, g.stream));
        LAUNCH(k_g2_decode_pair, 1, 32, g.stream, (size_t)1, dsig96, v.sig, v.ok_sig, 1, (g2*)nullptr);
        ok_sig = v.ok_sig;
    } else {              // struct inputs are already-decoded Jacobian points: normalise instead of decoding
        std::vector<g2> hs(k);
        for (size_t j = 0; j < k; j++) memcpy(&hs[j], sigs[j], sizeof(g2));
        CK(cudaMemcpyAsync(dsig, hs.data(), k * sizeof(g2), cudaMemcpyHostToDevice, g.stream));
        LAUNCH(k_g2_normalize, blocks_for(k, 32), 32, g.stream, k, dsig, v.sig);
    }
    // H(m): cached when this node has hashed the message before (its own SignHash, a prefetch, an earlier check)
    if (int e = launch_hm_batch(ar, k, msgs, v.hm, v.ok_hm)) return e;
    if ((long long)k <= g.coop_max) {       // one warp per check
        const size_t coop_cap = (size_t)g.sm_count * (size_t)(g.coop_wpsm > 0 ? g.coop_wpsm : 1);
        LAUNCH(k_pairing_coop, (unsigned)(k < coop_cap ? k : coop_cap), 32, g.stream, k, v.sig, v.pkneg, v.hm, (const uint8_t*)v.ok_hm, ok_sig, (const uint8_t*)nullptr, dres);
    } else
        LAUNCH(k_pairing_verify_split, blocks_for(2 * k, 64), 64, g.stream, k, v.sig, v.pkneg, v.hm, (const uint8_t*)v.ok_hm, ok_sig, (const uint8_t*)nullptr, dres, (const int*)nullptr);
    LAUNCH(k_pairing_fixup, heavy_blocks(k), TPB, g.stream, k, v.sig, v.pkneg, v.hm, (const uint8_t*)v.ok_hm, ok_sig, (const uint8_t*)nullptr, dres, (const int*)nullptr);
    CK(cudaMemcpyAsync(res, dres, k, cudaMemcpyDeviceToHost, g.stream));
    return 0;
}

enum CoOp { CO_VERIFY, CO_SIGN, CO_SIG_DES, CO_PK_DES, CO_GET_PK, CO_NOPS };
// one queued per-call request: a = signature struct (verify) / secret key (sign, get-pk) / serialized bytes (deserialize),
// b = public key struct (verify), out = the caller's struct; rc = the call's result, written by the combiner
struct CoReq { int op; const void* a; const void* b; const void* msg; size_t len; void* out; int rc; };
hb::FlatCombiner<CoReq> g_co;

size_t sign_pass_bytes(size_t k) { return k * (32 + 32 + sizeof(g2) + 1 + sizeof(g2a) + 1) + 2 * hm_batch_bytes(k) + 16 * 256; }
// SignHash of k items (sigma = sk H(m)): into h_out / h_ok (pinned host) at position p for item perm[p].  Keys with base-|z| digits
// (every sk < r) take the ladder over psi; hand-filled structs >= Z^4 a second sub-batch through the plain 255-bit ladder.
int launch_sign_pass(Arena& ar, const std::vector<CoReq*>& rq, g2* h_out, uint8_t* h_ok, std::vector<uint32_t>& perm) {
    const size_t k = rq.size();
    std::vector<uint64_t> dig; std::vector<uint8_t> sk; std::vector<uint32_t> ib; std::vector<HashMsg> ma, mb;
    perm.clear();
    for (size_t j = 0; j < k; j++) {
        const blsSecretKey* sec = (const blsSecretKey*)rq[j]->a; uint64_t d[4];
        const HashMsg m{rq[j]->msg, rq[j]->len};
        if (sk_digits_base_z(sec->d, d)) { dig.insert(dig.end(), d, d + 4); perm.push_back((uint32_t)j); ma.push_back(m); }
        else { sk.insert(sk.end(), (const uint8_t*)sec->d, (const uint8_t*)sec->d + 32); ib.push_back((uint32_t)j); mb.push_back(m); }
    }
    const size_t na = ma.size(), nb = mb.size();
    perm.insert(perm.end(), ib.begin(), ib.end());
    g2* dout = ar.take<g2>(k); uint8_t* dok = ar.take<uint8_t>(k);
    g2a* hm = ar.take<g2a>(k); uint8_t* hok = ar.take<uint8_t>(k);
    if (na) {
        uint64_t* ddig = ar.take<uint64_t>(4 * na);
        CK(cudaMemcpyAsync(ddig, dig.data(), 32 * na, cudaMemcpyHostToDevice, g.stream));
        if (int e = launch_hm_batch(ar, na, ma.data(), hm, hok)) return e;
        LAUNCH(k_sign_hm_gls_pair, blocks_for(2 * na, 32), 32, g.stream, na, (const uint64_t*)ddig, (const g2a*)hm, (const uint8_t*)hok, (size_t)1, dout, dok);
    }
    if (nb) {
        uint8_t* dsk = ar.take<uint8_t>(32 * nb);
        CK(cudaMemcpyAsync(dsk, sk.data(), 32 * nb, cudaMemcpyHostToDevice, g.stream));
        if (int e = launch_hm_batch(ar, nb, mb.data(), hm + na, hok + na)) return e;
        LAUNCH(k_sign_hm_pair, blocks_for(2 * nb, 32), 32, g.stream, nb, (const uint8_t*)dsk, (const g2a*)(hm + na), (const uint8_t*)(hok + na), (size_t)1, dout + na, dok + na);
    }
    CK(cudaMemcpyAsync(h_out, dout, k * sizeof(g2), cudaMemcpyDeviceToHost, g.stream));
    CK(cudaMemcpyAsync(h_ok, dok, k, cudaMemcpyDeviceToHost, g.stream));
    return 0;
}

// one device pass per operation kind present, one synchronise, then every caller's output and return value.  g.mu is held.
int co_launch(const std::vector<CoReq*>* by) {
    const size_t kv = by[CO_VERIFY].size(), ks = by[CO_SIGN].size(), kd2 = by[CO_SIG_DES].size(), kd1 = by[CO_PK_DES].size(), kg = by[CO_GET_PK].size();
    size_t dev = 4096, host = 8 * 256;
    if (kv) { dev += verify_pass_bytes(kv); host += kv + 256; }
    if (ks) { dev += sign_pass_bytes(ks); host += ks * (sizeof(g2) + 1) + 512; }
    if (kd2) { dev += kd2 * (96 + sizeof(g2) + 1) + 4 * 256; host += kd2 * (sizeof(g2) + 1) + 512; }
    if (kd1) { dev += kd1 * (48 + sizeof(g1) + 1) + 4 * 256; host += kd1 * (sizeof(g1) + 1) + 512; }
    if (kg) { dev += kg * (32 + sizeof(g1)) + 4 * 256; host += kg * sizeof(g1) + 512; }
    Scratch* sc; if (int e = reserve(g.stream, dev, &sc)) return e;
    uint8_t* pin; if (int e = reserve_pinned(host, &pin)) return e;
    Arena ar{sc->base, 0, sc->cap}, hp{pin, 0, g.pin_cap};
    uint8_t* v_res = nullptr; g2* s_out = nullptr; uint8_t* s_ok = nullptr; std::vector<uint32_t> s_perm;
    g2* d2_out = nullptr; uint8_t* d2_ok = nullptr; g1* d1_out = nullptr; uint8_t* d1_ok = nullptr; g1* pk_out = nullptr;
    if (kv) {
        std::vector<const blsSignature*> sigs(kv); std::vector<const blsPublicKey*> pubs(kv); std::vector<HashMsg> msgs(kv);
        for (size_t j = 0; j < kv; j++) { const CoReq* r = by[CO_VERIFY][j]; sigs[j] = (const blsSignature*)r->a; pubs[j] = (const blsPublicKey*)r->b; msgs[j] = {r->msg, r->len}; }
        v_res = hp.take<uint8_t>(kv);
        if (int e = verify_hash_locked(ar, kv, sigs.data(), nullptr, pubs.data(), nullptr, msgs.data(), v_res)) return e;
    }
    if (ks) {
        s_out = hp.take<g2>(ks); s_ok = hp.take<uint8_t>(ks);
        if (int e = launch_sign_pass(ar, by[CO_SIGN], s_out, s_ok, s_perm)) return e;
    }
    if (kd2) {            // Sign.Deserialize: lane-pair decode + subgroup test, written in the blsSignature layout
        std::vector<uint8_t> in(96 * kd2);
        for (size_t j = 0; j < kd2; j++) memcpy(&in[96 * j], by[CO_SIG_DES][j]->a, 96);
        uint8_t* din = ar.take<uint8_t>(96 * kd2); g2* dout = ar.take<g2>(kd2); uint8_t* dok = ar.take<uint8_t>(kd2);
        d2_out = hp.take<g2>(kd2); d2_ok = hp.take<uint8_t>(kd2);
        CK(cudaMemcpyAsync(din, in.data(), 96 * kd2, cudaMemcpyHostToDevice, g.stream));
        LAUNCH(k_g2_decode_pair, blocks_for(2 * kd2, 32), 32, g.stream, kd2, (const uint8_t*)din, (g2a*)nullptr, dok, 1, dout);
        CK(cudaMemcpyAsync(d2_out, dout, kd2 * sizeof(g2), cudaMemcpyDeviceToHost, g.stream));
        CK(cudaMemcpyAsync(d2_ok, dok, kd2, cudaMemcpyDeviceToHost, g.stream));
    }
    if (kd1) {            // PublicKey.Deserialize: decode + subgroup test, Jacobian with z = 1 (the blsPublicKey layout)
        std::vector<uint8_t> in(48 * kd1);
        for (size_t j = 0; j < kd1; j++) memcpy(&in[48 * j], by[CO_PK_DES][j]->a, 48);
        uint8_t* din = ar.take<uint8_t>(48 * kd1); g1* dout = ar.take<g1>(kd1); uint8_t* dok = ar.take<uint8_t>(kd1);
        d1_out = hp.take<g1>(kd1); d1_ok = hp.take<uint8_t>(kd1);
        CK(cudaMemcpyAsync(din, in.data(), 48 * kd1, cudaMemcpyHostToDevice, g.stream));
        LAUNCH(k_g1_decode_jac, heavy_blocks(kd1), TPB, g.stream, kd1, (const uint8_t*)din, dout, dok, 1);
        CK(cudaMemcpyAsync(d1_out, dout, kd1 * sizeof(g1), cudaMemcpyDeviceToHost, g.stream));
        CK(cudaMemcpyAsync(d1_ok, dok, kd1, cudaMemcpyDeviceToHost, g.stream));
    }
    if (kg) {             // GetPublicKey: sk * generator
        std::vector<uint8_t> sk(32 * kg);
        for (size_t j = 0; j < kg; j++) memcpy(&sk[32 * j], ((const blsSecretKey*)by[CO_GET_PK][j]->a)->d, 32);
        uint8_t* dsk = ar.take<uint8_t>(32 * kg); g1* dout = ar.take<g1>(kg);
        pk_out = hp.take<g1>(kg);
        CK(cudaMemcpyAsync(dsk, sk.data(), 32 * kg, cudaMemcpyHostToDevice, g.stream));
        LAUNCH(k_g1_mul_gen, blocks_for(kg, 32), 32, g.stream, kg, (const uint8_t*)dsk, dout);
        CK(cudaMemcpyAsync(pk_out, dout, kg * sizeof(g1), cudaMemcpyDeviceToHost, g.stream));
    }
    CK(cudaStreamSynchronize(g.stream));
    for (size_t j = 0; j < kv; j++) by[CO_VERIFY][j]->rc = v_res[j] ? 1 : 0;
    for (size_t p = 0; p < ks; p++) {
        CoReq* r = by[CO_SIGN][s_perm[p]];
        memcpy(r->out, &s_out[p], sizeof(g2)); r->rc = s_ok[p] ? 0 : -1;
    }
    for (size_t j = 0; j < kd2; j++) {            // undecodable: the caller's struct stays as it was
        CoReq* r = by[CO_SIG_DES][j];
        if (d2_ok[j]) memcpy(r->out, &d2_out[j], sizeof(g2));
        r->rc = d2_ok[j] ? 96 : 0;
    }
    for (size_t j = 0; j < kd1; j++) {
        CoReq* r = by[CO_PK_DES][j];
        if (d1_ok[j]) memcpy(r->out, &d1_out[j], sizeof(g1));
        r->rc = d1_ok[j] ? 48 : 0;
    }
    for (size_t j = 0; j < kg; j++) { memcpy(by[CO_GET_PK][j]->out, &pk_out[j], sizeof(g1)); by[CO_GET_PK][j]->rc = 0; }
    return 0;
}
void co_run(CoReq* const* batch, size_t n) {
    std::vector<CoReq*> by[CO_NOPS];
    for (size_t i = 0; i < n; i++) by[batch[i]->op].push_back(batch[i]);
    int e;
    try { e = co_launch(by); } catch (const std::exception&) { e = HBLS_ERR_CUDA; }      // (bad_alloc) the owners must still be woken
    if (e) for (size_t i = 0; i < n; i++) batch[i]->rc = e;
}
int co_submit(int op, const void* a, const void* b, const void* msg, size_t len, void* out) {
    CoReq r{op, a, b, msg, len, out, 0};
    g_co.submit(r, g.mu, [] { return g.coop_max; }, co_run);
    return r.rc;
}

}  // namespace

extern "C" {

void blsGetPublicKey(blsPublicKey* pub, const blsSecretKey* sec) {
    memset(pub, 0, sizeof *pub);
    if (ensure_init()) return;
    co_submit(CO_GET_PK, sec, nullptr, nullptr, 0, pub);
}
int blsSignHash(blsSignature* sig, const blsSecretKey* sec, const void* h, size_t size) {
    if (int e = ensure_init()) return e;
    // H(m) kept in the H(m) cache: the validator verifies the aggregate over the very message it signs here
    return co_submit(CO_SIGN, sec, nullptr, h, size, sig);
}
int blsVerifyHash(const blsSignature* sig, const blsPublicKey* pub, const void* h, size_t size) {
    if (ensure_init()) return 0;
    return co_submit(CO_VERIFY, sig, pub, h, size, nullptr) == 1 ? 1 : 0;
}
size_t blsPublicKeyDeserialize(blsPublicKey* pub, const void* buf, size_t bufSize) {
    if (bufSize < 48 || ensure_init()) return 0;
    return co_submit(CO_PK_DES, buf, nullptr, nullptr, 0, pub) == 48 ? 48 : 0;
}
size_t blsSignatureDeserialize(blsSignature* sig, const void* buf, size_t bufSize) {
    if (bufSize < 96 || ensure_init()) return 0;
    return co_submit(CO_SIG_DES, buf, nullptr, nullptr, 0, sig) == 96 ? 96 : 0;
}
int hbls_coalesce_stats(uint64_t* requests, uint64_t* batches, uint64_t* largest_batch) {
    const hb::CoalesceStats s = g_co.stats();
    if (requests) *requests = s.requests;
    if (batches) *batches = s.batches;
    if (largest_batch) *largest_batch = s.largest_batch;
    return 0;
}
void blsSign(blsSignature* sig, const blsSecretKey* sec, const void* m, size_t size) {
    uint8_t dg[64]; Sha512::digest((const uint8_t*)m, size, dg);
    if (blsSignHash(sig, sec, dg, 64) != 0) memset(sig, 0, sizeof *sig);
}
int blsVerify(const blsSignature* sig, const blsPublicKey* pub, const void* m, size_t size) {
    uint8_t dg[64]; Sha512::digest((const uint8_t*)m, size, dg);
    return blsVerifyHash(sig, pub, dg, 64);
}

// ------------------------------------------------------------------ committee table
int hbls_committee_create(hbls_committee** out, const uint8_t* pk48, size_t n, size_t* bad_index) {
    if (int e = ensure_init()) return e;
    if (!out) return HBLS_ERR_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    std::unique_ptr<hbls_committee> c(new hbls_committee); c->n = n;       // freed (with its device tables) on every early return
    size_t nn = n ? n : 1;
    CK(cudaMalloc(&c->table, nn * sizeof(g1a)));
    Scratch* sc; if (int e = reserve(g.stream, nn * 49 + 4096, &sc)) return e;
    Arena ar{sc->base, 0, sc->cap};
    uint8_t* din = ar.take<uint8_t>(nn * 48); uint8_t* dok = ar.take<uint8_t>(nn);
    std::vector<uint8_t> ok(nn, 1);
    if (n) {
        CK(cudaMemcpyAsync(din, pk48, n * 48, cudaMemcpyHostToDevice, g.stream));
        LAUNCH(k_g1_decode, blocks_for(n, TPB), TPB, g.stream, n, din, c->table, dok, 1, 0);
        CK(cudaMalloc(&c->total, sizeof(g1)));
        LAUNCH(k_g1_sum, 1, 128, g.stream, n, c->table, c->total);
        CK(cudaMemcpyAsync(ok.data(), dok, n, cudaMemcpyDeviceToHost, g.stream));
        CK(cudaStreamSynchronize(g.stream));
    }
    for (size_t i = 0; i < n; i++) if (!ok[i]) { if (bad_index) *bad_index = i; return HBLS_ERR_DECODE; }
    *out = c.release(); return 0;
}
void hbls_committee_destroy(hbls_committee* c) { if (!c) return; std::lock_guard<std::mutex> lk(g.mu); cudaDeviceSynchronize(); delete c; }
size_t hbls_committee_size(const hbls_committee* c) { return c ? c->n : 0; }

int hbls_mask_aggregate(const hbls_committee* c, const uint8_t* bitmap, size_t blen, uint8_t out_pk48[48]) {
    if (int e = ensure_init()) return e;
    if (!c || blen != ((c->n + 7) >> 3)) return HBLS_ERR_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    Scratch* sc; if (int e = reserve(g.stream, blen + 4096, &sc)) return e;
    Arena ar{sc->base, 0, sc->cap};
    uint8_t* dbm = ar.take<uint8_t>(blen ? blen : 1); g1* dacc = ar.take<g1>(1); uint8_t* dout = ar.take<uint8_t>(48);
    if (blen) CK(cudaMemcpyAsync(dbm, bitmap, blen, cudaMemcpyHostToDevice, g.stream));
    LAUNCH(k_mask_aggregate, 1, 32, g.stream, (size_t)1, c->n, c->table, dbm, blen, dacc);
    LAUNCH(k_g1_serialize, 1, 32, g.stream, (size_t)1, dacc, dout);
    CK(cudaMemcpyAsync(out_pk48, dout, 48, cudaMemcpyDeviceToHost, g.stream));
    CK(cudaStreamSynchronize(g.stream));
    return 0;
}

int hbls_aggregate_sigs(const uint8_t* sig96, size_t n, uint8_t out96[96]) {
    if (int e = ensure_init()) return e;
    std::lock_guard<std::mutex> lk(g.mu);
    size_t nn = n ? n : 1;
    Scratch* sc; if (int e = reserve(g.stream, nn * (96 + sizeof(g2a) + 1) + 4096, &sc)) return e;
    Arena ar{sc->base, 0, sc->cap};
    uint8_t* din = ar.take<uint8_t>(nn * 96); g2a* dpts = ar.take<g2a>(nn); uint8_t* dok = ar.take<uint8_t>(nn);
    g2* dsum = ar.take<g2>(1); uint8_t* dout = ar.take<uint8_t>(96);
    std::vector<uint8_t> ok(nn, 1);
    if (n) {
        CK(cudaMemcpyAsync(din, sig96, n * 96, cudaMemcpyHostToDevice, g.stream));
        LAUNCH(k_g2_decode, heavy_blocks(n), TPB, g.stream, n, din, dpts, dok, 1);
    }
    LAUNCH(k_g2_sum, 1, HB_SUM_THREADS, g.stream, n, dpts, dsum);
    LAUNCH(k_g2_serialize, 1, 32, g.stream, (size_t)1, dsum, dout);
    if (n) CK(cudaMemcpyAsync(ok.data(), dok, n, cudaMemcpyDeviceToHost, g.stream));
    CK(cudaMemcpyAsync(out96, dout, 96, cudaMemcpyDeviceToHost, g.stream));
    CK(cudaStreamSynchronize(g.stream));
    for (size_t i = 0; i < n; i++) if (!ok[i]) return HBLS_ERR_DECODE;
    return 0;
}

// ------------------------------------------------------------------ aggregate verification
int hbls_aggregate_verify_batch_device(const hbls_committee* c, size_t B, const void* d_bitmaps, size_t blen, const void* d_sigs96,
                                       const void* d_msgs, size_t msg_len, void* d_results, void* stream) {
    if (int e = ensure_init()) return e;
    if (!c || blen != ((c->n + 7) >> 3)) return HBLS_ERR_ARG;
    if (B == 0) return 0;
    std::lock_guard<std::mutex> lk(g.mu);
    cudaStream_t s = stream ? (cudaStream_t)stream : g.stream;
    Scratch* sc; if (int e = reserve(s, verify_scratch_bytes(B), &sc)) return e;
    ensure_stage_events(sc);
    Arena ar{sc->base, 0, sc->cap};
    int rc = agg_verify_device_locked(c, B, (const uint8_t*)d_bitmaps, blen, (const uint8_t*)d_sigs96, (const uint8_t*)d_msgs, msg_len, (uint8_t*)d_results, s, sc, ar, false);
    CK(cudaGetLastError());
    return rc;
}
// host-buffer form shared by the batch entry and the header-range entry: flags_out (nullable) receives the decode flags per round
static int agg_verify_host_locked(const hbls_committee* c, size_t B, const uint8_t* bitmaps, size_t blen, const uint8_t* sigs96,
                                  const uint8_t* msgs, size_t msg_len, uint8_t* results, uint8_t* flags_out) {
    size_t in_bytes = B * (blen + 96 + msg_len);
    Scratch* sc; if (int e = reserve(g.stream, verify_scratch_bytes(B) + in_bytes + 2 * B + 4096, &sc)) return e;
    ensure_stage_events(sc);
    Arena ar{sc->base, 0, sc->cap};
    uint8_t* dbm = ar.take<uint8_t>(B * blen + 1); uint8_t* dsig = ar.take<uint8_t>(B * 96); uint8_t* dmsg = ar.take<uint8_t>(B * msg_len + 1);
    uint8_t* dres = ar.take<uint8_t>(B); uint8_t* dflags = ar.take<uint8_t>(B);
    if (blen) CK(cudaMemcpyAsync(dbm, bitmaps, B * blen, cudaMemcpyHostToDevice, g.stream));
    CK(cudaMemcpyAsync(dsig, sigs96, B * 96, cudaMemcpyHostToDevice, g.stream));
    if (msg_len) CK(cudaMemcpyAsync(dmsg, msgs, B * msg_len, cudaMemcpyHostToDevice, g.stream));
    VerifyBufs v;
    const bool same = all_messages_equal(msgs, B, msg_len);
    agg_verify_device_locked(c, B, dbm, blen, dsig, dmsg, msg_len, dres, g.stream, sc, ar, same, &v, (same || B == 1) ? msgs : nullptr);
    CK(cudaMemcpyAsync(results, dres, B, cudaMemcpyDeviceToHost, g.stream));
    if (flags_out) {
        LAUNCH(k_pack_flags, blocks_for(B, 256), 256, g.stream, B, v.ok_sig, v.ok_hm, (const uint8_t*)nullptr, dflags);
        CK(cudaMemcpyAsync(flags_out, dflags, B, cudaMemcpyDeviceToHost, g.stream));
    }
    CK(cudaStreamSynchronize(g.stream));
    return 0;
}
int hbls_aggregate_verify_batch(const hbls_committee* c, size_t B, const uint8_t* bitmaps, size_t blen, const uint8_t* sigs96,
                                const uint8_t* msgs, size_t msg_len, uint8_t* results) {
    if (int e = ensure_init()) return e;
    if (!c || blen != ((c->n + 7) >> 3)) return HBLS_ERR_ARG;
    if (B == 0) return 0;
    std::lock_guard<std::mutex> lk(g.mu);
    return agg_verify_host_locked(c, B, bitmaps, blen, sigs96, msgs, msg_len, results, nullptr);
}
int hbls_aggregate_verify(const hbls_committee* c, const uint8_t* bitmap, size_t blen, const uint8_t sig96[96], const void* msg, size_t msg_len) {
    uint8_t res = 0;
    int rc = hbls_aggregate_verify_batch(c, 1, bitmap, blen, sig96, (const uint8_t*)msg, msg_len, &res);
    if (rc) return rc;
    return res ? 1 : 0;
}
int hbls_verify_headers(const hbls_committee* c, size_t n, const uint8_t* sigs96, const uint8_t* bitmaps, size_t blen,
                        const uint8_t* payloads, size_t payload_len, size_t quorum, uint8_t* status) {
    if (int e = ensure_init()) return e;
    if (!c || blen != ((c->n + 7) >> 3) || !status) return HBLS_ERR_ARG;        // DecodeSigBitmap: mask.SetMask length error (sig.go:43)
    if (n == 0) return 0;
    std::lock_guard<std::mutex> lk(g.mu);
    std::vector<uint8_t> res(n), flags(n);
    if (int e = agg_verify_host_locked(c, n, bitmaps, blen, sigs96, payloads, payload_len, res.data(), flags.data())) return e;
    for (size_t i = 0; i < n; i++) {
        // engine.go:630-640: DecodeSigBitmap (signature deserialise) -> IsQuorumAchievedByMask -> VerifyHash
        if (!(flags[i] & 1)) status[i] = HBLS_HDR_BAD_ENCODING;
        else if (quorum && (size_t)popcount_slots(bitmaps + i * blen, c->n) < quorum) status[i] = HBLS_HDR_NO_QUORUM;
        else status[i] = res[i] ? HBLS_HDR_OK : HBLS_HDR_BAD_SIG;
    }
    return 0;
}

int hbls_aggregate_verify_items(size_t k, const hbls_committee* const* committees, const uint8_t* bitmaps, const uint8_t* sigs96,
                                const uint8_t* msgs, size_t msg_len, uint8_t* results) {
    if (int e = ensure_init()) return e;
    if (k == 0) return 0;
    if (!committees || !results) return HBLS_ERR_ARG;
    size_t bm_bytes = 0;
    for (size_t j = 0; j < k; j++) { if (!committees[j]) return HBLS_ERR_ARG; bm_bytes += (committees[j]->n + 7) >> 3; }
    std::lock_guard<std::mutex> lk(g.mu);
    Scratch* sc; if (int e = reserve(g.stream, verify_scratch_bytes(k) + bm_bytes + k * (96 + msg_len + 1 + sizeof(mask_item)) + 4096, &sc)) return e;
    ensure_stage_events(sc);
    Arena ar{sc->base, 0, sc->cap};
    VerifyBufs v = carve_verify(ar, k);
    uint8_t* dbm = ar.take<uint8_t>(bm_bytes + 1); uint8_t* dsig = ar.take<uint8_t>(k * 96); uint8_t* dmsg = ar.take<uint8_t>(k * msg_len + 1);
    uint8_t* dres = ar.take<uint8_t>(k); mask_item* ditems = ar.take<mask_item>(k);
    std::vector<mask_item> items(k); size_t off = 0;
    for (size_t j = 0; j < k; j++) { items[j].table = committees[j]->table; items[j].bitmap = dbm + off; items[j].n = committees[j]->n; off += (committees[j]->n + 7) >> 3; }
    if (bm_bytes) CK(cudaMemcpyAsync(dbm, bitmaps, bm_bytes, cudaMemcpyHostToDevice, g.stream));
    CK(cudaMemcpyAsync(dsig, sigs96, k * 96, cudaMemcpyHostToDevice, g.stream));
    if (msg_len) CK(cudaMemcpyAsync(dmsg, msgs, k * msg_len, cudaMemcpyHostToDevice, g.stream));
    CK(cudaMemcpyAsync(ditems, items.data(), k * sizeof(mask_item), cudaMemcpyHostToDevice, g.stream));
    fork_point(k, sc, g.stream);
    STAGE_EV(0, sc, g.stream);
    LAUNCH(k_mask_aggregate_items, blocks_for(k * 32, 128), 128, g.stream, k, ditems, v.apk);
    launch_verify_tail(k, v, sc, dsig, dmsg, (uint32_t)msg_len, nullptr, dres, g.stream, all_messages_equal(msgs, k, msg_len));
    CK(cudaMemcpyAsync(results, dres, k, cudaMemcpyDeviceToHost, g.stream));
    CK(cudaStreamSynchronize(g.stream));          // items[] (pageable source of an async copy) stays alive until here
    return 0;
}

// shared body of hbls_verify_batch / hbls_verify_batch_status; flags_out (nullable): k_pack_flags bytes per item
static int verify_batch_locked(size_t k, const uint8_t* pk48, const uint8_t* sig96, const uint8_t* msgs, size_t msg_len, uint8_t* results, uint8_t* flags_out) {
    Scratch* sc; if (int e = reserve(g.stream, verify_scratch_bytes(k) + k * (48 + 96 + msg_len + 2) + 4096, &sc)) return e;
    ensure_stage_events(sc);
    Arena ar{sc->base, 0, sc->cap};
    VerifyBufs v = carve_verify(ar, k);
    uint8_t* dpk = ar.take<uint8_t>(k * 48); uint8_t* dsig = ar.take<uint8_t>(k * 96); uint8_t* dmsg = ar.take<uint8_t>(k * msg_len + 1);
    uint8_t* dres = ar.take<uint8_t>(k); uint8_t* dflags = ar.take<uint8_t>(k);
    CK(cudaMemcpyAsync(dpk, pk48, k * 48, cudaMemcpyHostToDevice, g.stream));
    CK(cudaMemcpyAsync(dsig, sig96, k * 96, cudaMemcpyHostToDevice, g.stream));
    if (msg_len) CK(cudaMemcpyAsync(dmsg, msgs, k * msg_len, cudaMemcpyHostToDevice, g.stream));
    fork_point(k, sc, g.stream);
    STAGE_EV(0, sc, g.stream);
    // keys stay Jacobian (z = 1): the same tail as a mask aggregate, so independent triples also go through the batched groups
    LAUNCH(k_g1_decode_jac, heavy_blocks(k), TPB, g.stream, k, dpk, v.apk, v.ok_pk, 1);
    launch_verify_tail(k, v, sc, dsig, dmsg, (uint32_t)msg_len, v.ok_pk, dres, g.stream, all_messages_equal(msgs, k, msg_len));
    CK(cudaMemcpyAsync(results, dres, k, cudaMemcpyDeviceToHost, g.stream));
    if (flags_out) {
        LAUNCH(k_pack_flags, blocks_for(k, 256), 256, g.stream, k, v.ok_sig, v.ok_hm, (const uint8_t*)v.ok_pk, dflags);
        CK(cudaMemcpyAsync(flags_out, dflags, k, cudaMemcpyDeviceToHost, g.stream));
    }
    CK(cudaStreamSynchronize(g.stream));
    return 0;
}
int hbls_verify_batch(size_t k, const uint8_t* pk48, const uint8_t* sig96, const uint8_t* msgs, size_t msg_len, uint8_t* results) {
    if (int e = ensure_init()) return e;
    if (k == 0) return 0;
    std::lock_guard<std::mutex> lk(g.mu);
    return verify_batch_locked(k, pk48, sig96, msgs, msg_len, results, nullptr);
}
// same check, but the caller learns WHY an item failed, in the order the reference meets the errors: the sender key is decoded
// first (BytesToBLSPublicKey, consensus/view_change_msg.go:159), then the signature (Sign.Deserialize, :168-179), then VerifyHash
int hbls_verify_batch_status(size_t k, const uint8_t* pk48, const uint8_t* sig96, const uint8_t* msgs, size_t msg_len, uint8_t* status) {
    if (int e = ensure_init()) return e;
    if (k == 0) return 0;
    if (!status) return HBLS_ERR_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    std::vector<uint8_t> flags(k);
    if (int e = verify_batch_locked(k, pk48, sig96, msgs, msg_len, status, flags.data())) return e;
    for (size_t j = 0; j < k; j++) {
        if (!(flags[j] & 4)) status[j] = HBLS_VB_BAD_KEY_ENCODING;
        else if (!(flags[j] & 1)) status[j] = HBLS_VB_BAD_SIG_ENCODING;
        else status[j] = status[j] == 1 ? HBLS_VB_OK : HBLS_VB_BAD_SIG;
    }
    return 0;
}

// ------------------------------------------------------------------ persistent Mask / running vote aggregate (SURVEY 8f.2)
int hbls_mask_create(hbls_mask** out, const hbls_committee* c) {
    if (int e = ensure_init()) return e;
    if (!out || !c) return HBLS_ERR_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    std::unique_ptr<hbls_mask> m(new hbls_mask); m->c = c; m->bitmap.assign((c->n + 7) >> 3, 0);
    CK(cudaMalloc(&m->d_acc, sizeof(g1)));
    CK(cudaMemsetAsync(m->d_acc, 0, sizeof(g1), g.stream));          // all-zero struct = identity (mask.go:88)
    CK(cudaStreamSynchronize(g.stream));
    *out = m.release(); return 0;
}
void hbls_mask_destroy(hbls_mask* m) { if (!m) return; std::lock_guard<std::mutex> lk(g.mu); cudaDeviceSynchronize(); delete m; }
int hbls_mask_clear(hbls_mask* m) {
    if (int e = ensure_init()) return e;
    if (!m) return HBLS_ERR_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    std::fill(m->bitmap.begin(), m->bitmap.end(), 0);
    CK(cudaMemsetAsync(m->d_acc, 0, sizeof(g1), g.stream));
    CK(cudaStreamSynchronize(g.stream));
    return 0;
}
// SetMask body (caller holds g.mu): apply the delta between m's bitmap and `bitmap` to the running aggregate key
static int set_mask_locked(hbls_mask* m, const uint8_t* bitmap, size_t blen) {
    const size_t n = m->c->n;
    std::vector<uint8_t> delta(2 * blen + 2, 0);                       // row 0: bits to Add (0 -> 1), row 1: bits to Sub (1 -> 0)
    bool any = false;
    for (size_t i = 0; i < n; i++) {                                   // only slots i < n exist (mask.go:121: for i := range m.Publics)
        const uint8_t msk = (uint8_t)(1u << (i & 7)); const bool was = m->bitmap[i >> 3] & msk, now = bitmap[i >> 3] & msk;
        if (!was && now) { delta[i >> 3] |= msk; any = true; }
        if (was && !now) { delta[blen + (i >> 3)] |= msk; any = true; }
    }
    if (!any) return 0;
    Scratch* sc; if (int e = reserve(g.stream, 2 * blen + 4096, &sc)) return e;
    Arena ar{sc->base, 0, sc->cap};
    uint8_t* dbm = ar.take<uint8_t>(2 * blen + 2); g1* dtmp = ar.take<g1>(2); int* drc = ar.take<int>(1);
    CK(cudaMemcpyAsync(dbm, delta.data(), 2 * blen, cudaMemcpyHostToDevice, g.stream));
    LAUNCH(k_mask_aggregate, 1, 64, g.stream, (size_t)2, n, m->c->table, dbm, blen, dtmp);
    LAUNCH(k_single, 1, 32, g.stream, (int)OP_G1_ADD, (const void*)m->d_acc, (const void*)(dtmp + 0), (void*)m->d_acc, drc, 0u);
    LAUNCH(k_single, 1, 32, g.stream, (int)OP_G1_SUB, (const void*)m->d_acc, (const void*)(dtmp + 1), (void*)m->d_acc, drc, 0u);
    CK(cudaStreamSynchronize(g.stream));
    for (size_t i = 0; i < n; i++) {
        const uint8_t msk = (uint8_t)(1u << (i & 7));
        m->bitmap[i >> 3] = (uint8_t)((m->bitmap[i >> 3] & ~msk) | (bitmap[i >> 3] & msk));
    }
    return 0;
}
int hbls_mask_set_mask(hbls_mask* m, const uint8_t* bitmap, size_t blen) {
    if (int e = ensure_init()) return e;
    if (!m || blen != m->bitmap.size()) return HBLS_ERR_ARG;          // mask.go:114-120 "mismatching bitmap lengths"
    std::lock_guard<std::mutex> lk(g.mu);
    return set_mask_locked(m, bitmap, blen);
}
int hbls_mask_set_bit(hbls_mask* m, size_t index, int enable) {
    if (int e = ensure_init()) return e;
    if (!m || index >= m->c->n) return HBLS_ERR_ARG;                   // mask.go:138-140 "index out of range"
    // read-modify-write of the bitmap under ONE hold of g.mu: concurrent SetBit calls on different bits all land
    std::lock_guard<std::mutex> lk(g.mu);
    std::vector<uint8_t> bm = m->bitmap;
    const uint8_t msk = (uint8_t)(1u << (index & 7));
    if (enable) bm[index >> 3] |= msk; else bm[index >> 3] &= (uint8_t)~msk;
    return set_mask_locked(m, bm.data(), bm.size());
}
int hbls_mask_count_enabled(const hbls_mask* m) {
    if (!m) return HBLS_ERR_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    return popcount_slots(m->bitmap.data(), m->c->n);
}
int hbls_mask_get(const hbls_mask* m, uint8_t* bitmap_out, size_t blen, uint8_t pk48_out[48]) {
    if (int e = ensure_init()) return e;
    if (!m || (bitmap_out && blen != m->bitmap.size())) return HBLS_ERR_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    if (bitmap_out) memcpy(bitmap_out, m->bitmap.data(), blen);
    if (pk48_out) {
        Scratch* sc; if (int e = reserve(g.stream, 4096, &sc)) return e;
        Arena ar{sc->base, 0, sc->cap};
        uint8_t* dout = ar.take<uint8_t>(48);
        LAUNCH(k_g1_serialize, 1, 32, g.stream, (size_t)1, (const g1*)m->d_acc, dout);
        CK(cudaMemcpyAsync(pk48_out, dout, 48, cudaMemcpyDeviceToHost, g.stream));
        CK(cudaStreamSynchronize(g.stream));
    }
    return 0;
}
int hbls_mask_verify(const hbls_mask* m, const uint8_t sig96[96], const void* msg, size_t msg_len) {
    if (int e = ensure_init()) return e;
    if (!m || !sig96) return HBLS_ERR_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    Scratch* sc; if (int e = reserve(g.stream, verify_pass_bytes(1), &sc)) return e;
    uint8_t* res; if (int e = reserve_pinned(1, &res)) return e;
    Arena ar{sc->base, 0, sc->cap};
    const HashMsg hm{msg, msg_len};
    if (int e = verify_hash_locked(ar, 1, nullptr, sig96, nullptr, m->d_acc, &hm, res)) return e;
    CK(cudaStreamSynchronize(g.stream));
    return res[0] ? 1 : 0;
}
int hbls_ballot_box_create(hbls_ballot_box** out, const hbls_committee* c) {
    if (int e = ensure_init()) return e;
    if (!out || !c) return HBLS_ERR_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    std::unique_ptr<hbls_ballot_box> b(new hbls_ballot_box); b->c = c; b->collected.assign((c->n + 7) >> 3, 0);
    CK(cudaMalloc(&b->d_sum, sizeof(g2)));
    CK(cudaMemsetAsync(b->d_sum, 0, sizeof(g2), g.stream));
    CK(cudaStreamSynchronize(g.stream));
    *out = b.release(); return 0;
}
void hbls_ballot_box_destroy(hbls_ballot_box* b) { if (!b) return; std::lock_guard<std::mutex> lk(g.mu); cudaDeviceSynchronize(); delete b; }
int hbls_ballot_box_add_vote(hbls_ballot_box* b, const uint8_t* signer_bitmap, size_t blen, const uint8_t sig96[96]) {
    if (int e = ensure_init()) return e;
    if (!b || !signer_bitmap || blen != b->collected.size()) return HBLS_ERR_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    const size_t n = b->c->n;
    for (size_t i = 0; i < n; i++)                                      // quorum.go:168-181: skip a ballot that shares a signer with a collected one
        if ((signer_bitmap[i >> 3] >> (i & 7)) & 1 && (b->collected[i >> 3] >> (i & 7)) & 1) return 1;
    Scratch* sc; if (int e = reserve(g.stream, 4096, &sc)) return e;
    Arena ar{sc->base, 0, sc->cap};
    uint8_t* dsig = ar.take<uint8_t>(96); int* drc = ar.take<int>(1);
    CK(cudaMemcpyAsync(dsig, sig96, 96, cudaMemcpyHostToDevice, g.stream));
    LAUNCH(k_single, 1, 32, g.stream, (int)OP_G2_DES_ADD, (const void*)dsig, (const void*)nullptr, (void*)b->d_sum, drc, 0u);
    int rc = 0;
    CK(cudaMemcpyAsync(&rc, drc, sizeof(int), cudaMemcpyDeviceToHost, g.stream));
    CK(cudaStreamSynchronize(g.stream));
    if (rc != 96) return HBLS_ERR_DECODE;
    for (size_t i = 0; i < n; i++) if ((signer_bitmap[i >> 3] >> (i & 7)) & 1) b->collected[i >> 3] |= (uint8_t)(1u << (i & 7));
    return 0;
}
int hbls_ballot_box_aggregate(const hbls_ballot_box* b, uint8_t out_sig96[96], uint8_t* bitmap_out, size_t blen) {
    if (int e = ensure_init()) return e;
    if (!b || !out_sig96 || (bitmap_out && blen != b->collected.size())) return HBLS_ERR_ARG;
    std::lock_guard<std::mutex> lk(g.mu);
    Scratch* sc; if (int e = reserve(g.stream, 4096, &sc)) return e;
    Arena ar{sc->base, 0, sc->cap};
    uint8_t* dout = ar.take<uint8_t>(96);
    LAUNCH(k_g2_serialize, 1, 32, g.stream, (size_t)1, (const g2*)b->d_sum, dout);
    CK(cudaMemcpyAsync(out_sig96, dout, 96, cudaMemcpyDeviceToHost, g.stream));
    CK(cudaStreamSynchronize(g.stream));
    if (bitmap_out) memcpy(bitmap_out, b->collected.data(), blen);
    return 0;
}

// ------------------------------------------------------------------ ONE batch split over several GPUs (SURVEY 8e, BASELINE configs[3])
struct PartialRecord { g2 S; fp2 f[6]; uint32_t n_items; uint32_t n_bad; };
// the wire record is the first HBLS_PARTIAL_BYTES of the struct (field elements are 16-byte aligned: the struct may end in padding)
static_assert(offsetof(PartialRecord, n_bad) + sizeof(uint32_t) == HBLS_PARTIAL_BYTES && sizeof(PartialRecord) >= HBLS_PARTIAL_BYTES, "partial record layout");
int hbls_rlc_partial(size_t k, const uint8_t* pk48, const uint8_t* sig96, const uint8_t* msgs, size_t msg_len, uint8_t record[HBLS_PARTIAL_BYTES]) {
    if (int e = ensure_init()) return e;
    if (!record) return HBLS_ERR_ARG;
    PartialRecord rec; memset(&rec, 0, sizeof rec);
    std::lock_guard<std::mutex> lk(g.mu);
    const size_t kk = k ? k : 1;
    const unsigned W = (unsigned)(kk < (size_t)g.sm_count * 2 ? kk : (size_t)g.sm_count * 2);      // warps that multiply Miller values into partial products
    Scratch* sc; if (int e = reserve(g.stream, verify_scratch_bytes(kk) + kk * (48 + 96 + msg_len + 8) + (W + 2) * 6 * sizeof(fp2) + sizeof(g2) + 8192, &sc)) return e;
    Arena ar{sc->base, 0, sc->cap};
    VerifyBufs v = carve_verify(ar, kk);
    uint8_t* dpk = ar.take<uint8_t>(kk * 48); uint8_t* dsig = ar.take<uint8_t>(kk * 96); uint8_t* dmsg = ar.take<uint8_t>(kk * msg_len + 1);
    uint64_t* dco = ar.take<uint64_t>(kk); fp2* dpart = ar.take<fp2>((size_t)W * 6); fp2* dprod = ar.take<fp2>(6); g2* dS = ar.take<g2>(1);
    if (k) {
        const std::vector<uint64_t> co = rlc_draw_items(k);
        CK(cudaMemcpyAsync(dpk, pk48, k * 48, cudaMemcpyHostToDevice, g.stream));
        CK(cudaMemcpyAsync(dsig, sig96, k * 96, cudaMemcpyHostToDevice, g.stream));
        if (msg_len) CK(cudaMemcpyAsync(dmsg, msgs, k * msg_len, cudaMemcpyHostToDevice, g.stream));
        CK(cudaMemcpyAsync(dco, co.data(), k * 8, cudaMemcpyHostToDevice, g.stream));
        CK(cudaStreamSynchronize(g.stream));                    // co is a local: the copy must have read it before it goes out of scope
    }
    CK(cudaMemsetAsync(v.counts, 0, 2 * sizeof(unsigned), g.stream));
    LAUNCH(k_g1_decode_jac, heavy_blocks(kk), TPB, g.stream, k, dpk, v.apk, v.ok_pk, 1);
    const bool pairs = (long long)k <= g.coop_max;
    if (pairs) { LAUNCH(k_g2_decode_pair, blocks_for(2 * kk, 32), 32, g.stream, k, dsig, v.sig, v.ok_sig, 1); launch_hash_small(g.stream, k, dmsg, (uint32_t)msg_len, v.hm, v.ok_hm); }
    else { LAUNCH(k_g2_decode, heavy_blocks(kk), TPB, g.stream, k, dsig, v.sig, v.ok_sig, 1); LAUNCH(k_hash_to_g2, heavy_blocks(kk), TPB, g.stream, k, dmsg, (uint32_t)msg_len, v.hm, v.ok_hm); }
    rlc_coeffs none{};
    LAUNCH(k_rlc_scale, heavy_blocks(kk), TPB, g.stream, k, (size_t)1, v.apk, v.sig, v.hm, v.ok_sig, v.ok_hm, (const uint8_t*)v.ok_pk, none, (const uint64_t*)dco, v.pk_scaled, v.S, v.bad);
    LAUNCH(k_rlc_partial_coop, W, 32, g.stream, k, v.pk_scaled, v.hm, v.bad, dpart, v.counts);
    LAUNCH(k_rlc_reduce_coop, 1, 32, g.stream, (size_t)W, dpart, dprod);
    LAUNCH(k_g2_sum_jac, 1, HB_SUM_THREADS, g.stream, k, v.S, dS);
    unsigned counts[2] = {0, 0};
    CK(cudaMemcpyAsync(&rec.S, dS, sizeof(g2), cudaMemcpyDeviceToHost, g.stream));
    CK(cudaMemcpyAsync(rec.f, dprod, 6 * sizeof(fp2), cudaMemcpyDeviceToHost, g.stream));
    CK(cudaMemcpyAsync(counts, v.counts, sizeof counts, cudaMemcpyDeviceToHost, g.stream));
    CK(cudaStreamSynchronize(g.stream));
    rec.n_items = (uint32_t)k; rec.n_bad = counts[0];
    memcpy(record, &rec, HBLS_PARTIAL_BYTES);
    return 0;
}
int hbls_rlc_fold(size_t n, const uint8_t* records) {
    if (int e = ensure_init()) return e;
    if (!records) return HBLS_ERR_ARG;
    size_t items = 0, bad = 0;
    for (size_t p = 0; p < n; p++) { PartialRecord r; memcpy(&r, records + p * HBLS_PARTIAL_BYTES, HBLS_PARTIAL_BYTES); items += r.n_items; bad += r.n_bad; }
    if (bad || items == 0) return 0;                                  // an undecodable / identity item somewhere, or nothing to prove: callers verify exactly
    std::lock_guard<std::mutex> lk(g.mu);
    Scratch* sc; if (int e = reserve(g.stream, n * (sizeof(g2) + 6 * sizeof(fp2)) + sizeof(g2) + sizeof(g2a) + 4096, &sc)) return e;
    Arena ar{sc->base, 0, sc->cap};
    g2* dS = ar.take<g2>(n); fp2* dparts = ar.take<fp2>(n * 6); g2* dsum = ar.take<g2>(1); g2a* dsg = ar.take<g2a>(1); uint8_t* dres = ar.take<uint8_t>(1);
    std::vector<g2> hs(n); std::vector<fp2> hf(n * 6);
    for (size_t p = 0; p < n; p++) { PartialRecord r; memcpy(&r, records + p * HBLS_PARTIAL_BYTES, HBLS_PARTIAL_BYTES); hs[p] = r.S; for (int i = 0; i < 6; i++) hf[6 * p + i] = r.f[i]; }
    CK(cudaMemcpyAsync(dS, hs.data(), n * sizeof(g2), cudaMemcpyHostToDevice, g.stream));
    CK(cudaMemcpyAsync(dparts, hf.data(), n * 6 * sizeof(fp2), cudaMemcpyHostToDevice, g.stream));
    LAUNCH(k_g2_sum_jac, 1, HB_SUM_THREADS, g.stream, n, dS, dsum);
    LAUNCH(k_g2_normalize, 1, 32, g.stream, (size_t)1, dsum, dsg);
    LAUNCH(k_rlc_fold_coop, 1, 32, g.stream, n, dparts, dsg, dres);
    uint8_t res = 0;
    CK(cudaMemcpyAsync(&res, dres, 1, cudaMemcpyDeviceToHost, g.stream));
    CK(cudaStreamSynchronize(g.stream));                              // hs / hf stay alive until the copies are done
    return res ? 1 : 0;
}

int hbls_sign_hash_batch(size_t k, const uint8_t* sk32, const uint8_t* msgs, size_t msg_len, uint8_t* sig96_out, uint8_t* ok) {
    if (int e = ensure_init()) return e;
    if (k == 0) return 0;
    std::lock_guard<std::mutex> lk(g.mu);
    Scratch* sc; if (int e = reserve(g.stream, k * (32 + msg_len + sizeof(g2) + 96 + 1) + 4096, &sc)) return e;
    Arena ar{sc->base, 0, sc->cap};
    uint8_t* dsk = ar.take<uint8_t>(k * 32); uint8_t* dmsg = ar.take<uint8_t>(k * msg_len + 1); g2* dpts = ar.take<g2>(k);
    uint8_t* dout = ar.take<uint8_t>(k * 96); uint8_t* dok = ar.take<uint8_t>(k);
    CK(cudaMemcpyAsync(dsk, sk32, k * 32, cudaMemcpyHostToDevice, g.stream));
    if (msg_len) CK(cudaMemcpyAsync(dmsg, msgs, k * msg_len, cudaMemcpyHostToDevice, g.stream));
    LAUNCH(k_sign_hash, blocks_for(k, TPB), TPB, g.stream, k, dsk, dmsg, (uint32_t)msg_len, dpts, dok);
    LAUNCH(k_g2_serialize, blocks_for(k, TPB), TPB, g.stream, k, dpts, dout);
    CK(cudaMemcpyAsync(sig96_out, dout, k * 96, cudaMemcpyDeviceToHost, g.stream));
    CK(cudaMemcpyAsync(ok, dok, k, cudaMemcpyDeviceToHost, g.stream));
    CK(cudaStreamSynchronize(g.stream));
    return 0;
}
int hbls_get_public_key_batch(size_t k, const uint8_t* sk32, uint8_t* pk48_out) {
    if (int e = ensure_init()) return e;
    if (k == 0) return 0;
    std::lock_guard<std::mutex> lk(g.mu);
    Scratch* sc; if (int e = reserve(g.stream, k * (32 + sizeof(g1) + 48) + 4096, &sc)) return e;
    Arena ar{sc->base, 0, sc->cap};
    uint8_t* dsk = ar.take<uint8_t>(k * 32); g1* dpts = ar.take<g1>(k); uint8_t* dout = ar.take<uint8_t>(k * 48);
    CK(cudaMemcpyAsync(dsk, sk32, k * 32, cudaMemcpyHostToDevice, g.stream));
    LAUNCH(k_g1_mul_gen, blocks_for(k, TPB), TPB, g.stream, k, dsk, dpts);
    LAUNCH(k_g1_serialize, blocks_for(k, TPB), TPB, g.stream, k, dpts, dout);
    CK(cudaMemcpyAsync(pk48_out, dout, k * 48, cudaMemcpyDeviceToHost, g.stream));
    CK(cudaStreamSynchronize(g.stream));
    return 0;
}

int hbls_fp_mul_batch(size_t n, const uint8_t* a48, const uint8_t* b48, uint8_t* out48) {
    if (int e = ensure_init()) return e;
    if (n == 0) return 0;
    std::lock_guard<std::mutex> lk(g.mu);
    Scratch* sc; if (int e = reserve(g.stream, n * 144 + 4096, &sc)) return e;
    Arena ar{sc->base, 0, sc->cap};
    uint8_t* da = ar.take<uint8_t>(n * 48); uint8_t* db = ar.take<uint8_t>(n * 48); uint8_t* dout = ar.take<uint8_t>(n * 48);
    CK(cudaMemcpyAsync(da, a48, n * 48, cudaMemcpyHostToDevice, g.stream));
    CK(cudaMemcpyAsync(db, b48, n * 48, cudaMemcpyHostToDevice, g.stream));
    LAUNCH(k_fp_mul, blocks_for(n, 128), 128, g.stream, n, da, db, dout);
    CK(cudaMemcpyAsync(out48, dout, n * 48, cudaMemcpyDeviceToHost, g.stream));
    CK(cudaStreamSynchronize(g.stream));
    return 0;
}

void hbls_stage_timing_enable(int on) {
    std::lock_guard<std::mutex> lk(g.mu);
    g.stage_timing = on != 0; g.stage_sc = nullptr;
}
int hbls_stage_timing_get(float* ms_out, int max_stages) {
    std::lock_guard<std::mutex> lk(g.mu);
    Scratch* sc = g.stage_sc;
    if (!sc || !sc->ev_ok) return 0;
    if (cudaEventSynchronize(sc->ev[6]) != cudaSuccess) return 0;
    int n = max_stages < 6 ? max_stages : 6;
    for (int i = 0; i < n; i++) { float ms = 0; cudaEventElapsedTime(&ms, sc->ev[i], sc->ev[i + 1]); ms_out[i] = ms; }
    // 7th value: the line kernel's part of stage 5 when the batched pairing ran as two kernels (first chunk), else 0
    if (max_stages >= 7) { float ms = 0; if (sc->ev7_set) cudaEventElapsedTime(&ms, sc->ev[5], sc->ev[7]); ms_out[6] = ms; n = 7; }
    return n;
}
int hbls_selftest_split(uint32_t iters) {
    if (int e = ensure_init()) return e;
    std::lock_guard<std::mutex> lk(g.mu);
    Scratch* sc; if (int e = reserve(g.stream, 4096, &sc)) return e;
    uint32_t* d = reinterpret_cast<uint32_t*>(sc->base);
    CK(cudaMemsetAsync(d, 0, 4, g.stream));
    LAUNCH(k_selftest_fp2h, 8, 64, g.stream, iters, 20240922u, d);
    uint32_t bad = 0;
    CK(cudaMemcpyAsync(&bad, d, 4, cudaMemcpyDeviceToHost, g.stream));
    CK(cudaStreamSynchronize(g.stream));
    return (int)bad;
}
double hbls_probe_mac32_per_s(int iters, double* sm_clock_hz) {
    if (ensure_init()) return -1.0;
    std::lock_guard<std::mutex> lk(g.mu);
    Scratch* sc; if (reserve(g.stream, 4096, &sc)) return -1.0;
    uint32_t* sink = reinterpret_cast<uint32_t*>(sc->base);
    unsigned long long* cyc = reinterpret_cast<unsigned long long*>(sc->base + 256);
    constexpr int K = 4;
    const int threads = 256, blocks = g.sm_count * 2;                  // one wave: 2 x 256 threads x 94 registers per SM
    cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
    LAUNCH(k_probe_carry<K>, blocks, threads, g.stream, iters / 8 + 1, 12345u, sink, cyc);     // warm-up
    cudaEventRecord(e0, g.stream);
    LAUNCH(k_probe_carry<K>, blocks, threads, g.stream, iters, 12345u, sink, cyc);
    cudaEventRecord(e1, g.stream);
    if (cudaStreamSynchronize(g.stream) != cudaSuccess) return -1.0;
    float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (sm_clock_hz) { int khz = 0; cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, g.device); *sm_clock_hz = khz * 1e3; }   // maximum SM clock
    double macs = (double)blocks * threads * (double)iters * K * 6.0;  // lane_mad = 6 IMAD.WIDE
    return macs / (ms * 1e-3);
}

}  // extern "C"
