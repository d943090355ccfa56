// harmony_b200/host/hbls_concurrency_test.cpp -- concurrent per-call use of the C ABI, the way cgo calls it: many OS threads
// (goroutines pinned for the duration of a cgo call) calling blsGetPublicKey / blsSignHash / blsVerifyHash / blsSignatureDeserialize /
// blsPublicKeyDeserialize at once.  Every call runs once alone first; the concurrent burst must return exactly the same bytes and
// values.  Needs a GPU.  Exit code 0 = all passed.   usage: hbls_concurrency_test [THREADS] [CALLS_PER_THREAD]
#include <atomic>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <thread>
#include <vector>
#include "../../include/hbls.h"

namespace {
struct Case {                       // one call and what it returned when it ran alone
    int kind;                       // 0 GetPublicKey, 1 SignHash, 2 VerifyHash, 3 Signature.Deserialize, 4 PublicKey.Deserialize
    int key, msg;                   // indices into the key / message pools
    uint8_t bytes[96];              // serialized input of kinds 3 / 4
    int want_rc; uint8_t want_out[288];
};
std::vector<blsSecretKey> g_sk; std::vector<blsPublicKey> g_pk; std::vector<blsSignature> g_sig;     // g_sig[key][msg] flattened
std::vector<std::vector<uint8_t>> g_msg;
const int NMSG = 6;

int run(Case& c, uint8_t out[288]) {
    memset(out, 0, 288);
    const std::vector<uint8_t>& m = g_msg[c.msg];
    switch (c.kind) {
    case 0: { blsPublicKey p; blsGetPublicKey(&p, &g_sk[c.key]); memcpy(out, &p, sizeof p); return 0; }
    case 1: { blsSignature s; int rc = blsSignHash(&s, &g_sk[c.key], m.data(), m.size()); memcpy(out, &s, sizeof s); return rc; }
    case 2: return blsVerifyHash(&g_sig[c.key * NMSG + (c.msg % NMSG)], &g_pk[(c.key + (c.msg >= NMSG)) % g_pk.size()], g_msg[c.msg % NMSG].data(), g_msg[c.msg % NMSG].size());
    case 3: { blsSignature s; memset(&s, 0x77, sizeof s); size_t n = blsSignatureDeserialize(&s, c.bytes, 96); memcpy(out, &s, sizeof s); return (int)n; }
    default: { blsPublicKey p; memset(&p, 0x77, sizeof p); size_t n = blsPublicKeyDeserialize(&p, c.bytes, 48); memcpy(out, &p, sizeof p); return (int)n; }
    }
}
}  // namespace

int main(int argc, char** argv) {
    const int T = argc > 1 ? atoi(argv[1]) : 64, N = argc > 2 ? atoi(argv[2]) : 16;
    if (blsInit(HBLS_BLS12_381, HBLS_COMPILED_TIME_VAR) != 0) { fprintf(stderr, "blsInit failed (no GPU?)\n"); return 2; }
    const int K = 8;
    srand(12345);
    g_sk.resize(K); g_pk.resize(K);
    for (int i = 0; i < K; i++) { blsSecretKeySetByCSPRNG(&g_sk[i]); blsGetPublicKey(&g_pk[i], &g_sk[i]); }
    for (int j = 0; j < NMSG; j++) { std::vector<uint8_t> m(j == 5 ? 32 : 48); for (auto& b : m) b = (uint8_t)rand(); g_msg.push_back(m); }
    for (int j = 0; j < NMSG; j++) { std::vector<uint8_t> m(48); for (auto& b : m) b = (uint8_t)rand(); g_msg.push_back(m); }   // never signed
    g_sig.resize(K * NMSG);
    for (int i = 0; i < K; i++) for (int j = 0; j < NMSG; j++) blsSignHash(&g_sig[i * NMSG + j], &g_sk[i], g_msg[j].data(), g_msg[j].size());
    std::vector<Case> cases((size_t)T * N);
    for (auto& c : cases) {
        c.kind = rand() % 5; c.key = rand() % K; c.msg = rand() % (2 * NMSG);
        if (c.kind == 3) {
            const int v = rand() % 3;
            if (v == 0) blsSignatureSerialize(c.bytes, 96, &g_sig[c.key * NMSG + c.msg % NMSG]);
            else for (auto& b : c.bytes) b = (uint8_t)rand();
            if (v == 2) { c.bytes[47] &= 0x19; c.bytes[95] &= 0x19; }
        }
        if (c.kind == 4) {
            if (rand() % 2) blsPublicKeySerialize(c.bytes, 48, &g_pk[c.key]);
            else { for (int b = 0; b < 48; b++) c.bytes[b] = (uint8_t)rand(); c.bytes[47] &= 0x19; }
        }
        c.want_rc = run(c, c.want_out);                       // alone
        if (c.kind == 2 && c.want_rc != (c.msg < NMSG ? 1 : 0)) { fprintf(stderr, "VerifyHash alone returned %d\n", c.want_rc); return 1; }
        if (c.kind == 1 && c.want_rc != 0) { fprintf(stderr, "SignHash alone returned %d\n", c.want_rc); return 1; }
    }
    uint64_t r0 = 0, b0 = 0, l0 = 0; hbls_coalesce_stats(&r0, &b0, &l0);
    std::mutex mu; std::condition_variable cv; int ready = 0; bool go = false;
    std::atomic<int> bad{0};
    std::vector<std::thread> th;
    for (int t = 0; t < T; t++)
        th.emplace_back([&, t] {
            { std::unique_lock<std::mutex> lk(mu); ready++; cv.notify_all(); cv.wait(lk, [&] { return go; }); }
            for (int i = 0; i < N; i++) {
                Case& c = cases[(size_t)t * N + i]; uint8_t out[288];
                const int rc = run(c, out);
                if (rc != c.want_rc || memcmp(out, c.want_out, 288) != 0) {
                    if (bad++ < 5) fprintf(stderr, "mismatch: thread %d call %d kind %d rc %d (alone %d)\n", t, i, c.kind, rc, c.want_rc);
                }
            }
        });
    { std::unique_lock<std::mutex> lk(mu); cv.wait(lk, [&] { return ready == T; }); go = true; cv.notify_all(); }
    for (auto& x : th) x.join();
    uint64_t r1 = 0, b1 = 0, l1 = 0; hbls_coalesce_stats(&r1, &b1, &l1);
    printf("concurrent calls %d: requests %llu in %llu batches, largest batch %llu\n", T * N, (unsigned long long)(r1 - r0),
           (unsigned long long)(b1 - b0), (unsigned long long)l1);
    int fail = bad.load();
    if (r1 - r0 != (uint64_t)T * N) { fprintf(stderr, "coalesce stats counted %llu requests\n", (unsigned long long)(r1 - r0)); fail++; }
    if (fail) { fprintf(stderr, "%d failures\n", fail); return 1; }
    printf("all checks passed\n");
    return 0;
}
