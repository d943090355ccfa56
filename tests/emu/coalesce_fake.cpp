// tests/emu/coalesce_fake.cpp -- TEST HARNESS ONLY: the request combiner of harmony_b200/csrc/coalesce.hpp driven by a fake
// executor (result = a pure function of the input) from many threads; built by tests/test_coalesce_cpu.py under -fsanitize=thread
// and -fsanitize=address.  Prints "all checks passed" and exits 0, or names the first failed check and exits 1.
//   usage: coalesce_fake THREADS REQUESTS_PER_THREAD CAP
#include "../../harmony_b200/csrc/coalesce.hpp"
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <thread>
#include <vector>

struct Req { uint64_t in = 0, out = 0; int owner = -1; };
static uint64_t f(uint64_t x) { x ^= x >> 31; x *= 0x9e3779b97f4a7c15ull; return x ^ (x >> 29); }

static std::atomic<int> failures{0};
#define CHECK(c, ...) do { if (!(c)) { if (failures++ == 0) { fprintf(stderr, "FAILED %s: ", #c); fprintf(stderr, __VA_ARGS__); fputc('\n', stderr); } } } while (0)
static thread_local int tid = -1;

int main(int argc, char** argv) {
    const int T = argc > 1 ? atoi(argv[1]) : 64, N = argc > 2 ? atoi(argv[2]) : 5000;
    const long long cap = argc > 3 ? atoll(argv[3]) : 16;
    hb::FlatCombiner<Req> co;
    std::mutex big;                                   // stands in for the library mutex
    std::atomic<int> inside{0};
    std::atomic<uint64_t> executed{0}, multi{0}, sized{0};
    auto exec = [&](Req* const* b, size_t n) {
        CHECK(inside.fetch_add(1) == 0, "executor entered twice at once");
        CHECK(n >= 1 && (long long)n <= cap, "batch of %zu (cap %lld)", n, cap);
        bool own = false;
        for (size_t i = 0; i < n; i++) { b[i]->out = f(b[i]->in); own |= b[i]->owner == tid; }
        CHECK(own, "thread %d ran a batch without its own request (it ran another one after its request completed)", tid);
        executed += n; sized += n; if (n > 1) multi++;
        inside.fetch_sub(1);
    };
    auto capf = [&] { return cap; };

    // 1. a lone caller: every request is a batch of one, run by the caller itself without waiting for anyone
    tid = 0;
    for (int i = 0; i < 200; i++) {
        Req r; r.in = 7000000 + i; r.owner = 0;
        const hb::CoalesceStats before = co.stats();
        co.submit(r, big, capf, exec);
        const hb::CoalesceStats after = co.stats();
        CHECK(r.out == f(r.in), "lone result");
        CHECK(after.requests == before.requests + 1 && after.batches == before.batches + 1 && after.handoffs == before.handoffs, "lone request %d not a batch of one", i);
    }
    CHECK(co.stats().largest_batch == 1 && multi == 0, "lone caller saw a batch > 1");

    // 2. T threads x N requests, released together; one more thread holds the executor lock now and then (a long batch call)
    std::atomic<bool> go{false}, stop{false};
    std::vector<std::thread> th;
    for (int t = 1; t <= T; t++)
        th.emplace_back([&, t] {
            tid = t;
            while (!go.load()) std::this_thread::yield();
            for (int i = 0; i < N; i++) {
                Req r; r.in = ((uint64_t)t << 32) | (uint64_t)i; r.owner = t;
                co.submit(r, big, capf, exec);
                CHECK(r.out == f(r.in), "thread %d request %d got %llx", t, i, (unsigned long long)r.out);
            }
        });
    std::thread holder([&] {
        while (!go.load()) std::this_thread::yield();
        while (!stop.load()) {
            { std::lock_guard<std::mutex> lk(big); std::this_thread::sleep_for(std::chrono::microseconds(500)); }
            std::this_thread::sleep_for(std::chrono::milliseconds(2));
        }
    });
    go = true;
    for (auto& x : th) x.join();
    stop = true; holder.join();
    const hb::CoalesceStats s = co.stats();
    const uint64_t total = 200 + (uint64_t)T * N;
    CHECK(s.requests == total && executed == total && sized == total, "requests %llu executed %llu of %llu",
          (unsigned long long)s.requests, (unsigned long long)executed.load(), (unsigned long long)total);
    CHECK((long long)s.largest_batch <= cap, "largest batch %llu > cap", (unsigned long long)s.largest_batch);
    if (T > 1) CHECK(multi > 0 && s.batches < s.requests, "no coalescing under contention (%llu batches)", (unsigned long long)s.batches);
    printf("requests %llu batches %llu largest %llu handoffs %llu\n", (unsigned long long)s.requests, (unsigned long long)s.batches,
           (unsigned long long)s.largest_batch, (unsigned long long)s.handoffs);
    if (failures) return 1;
    printf("all checks passed\n");
    return 0;
}
