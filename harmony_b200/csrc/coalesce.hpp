// harmony_b200/csrc/coalesce.hpp -- flat combining of concurrent per-call requests into shared batches (host only, no CUDA).
//
// A caller puts its request on a queue (own small mutex) and waits.  If no combiner is active it becomes the combiner: it takes
// the executor lock first (the library mutex, which may be held by a long batch call), and only then drains up to cap() pending
// requests -- everything that queued while it waited for the lock leaves in the same batch.  It runs them, marks them done, wakes
// their owners and, if requests are still pending, hands the combiner role to the oldest waiter.  A caller therefore executes at
// most ONE batch (the one holding its own request), and a lone caller runs a batch of one at once.  No extra thread, no timer.
//
// Exec: run(Req* const* batch, size_t n) called with the executor lock held; must not throw.
#pragma once
#include <algorithm>
#include <condition_variable>
#include <cstddef>
#include <cstdint>
#include <mutex>

namespace hb {

struct CoalesceStats { uint64_t requests = 0, batches = 0, largest_batch = 0, handoffs = 0; };

template <class Req> class FlatCombiner {
    struct Slot {
        Req* req; Slot* next = nullptr;
        bool done = false, promoted = false;
        std::condition_variable cv;
    };
    std::mutex qmu_;
    Slot *head_ = nullptr, *tail_ = nullptr;
    bool active_ = false;                 // a combiner holds the role (invariant: !active_ => queue empty)
    CoalesceStats stats_;

  public:
    // cap(): batch size limit, read with the executor lock held (>= 1 is enforced)
    template <class Lock, class Cap, class Exec> void submit(Req& r, Lock& exec_lock, Cap&& cap, Exec&& exec) {
        Slot me; me.req = &r;
        {
            std::unique_lock<std::mutex> q(qmu_);
            if (tail_) tail_->next = &me; else head_ = &me;
            tail_ = &me;
            stats_.requests++;
            if (active_) {
                me.cv.wait(q, [&] { return me.done || me.promoted; });
                if (me.done) return;
            } else active_ = true;
        }
        // combiner: our slot is at the head of the queue (fresh queue, or handed the role as the oldest waiter)
        Req* batch_buf[64]; Req** batch = batch_buf; Req** heap = nullptr;
        Slot* first; size_t n = 0;
        {
            std::lock_guard<Lock> big(exec_lock);
            size_t lim = (size_t)std::max<long long>(1, (long long)cap());
            {
                std::lock_guard<std::mutex> q(qmu_);
                first = head_;
                Slot* s = head_;
                while (s && n < lim) { n++; s = s->next; }
                if (n > 64) batch = heap = new Req*[n];
                s = head_;
                for (size_t i = 0; i < n; i++) { batch[i] = s->req; s = s->next; }
                head_ = s; if (!head_) tail_ = nullptr;
                stats_.batches++; if (n > stats_.largest_batch) stats_.largest_batch = n;
            }
            exec(static_cast<Req* const*>(batch), n);
        }
        delete[] heap;
        std::lock_guard<std::mutex> q(qmu_);
        Slot* s = first;
        for (size_t i = 0; i < n; i++) {
            Slot* nx = s->next;           // read before the owner may return and free its slot
            s->done = true;
            if (s != &me) s->cv.notify_one();
            s = nx;
        }
        if (head_) { head_->promoted = true; stats_.handoffs++; head_->cv.notify_one(); }
        else active_ = false;
    }

    CoalesceStats stats() { std::lock_guard<std::mutex> q(qmu_); return stats_; }
};

}  // namespace hb
