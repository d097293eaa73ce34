// dh_hostenc.cpp — see dh_hostenc.hpp.  Format: src/db_reader/biwi.rs:81-103 (read_depth):
//   u32 width, u32 height, then until width*height pixels are covered
//   [u32 n_empty][u32 n_full][n_full x u16], little endian.
#include "dh_hostenc.hpp"

#include <algorithm>
#include <cstdlib>
#include <cstdint>
#include <cstring>

#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#if defined(__linux__)
#include <sched.h>
#endif

namespace dh {

namespace {
constexpr size_t kGroup = 16;  // pixels per group = 32 bytes

inline bool group_is_zero(const uint16_t* p) {
#if defined(__SSE2__)
    const __m128i a = _mm_loadu_si128(reinterpret_cast<const __m128i*>(p));
    const __m128i b = _mm_loadu_si128(reinterpret_cast<const __m128i*>(p + 8));
    return _mm_movemask_epi8(_mm_cmpeq_epi8(_mm_or_si128(a, b), _mm_setzero_si128())) == 0xffff;
#else
    uint64_t w[4];
    std::memcpy(w, p, 32);
    return ((w[0] | w[1]) | (w[2] | w[3])) == 0;
#endif
}
inline void put_u32(uint8_t* o, uint32_t v) {  // little endian, any alignment
    o[0] = (uint8_t)v; o[1] = (uint8_t)(v >> 8); o[2] = (uint8_t)(v >> 16); o[3] = (uint8_t)(v >> 24);
}
// Ordinary stores: the copy engine's reads of the pinned slot are then served from the last-level
// cache (streaming stores did not help, DESIGN.md section 5)
inline void put_pixels(uint8_t* o, const uint16_t* src, size_t n) {
#if defined(__BYTE_ORDER__) && __BYTE_ORDER__ == __ORDER_LITTLE_ENDIAN__
    std::memcpy(o, src, n * 2);
#else
    for (size_t i = 0; i < n; ++i) { o[2 * i] = (uint8_t)src[i]; o[2 * i + 1] = (uint8_t)(src[i] >> 8); }
#endif
}
}  // namespace

size_t rle_frame_bound(uint32_t w, uint32_t h) {
    const size_t npx = (size_t)w * h;
    return (8 + 2 * npx + 8 * (npx / (2 * kGroup) + 3) + 15) & ~(size_t)15;
}

size_t rle_encode_frame(const uint16_t* src, uint32_t w, uint32_t h, uint8_t* dst) {
    const size_t npx = (size_t)w * h;
    const size_t n_groups = npx / kGroup, tail = npx - n_groups * kGroup;
    uint8_t* o = dst;
    put_u32(o, w);
    put_u32(o + 4, h);
    o += 8;
    bool tail_zero = true;
    for (size_t i = n_groups * kGroup; i < npx; ++i) tail_zero = tail_zero && src[i] == 0;
    size_t g = 0, covered = 0;
    while (covered < npx) {
        const size_t g0 = g;
        while (g < n_groups && group_is_zero(src + g * kGroup)) ++g;
        size_t n_empty = (g - g0) * kGroup;
        const size_t f0 = g;
        while (g < n_groups && !group_is_zero(src + g * kGroup)) ++g;
        size_t n_full = (g - f0) * kGroup;
        if (g == n_groups && tail) {
            // the last, partial group joins the run it follows: an all-zero tail extends an empty run
            // that reaches it, anything else is copied as pixels
            if (n_full == 0 && tail_zero) n_empty += tail;
            else n_full += tail;
        }
        put_u32(o, (uint32_t)n_empty);
        put_u32(o + 4, (uint32_t)n_full);
        put_pixels(o + 8, src + f0 * kGroup, n_full);
        o += 8 + 2 * n_full;
        covered += n_empty + n_full;
    }
    while ((o - dst) & 3) *o++ = 0;  // files start at multiples of 4 bytes inside a blob
    return (size_t)(o - dst);
}

double rle_sample_density(const uint16_t* src, size_t npx, size_t step) {
    const size_t n_groups = npx / kGroup;
    if (n_groups == 0) return 1.0;
    if (step == 0) step = 1;
    size_t seen = 0, full = 0;
    for (size_t g = 0; g < n_groups; g += step) {
        ++seen;
        full += group_is_zero(src + g * kGroup) ? 0u : 1u;
    }
    return (double)full / (double)seen;
}

unsigned default_encode_threads() {
    if (const char* v = std::getenv("DH_ENCODE_THREADS")) {
        const long x = std::strtol(v, nullptr, 10);
        if (x > 0) return (unsigned)std::min<long>(x, 256);
    }
    unsigned n = 0;
#if defined(__linux__)
    cpu_set_t set;
    CPU_ZERO(&set);
    if (sched_getaffinity(0, sizeof(set), &set) == 0) n = (unsigned)CPU_COUNT(&set);
#endif
    if (n == 0) n = std::thread::hardware_concurrency();
    if (n == 0) n = 4;
    if (n > 4) n -= 1;  // the calling thread keeps a core: it feeds the copy engine while the workers write
    return std::min(n, 16u);
}

// ------------------------------------------------------------------------------------------------ pool
WorkerPool::WorkerPool(unsigned n_threads) {
    if (n_threads == 0) n_threads = 1;
    threads_.reserve(n_threads);
    for (unsigned i = 0; i < n_threads; ++i) threads_.emplace_back([this] { worker(); });
}

WorkerPool::~WorkerPool() {
    {
        std::lock_guard<std::mutex> lk(mu_);
        stop_ = true;
    }
    cv_work_.notify_all();
    for (auto& t : threads_) t.join();
}

uint64_t WorkerPool::run(uint32_t n, std::function<void(uint32_t)> fn) {
    std::unique_lock<std::mutex> lk(mu_);
    const uint64_t ticket = next_ticket_++;
    if (n == 0) {
        finished_.push_back(ticket);
        while (true) {
            auto it = std::find(finished_.begin(), finished_.end(), finished_upto_ + 1);
            if (it == finished_.end()) break;
            finished_.erase(it);
            ++finished_upto_;
        }
        return ticket;
    }
    Job* j = new Job();
    j->ticket = ticket;
    j->n = n;
    j->fn = std::move(fn);
    queue_.push_back(j);
    lk.unlock();
    cv_work_.notify_all();
    return ticket;
}

void WorkerPool::wait(uint64_t ticket) {
    std::unique_lock<std::mutex> lk(mu_);
    cv_done_.wait(lk, [&] {
        return ticket <= finished_upto_ || std::find(finished_.begin(), finished_.end(), ticket) != finished_.end();
    });
}

bool WorkerPool::done(uint64_t ticket) {
    std::lock_guard<std::mutex> lk(mu_);
    return ticket <= finished_upto_ || std::find(finished_.begin(), finished_.end(), ticket) != finished_.end();
}

bool WorkerPool::wait_for(uint64_t ticket, unsigned micros) {
    std::unique_lock<std::mutex> lk(mu_);
    return cv_done_.wait_for(lk, std::chrono::microseconds(micros), [&] {
        return ticket <= finished_upto_ || std::find(finished_.begin(), finished_.end(), ticket) != finished_.end();
    });
}

void WorkerPool::worker() {
    std::unique_lock<std::mutex> lk(mu_);
    for (;;) {
        cv_work_.wait(lk, [&] { return stop_ || !queue_.empty(); });
        if (queue_.empty()) return;  // stop_
        Job* j = queue_.front();
        const uint32_t i = j->next.fetch_add(1);
        if (i + 1 >= j->n) queue_.erase(queue_.begin());  // the last index is handed out: the next job comes up
        lk.unlock();
        bool last = false;
        if (i < j->n) {
            j->fn(i);
            last = j->done.fetch_add(1) + 1 == j->n;
        }
        lk.lock();
        if (last) {
            finished_.push_back(j->ticket);
            while (true) {
                auto it = std::find(finished_.begin(), finished_.end(), finished_upto_ + 1);
                if (it == finished_.end()) break;
                finished_.erase(it);
                ++finished_upto_;
            }
            delete j;
            cv_done_.notify_all();
        }
    }
}

}  // namespace dh
