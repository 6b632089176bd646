// Best-fit pool of memory blocks over an allocate and a release function (no CUDA here: the
// device pool of a context and the process-wide pinned pool are two instances, see api.cu, and
// tests compile this header with a fake allocator).
#pragma once

#include <stddef.h>

#include <functional>
#include <mutex>
#include <unordered_map>
#include <utility>
#include <vector>

namespace mxb {

// take() hands out the smallest cached block that fits `bytes` without wasting more than
// bytes / slack_div, else a new block from `alloc` (nullptr on failure).  give() caches a block
// of at least `min_cached` bytes while the cache stays within `limit`, and releases the others.
// Every block handed out is in the live map until it is given back; cached blocks are released
// by trim() only (not on destruction: the pinned pool lives until the process exits).  Thread-safe: a block may be
// given back from whichever thread drops its owner (a Python GC).
class BlockPool {
public:
    using Alloc = std::function<void *(size_t)>;
    using Release = std::function<void(void *)>;

    BlockPool(Alloc alloc, Release release, size_t slack_div, size_t min_cached, size_t limit = 0)
        : alloc_(std::move(alloc)), release_(std::move(release)), slack_div_(slack_div),
          min_cached_(min_cached), limit_(limit) {}
    BlockPool(const BlockPool &) = delete;
    BlockPool &operator=(const BlockPool &) = delete;

    void set_limit(size_t limit) {
        std::lock_guard<std::mutex> lock(mu_);
        limit_ = limit;
    }

    // nullptr for 0 bytes, on failure, and (only_cached) when no cached block fits.
    void *take(size_t bytes, bool only_cached = false) {
        if (bytes == 0) return nullptr;
        if (bytes >= min_cached_) {
            std::lock_guard<std::mutex> lock(mu_);
            int best = -1;
            for (int i = 0; i < (int)free_.size(); ++i) {
                const size_t sz = free_[i].first;
                if (sz >= bytes && sz - bytes <= bytes / slack_div_ &&
                    (best < 0 || sz < free_[best].first))
                    best = i;
            }
            if (best >= 0) {
                void *p = free_[best].second;
                const size_t sz = free_[best].first;
                try {
                    live_.emplace(p, sz);
                } catch (...) {
                    return nullptr;
                }
                free_.erase(free_.begin() + best);
                cached_bytes_ -= sz;
                live_bytes_ += sz;
                return p;
            }
        }
        if (only_cached) return nullptr;
        void *p = alloc_(bytes);
        if (!p) return nullptr;
        std::lock_guard<std::mutex> lock(mu_);
        try {
            live_.emplace(p, bytes);
        } catch (...) {
            release_(p);
            return nullptr;
        }
        live_bytes_ += bytes;
        return p;
    }

    // false: `p` is not a live block of this pool (nothing happens).  before_cache runs, outside
    // the lock, when the block is about to be cached rather than released.
    bool give(void *p, const std::function<void()> &before_cache = nullptr) {
        size_t sz = 0;
        {
            std::lock_guard<std::mutex> lock(mu_);
            auto it = live_.find(p);
            if (it == live_.end()) return false;
            sz = it->second;
            live_.erase(it);
            live_bytes_ -= sz;
            if (sz < min_cached_ || cached_bytes_ + sz > limit_) sz = 0;
        }
        if (sz != 0) {
            if (before_cache) before_cache();
            std::lock_guard<std::mutex> lock(mu_);
            if (cached_bytes_ + sz <= limit_) {
                try {
                    free_.emplace_back(sz, p);
                    cached_bytes_ += sz;
                    return true;
                } catch (...) {}
            }
        }
        release_(p);
        return true;
    }

    // Releases every cached block.
    void trim() {
        std::lock_guard<std::mutex> lock(mu_);
        for (auto &ent : free_) release_(ent.second);
        free_.clear();
        cached_bytes_ = 0;
    }

    void stats(size_t *live_bytes, size_t *cached_bytes) const {
        std::lock_guard<std::mutex> lock(mu_);
        if (live_bytes) *live_bytes = live_bytes_;
        if (cached_bytes) *cached_bytes = cached_bytes_;
    }

private:
    Alloc alloc_;
    Release release_;
    const size_t slack_div_, min_cached_;
    size_t limit_;
    mutable std::mutex mu_;
    std::unordered_map<void *, size_t> live_;
    std::vector<std::pair<size_t, void *>> free_;
    size_t live_bytes_ = 0, cached_bytes_ = 0;
};

}  // namespace mxb
