// KV page allocator of one cache (host side only: no CUDA call, so tests can compile it into a plain host program).
//
// A cache owns `pool_pages` pages of kKvPage tokens ([L][pool_pages][nkv][64][d] on the device) and a page table
// [max_batch, pages_per_seq]: entry (s, p) names the pool page that holds tokens [64 p, 64 (p + 1)) of slot s.
//
// Policy (deterministic, so every tensor-parallel rank makes the same choices):
//   * page p of slot s takes the slot's HOME page s * pages_per_seq + p when that page exists in the pool and is free, otherwise the
//     lowest-numbered free page.  A pool of max_batch * pages_per_seq pages without forks therefore keeps the identity table;
//   * a table entry without a page names the slot's home page if it exists, else page 0, so a stray read stays inside the pool;
//   * reserve() takes every page a call will write, or nothing: a call the pool cannot cover leaves every count and entry unchanged;
//   * a page returns to the free list when its reference count drops to 0.
//
// Fork invariant: fork() shares only the FULL pages of the source (refcount + 1).  Appends write positions >= the slot's length, and
// every shared page lies wholly below the length of each slot that holds it, so a shared page is never written again.  The source's
// partial last page is not shared: the caller copies it into the fresh page fork() takes for the destination.
#pragma once
#include <algorithm>
#include <cstdint>
#include <set>
#include <utility>
#include <vector>

namespace fl {

class KvPool {
public:
    static constexpr int kPage = 64;       // tokens per page (kKvPage)

    KvPool() = default;
    KvPool(int max_batch, int pages_per_seq, int pool_pages) { init(max_batch, pages_per_seq, pool_pages); }

    void init(int max_batch, int pages_per_seq, int pool_pages) {
        B_ = max_batch; P_ = pages_per_seq; N_ = pool_pages;
        ref_.assign((size_t)N_, 0);
        free_.clear();
        for (int i = 0; i < N_; ++i) free_.insert(free_.end(), i);
        pages_.assign((size_t)B_, {});
        table_.assign((size_t)B_ * P_, 0);
        for (int s = 0; s < B_; ++s)
            for (int p = 0; p < P_; ++p) table_[(size_t)s * P_ + p] = unassigned(s, p);
        device_ = table_;
        dirty_.clear();
    }

    int max_batch() const { return B_; }
    int pages_per_seq() const { return P_; }
    int total_pages() const { return N_; }
    int free_pages() const { return (int)free_.size(); }
    int refcount(int page) const { return ref_[(size_t)page]; }
    const std::vector<int>& slot_pages(int s) const { return pages_[(size_t)s]; }
    const std::vector<int>& table() const { return table_; }     // the table the device holds after the next flush()

    static int pages_for(int64_t tokens) { return (int)((tokens + kPage - 1) / kPage); }

    // Pages slot s lacks to hold `tokens` tokens.
    int missing(int s, int64_t tokens) const {
        const int have = (int)pages_[(size_t)s].size(), want = pages_for(tokens);
        return want > have ? want - have : 0;
    }

    // Gives each (slot, tokens) pair pages for positions [0, tokens): all of them, or -- when the free pages do not cover the total --
    // none, returning false.  Slots are served in ascending order, whatever the order of `req`.
    bool reserve(std::vector<std::pair<int, int64_t>> req) {
        int64_t need = 0;
        for (const auto& r : req) need += missing(r.first, r.second);
        if (need > (int64_t)free_.size()) return false;
        std::sort(req.begin(), req.end());
        for (const auto& r : req)
            while ((int)pages_[(size_t)r.first].size() < pages_for(r.second)) take(r.first);
        return true;
    }

    // Drops slot s's references; its table entries fall back to the unassigned default.
    void release(int s) {
        std::vector<int>& v = pages_[(size_t)s];
        for (size_t p = 0; p < v.size(); ++p) {
            if (--ref_[(size_t)v[p]] == 0) free_.insert(v[p]);
            set_entry(s, (int)p, unassigned(s, (int)p));
        }
        v.clear();
    }
    void release_all() {
        for (int s = 0; s < B_; ++s) release(s);
    }

    // Makes the empty slot dst a copy of src's first `len` tokens: src's full pages are shared, and a partial last page gets a fresh
    // page for dst, returned as (src page, dst page) for the caller to copy; (-1, -1) when len is a multiple of 64.  Returns false and
    // changes nothing when dst holds pages, src holds fewer than len tokens' pages, or no page is free for the partial copy.
    bool fork(int src, int dst, int64_t len, std::pair<int, int>* copy) {
        const std::vector<int>& sp = pages_[(size_t)src];
        const int full = (int)(len / kPage);
        const bool partial = len % kPage != 0;
        if (src == dst || !pages_[(size_t)dst].empty() || (int)sp.size() < pages_for(len)) return false;
        if (partial && free_.empty()) return false;
        for (int p = 0; p < full; ++p) {
            ++ref_[(size_t)sp[(size_t)p]];
            pages_[(size_t)dst].push_back(sp[(size_t)p]);
            set_entry(dst, p, sp[(size_t)p]);
        }
        *copy = {-1, -1};
        if (partial) *copy = {sp[(size_t)full], take(dst)};
        return true;
    }

    // Entries whose page changed since the last flush, as (index into the [max_batch, pages_per_seq] table, page); the caller writes
    // them to the device table.  Entries that changed and changed back are not listed.
    std::vector<std::pair<int, int>> flush() {
        std::vector<std::pair<int, int>> out;
        for (int i : dirty_)
            if (device_[(size_t)i] != table_[(size_t)i]) {
                out.push_back({i, table_[(size_t)i]});
                device_[(size_t)i] = table_[(size_t)i];
            }
        dirty_.clear();
        return out;
    }

private:
    int unassigned(int s, int p) const {
        const int64_t home = (int64_t)s * P_ + p;
        return home < N_ ? (int)home : 0;
    }
    void set_entry(int s, int p, int page) {
        const int i = s * P_ + p;
        table_[(size_t)i] = page;
        dirty_.insert(i);
    }
    // Appends one page to slot s: its home page if that is free, else the lowest free page.  The caller checked a page is free.
    int take(int s) {
        const int p = (int)pages_[(size_t)s].size();
        const int64_t home = (int64_t)s * P_ + p;
        int page;
        if (home < N_ && ref_[(size_t)home] == 0) {
            page = (int)home;
            free_.erase(page);
        } else {
            page = *free_.begin();
            free_.erase(free_.begin());
        }
        ref_[(size_t)page] = 1;
        pages_[(size_t)s].push_back(page);
        set_entry(s, p, page);
        return page;
    }

    int B_ = 0, P_ = 0, N_ = 0;
    std::vector<int> ref_;                 // [pool pages] references: slots holding the page
    std::set<int> free_;                   // pages with no reference, ascending
    std::vector<std::vector<int>> pages_;  // [slot] its pages, in position order
    std::vector<int> table_;               // [max_batch * pages_per_seq] the table as it should be on the device
    std::vector<int> device_;              // the table as it is on the device (after the last flush)
    std::set<int> dirty_;                  // entries set since the last flush
};

}  // namespace fl
