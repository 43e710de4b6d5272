// The device scratch of a single-device context: one stack arena, taken in scopes.
//
// Every temporary device buffer of a call is a region of its context's arena.  A scratch_scope records the top of the
// arena when it opens and restores it when it closes, which releases every region taken inside it; scopes nest and are
// released in stack order (a host entry point opens one, and so does the _dev entry point or helper it calls).  Each
// region starts on a 256-byte boundary, and two live regions never overlap.
//
// Reusing a released region is safe because of stream order: whatever is given the same memory next is written by
// work enqueued on the context stream after the work that read it.  So work on another stream that reads a region must
// be joined into the context stream (an event wait) before the scope that took the region closes.
//
// Blocks never move while a scope is open.  A request that does not fit in what is left of the current block takes an
// overflow block.  When an outermost scope closes and overflow blocks exist, the arena synchronises the stream that
// scope was opened on, frees every block and allocates one block of the peak depth plus 1/8, on the device that was
// current when the scope opened (a caller that holds one scope per device may close them under any device).  So the
// call that grows the arena pays for it, and repeated calls of that shape make no cudaMalloc, no cudaFree and no
// synchronisation.  The footprint is the deepest stack of any single call, except while a call grows the arena: the
// old block and the overflow blocks then exist together until that call ends.
//
// A context is used by one host thread at a time.  multi_batch_partials opens a scope on its first shard on the calling
// thread, and the host localisations (locate.cuh) one on every shard they use; each shard's worker thread then nests
// its own scopes inside it while the caller waits for it in join.
#pragma once
#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>
#include <vector>

class scratch_arena {
  public:
    static constexpr size_t ALIGN = 256;
    struct mark {
        size_t block, off, used;
    };

    scratch_arena() = default;
    scratch_arena(const scratch_arena&) = delete;
    scratch_arena& operator=(const scratch_arena&) = delete;
    ~scratch_arena() {
        for (const block& b : blocks_) cudaFree(b.base);
    }

    // A region of `bytes` in the innermost open scope (an empty request still gets a region of its own).
    cudaError_t take(size_t bytes, void** out) {
        size_t need = bytes ? (bytes + ALIGN - 1) / ALIGN * ALIGN : ALIGN;
        if (blocks_.empty() || off_ + need > blocks_[cur_].cap) {
            // the blocks after the current one hold no live region: take the first that fits, else a new one
            size_t b = blocks_.empty() ? 0 : cur_ + 1;
            while (b < blocks_.size() && blocks_[b].cap < need) b++;
            if (b == blocks_.size()) {
                block nb{nullptr, need};
                if (cudaError_t e = cudaMalloc((void**)&nb.base, nb.cap)) return e;
                blocks_.push_back(nb);
            }
            cur_ = b;
            off_ = 0;
        }
        *out = blocks_[cur_].base + off_;
        off_ += need;
        used_ += need;
        if (used_ > peak_) peak_ = used_;
        return cudaSuccess;
    }

  private:
    friend class scratch_scope;
    struct block {
        uint8_t* base;
        size_t cap;
    };
    mark open(cudaStream_t stream) {
        if (depth_++ == 0) {
            stream_ = stream;
            cudaGetDevice(&device_);
        }
        return {cur_, off_, used_};
    }
    void close(const mark& m) {
        cur_ = m.block;
        off_ = m.off;
        used_ = m.used;
        if (--depth_ == 0 && blocks_.size() > 1) consolidate();
    }
    // One block in place of the grown ones.  A failure here fails no call: when the stream does not synchronise the
    // blocks stay, and when cudaMalloc fails (its error cleared) the next region taken allocates what it needs.
    void consolidate() {
        int current = 0;
        if (cudaGetDevice(&current) != cudaSuccess || cudaSetDevice(device_) != cudaSuccess) return;
        if (cudaStreamSynchronize(stream_) == cudaSuccess) {
            for (const block& b : blocks_) cudaFree(b.base);
            blocks_.clear();
            block nb{nullptr, peak_ + peak_ / 8};
            if (cudaMalloc((void**)&nb.base, nb.cap) == cudaSuccess) blocks_.push_back(nb);
            else (void)cudaGetLastError();
        }
        cudaSetDevice(current);
    }

    std::vector<block> blocks_;  // blocks_[0] and, while the arena grows, the overflow blocks after it
    size_t cur_ = 0, off_ = 0;   // the top: offset `off_` in blocks_[cur_]
    size_t used_ = 0;            // bytes of the live regions (the depth of the stack)
    size_t peak_ = 0;            // the deepest stack so far
    int depth_ = 0;              // open scopes
    cudaStream_t stream_ = nullptr;   // the stream and device of the outermost open scope
    int device_ = 0;
};

class scratch_scope {
  public:
    scratch_scope(scratch_arena& a, cudaStream_t stream) : a_(a), m_(a.open(stream)) {}
    ~scratch_scope() { a_.close(m_); }
    scratch_scope(const scratch_scope&) = delete;
    scratch_scope& operator=(const scratch_scope&) = delete;

  private:
    scratch_arena& a_;
    scratch_arena::mark m_;
};
