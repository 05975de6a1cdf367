// Multi-GPU plumbing of libcmf_sm100: NCCL bound at run time (dlopen, so the library loads on hosts without NCCL and
// shares the instance a host framework has already loaded), and the worker threads of the single-process multi-GPU
// handle (one host thread per device, driven from the one calling thread -- SURVEY.md section 8b "threading").
#pragma once

#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>   // types and enums only: every entry point is resolved with dlsym

#include <condition_variable>
#include <exception>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

namespace cmf {

struct NcclApi {
    void *lib = nullptr;
    std::string why;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*ReduceScatter)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    ncclResult_t (*GetVersion)(int *) = nullptr;

    bool ok() const { return lib != nullptr; }

    static NcclApi &get() {
        static NcclApi api;
        static std::once_flag once;
        std::call_once(once, [] { api.load(); });
        return api;
    }

  private:
    template <typename F>
    bool sym(F &f, const char *name) {
        f = reinterpret_cast<F>(dlsym(lib, name));
        if (!f) { why = std::string("NCCL symbol missing: ") + name; return false; }
        return true;
    }
    void load() {
        // RTLD_NOLOAD first: reuse the NCCL a host framework (torch) has already mapped, so both sides talk to one library
        const char *names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char *n : names) { lib = dlopen(n, RTLD_NOW | RTLD_NOLOAD); if (lib) break; }
        if (!lib && getenv("CMF_NCCL_LIB")) lib = dlopen(getenv("CMF_NCCL_LIB"), RTLD_NOW | RTLD_GLOBAL);
        for (const char *n : names) { if (lib) break; lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL); }
        if (!lib) { why = std::string("libnccl.so.2 not found (") + (dlerror() ? dlerror() : "") + ")"; return; }
        const bool all = sym(GetUniqueId, "ncclGetUniqueId") && sym(CommInitRank, "ncclCommInitRank") &&
                         sym(CommInitAll, "ncclCommInitAll") && sym(CommDestroy, "ncclCommDestroy") &&
                         sym(AllReduce, "ncclAllReduce") && sym(ReduceScatter, "ncclReduceScatter") &&
                         sym(AllGather, "ncclAllGather") && sym(Broadcast, "ncclBroadcast") && sym(Send, "ncclSend") &&
                         sym(Recv, "ncclRecv") && sym(GroupStart, "ncclGroupStart") && sym(GroupEnd, "ncclGroupEnd") &&
                         sym(GetErrorString, "ncclGetErrorString") && sym(GetVersion, "ncclGetVersion");
        if (!all) lib = nullptr;
    }
};

// One rank's communicator.  `world == 1` (or comm == nullptr) makes every collective a no-op.
struct Comm {
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1;
};

// Persistent worker threads of a single-process multi-GPU handle: run_all(fn) runs fn(rank) on every worker
// concurrently (the ranks meet inside NCCL collectives, so they must run at the same time) and rethrows the first
// failure on the calling thread.
class Workers {
  public:
    explicit Workers(int n) : n_(n), tasks_(n), errs_(n), state_(n, 0) {
        for (int i = 0; i < n; ++i) threads_.emplace_back([this, i] { loop(i); });
    }
    ~Workers() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto &t : threads_) t.join();
    }
    void run_all(const std::function<void(int)> &fn) {
        {
            std::lock_guard<std::mutex> lk(mu_);
            for (int i = 0; i < n_; ++i) { tasks_[i] = fn; errs_[i] = nullptr; state_[i] = 1; }
            pending_ = n_;
        }
        cv_.notify_all();
        std::unique_lock<std::mutex> lk(mu_);
        done_.wait(lk, [this] { return pending_ == 0; });
        for (int i = 0; i < n_; ++i)
            if (errs_[i]) std::rethrow_exception(errs_[i]);
    }
    int size() const { return n_; }

  private:
    void loop(int i) {
        for (;;) {
            std::function<void(int)> fn;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [this, i] { return stop_ || state_[i] == 1; });
                if (stop_) return;
                fn = tasks_[i];
                state_[i] = 2;
            }
            std::exception_ptr err = nullptr;
            try { fn(i); } catch (...) { err = std::current_exception(); }
            {
                std::lock_guard<std::mutex> lk(mu_);
                errs_[i] = err;
                state_[i] = 0;
                if (--pending_ == 0) done_.notify_all();
            }
        }
    }
    int n_;
    std::vector<std::function<void(int)>> tasks_;
    std::vector<std::exception_ptr> errs_;
    std::vector<int> state_;
    std::vector<std::thread> threads_;
    std::mutex mu_;
    std::condition_variable cv_, done_;
    int pending_ = 0;
    bool stop_ = false;
};

}  // namespace cmf
