// parallel.cu — Matcher::match_list_parallel (src/matcher/parallel.rs:18-89) across the GPUs of one node, behind
// the C ABI (include/frz_cuda.h: frz_comm_*, frz_match_list_parallel*).
//
// Reference shape                                        here
//   threads claim 2048-item chunks (parallel.rs:33-63)    GPUs own contiguous index-range shards (SURVEY.md §8(e))
//   matcher.clone() per thread (parallel.rs:46)           frz_matcher_clone per GPU, cached per communicator rank
//   per-thread reverse + radix sort (parallel.rs:67-73)   frz_match_shard_device: the local run stays in HBM
//   join, Vec<Vec<Match>> (parallel.rs:77)                host-out: k_place — every GPU stores its matches at their merged
//   k_merge_matches_by_* (src/k_merge.rs:90-131)            positions in the peers' slice buffers (merge + exchange in one pass)
//                                                         device-out: ONE ncclAllGather of the runs + frz_merge_runs_ex
//   returned Vec<Match>                                   every GPU copies ITS slice of the merged list to the host
//                                                         buffer: the D2H runs over all PCIe links at once
//
// Host-out calls (the caller wants the list in host memory, the bench's `value`) do better than gather-then-merge:
// every rank's per-score table crosses the shared host block, after which every rank KNOWS the merged position of each
// of its matches, and ONE kernel (k_place) stores them straight into the peer GPUs' slice buffers over NVLink (P2P stores
// into cudaIpc-mapped / peer-enabled memory), after which every GPU copies its slice out — the k-way merge and the exchange
// are the same pass, no NCCL kernel, no receive buffer, no second scatter.  The all-gather form remains for device-out
// calls and as the fallback when peer memory cannot be mapped (FRZ_PARALLEL_EXCHANGE=allgather forces it).
//
// The only per-step collective is that all-gather.  The match counts (the `Vec` lengths the k-merge reads) are
// published by each GPU into a small pinned host block shared by all ranks — a 1-thread kernel right after the tile
// scan, i.e. BEFORE the scoring kernels — and every rank's host thread polls the block; the same block carries the
// "my slice has landed" flags that end a host-out step.  In the multi-process form the block (and the output
// buffer) is a memfd segment that every rank maps and pins.
//
// NCCL is resolved with dlopen at the first multi-GPU use: the library itself has no NCCL link dependency, a
// process that already carries PyTorch's libnccl.so.2 shares it, and single-GPU users never need it.
#include <dlfcn.h>
#include <ctype.h>
#include <fcntl.h>
#include <nccl.h>
#include <sched.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/syscall.h>
#include <time.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "frz_device.cuh"
#include "frz_host.h"

#if defined(__x86_64__)
#include <immintrin.h>
#define FRZ_CPU_RELAX() _mm_pause()
#else
#define FRZ_CPU_RELAX() ((void)0)
#endif

namespace {

// ------------------------------------------------------------------------------------- NCCL, loaded lazily
struct NcclApi {
    void* handle = nullptr;
    std::string error;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommInitAll) CommInitAll = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
    decltype(&ncclGetVersion) GetVersion = nullptr;
};

NcclApi& nccl_api() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* names[] = {"libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (api.handle) break;
        }
        if (!api.handle) {
            const char* e = dlerror();
            api.error = std::string("cannot load libnccl.so.2: ") + (e ? e : "?");
            return;
        }
        auto sym = [&](const char* name) -> void* {
            void* p = dlsym(api.handle, name);
            if (!p && api.error.empty()) api.error = std::string("libnccl lacks ") + name;
            return p;
        };
        api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
        api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
        api.CommInitAll = reinterpret_cast<decltype(api.CommInitAll)>(sym("ncclCommInitAll"));
        api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
        api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
        api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
        api.GetVersion = reinterpret_cast<decltype(api.GetVersion)>(sym("ncclGetVersion"));
    });
    return api;
}

frz_status nccl_ready() {
    NcclApi& a = nccl_api();
    if (!a.handle || !a.error.empty()) return frz_fail(FRZ_ERR_NCCL, "%s", a.error.empty() ? "NCCL unavailable" : a.error.c_str());
    return FRZ_OK;
}

#define FRZ_NCCL_TRY(expr)                                                                                       \
    do {                                                                                                         \
        ncclResult_t _r = (expr);                                                                                \
        if (_r != ncclSuccess)                                                                                   \
            return frz_fail(FRZ_ERR_NCCL, "%s failed: %s (%s:%d)", #expr, nccl_api().GetErrorString(_r), __FILE__, __LINE__); \
    } while (0)

// ------------------------------------------------------------------------- shared pinned host memory
// A host allocation every rank's GPU can write.  Local form: cudaHostAlloc(portable | mapped).  Multi-process form:
// rank 0 creates a memfd, the other ranks open it through /proc/<pid>/fd/<n>, everybody maps it MAP_SHARED and
// registers the mapping with CUDA.  The (pid, fd) pair travels over the communicator itself.
struct HostBlock {
    void* ptr = nullptr;
    uint64_t bytes = 0;
    int fd = -1;          // memfd (owner) or the opened peer fd; -1 for cudaHostAlloc memory
    bool registered = false;
};

constexpr uint64_t kCtrlBytes = 8192;
constexpr int kMaxWorld = FRZ_MERGE_MAX_RUNS;   // 64
// control block layout (uint64 words): [parity][rank] for each of the three flag families
constexpr int kCtrlCount = 0;                   // (seq << 32) | match count of the rank's run
constexpr int kCtrlDone = 2 * kMaxWorld;        // seq: the rank's slice of the merged list is in host memory
constexpr int kCtrlBarrier = 4 * kMaxWorld;     // seq: frz_comm_barrier
constexpr int kCtrlTable = 6 * kMaxWorld;       // seq: the rank's score table is in the shared table block
constexpr int kCtrlPlaceErr = 8 * kMaxWorld;    // [rank]: seq of a k_place launch whose wait for the peers timed out
constexpr int kTableBins = 1024;                // longest single-pass score table (sort.cu)

__global__ void k_publish(volatile unsigned long long* slot, const unsigned long long* d_count, unsigned long long seq) {
    const unsigned long long c = d_count ? *d_count : 0ull;
    *slot = (seq << 32) | (c & 0xFFFFFFFFull);
    __threadfence_system();
}

// the rank's per-score table (how many matches of its run score higher than s) → shared host block, then the flag
__global__ void __launch_bounds__(256) k_publish_table(volatile uint32_t* dst, const uint32_t* __restrict__ table, int bins,
                                                       volatile unsigned long long* flag, unsigned long long seq) {
    for (int i = threadIdx.x; i < bins; i += blockDim.x) dst[i] = table ? table[i] : 0u;
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        *flag = seq << 32;
        __threadfence_system();
    }
}

// ---- P2P placement: the exchange and the k-way merge in one pass over peer memory ------------------------------------
// Rank q holds run q sorted; with every rank's score table it knows pos0[s] (merged position of the first element of its
// score-s block) and gt[s] (how many of its elements score higher), so element i with score s belongs at merged position
// pos0[s] + (i - gt[s]).  Position x lives in the slice of rank p with lo[p] <= x < lo[p + 1] (lo[p] = total * p / world): the
// element is stored into rank p's slice buffer, which is this GPU's own memory for p == q and NVLink peer memory otherwise.
// Consecutive elements of a score block land on consecutive addresses, so the stores coalesce.  The block that finishes
// last raises this rank's flag in every peer's header (after a system-scope fence) and then waits for every peer's flag
// in its OWN header: when the kernel ends, this rank's slice is complete and the stream-ordered device→host copy may run.
constexpr size_t kPlaceHeaderBytes = 2048;
struct PlaceHeader {
    unsigned long long arrived[2][kMaxWorld];   // [step parity][source rank] = step sequence number
    unsigned int blocks_done;                   // last-block detection of the owner's own k_place launch
};
static_assert(sizeof(PlaceHeader) <= kPlaceHeaderBytes, "place header");
struct PlaceMeta {
    unsigned char* peer[kMaxWorld];             // every rank's place buffer (header + slice elements) as mapped on THIS device
    unsigned long long lo[kMaxWorld + 1];       // slice boundaries in the merged list
    unsigned long long total;
    int world, rank, bins, parity;
};
__global__ void __launch_bounds__(256) k_place(const FrzMatchDev* __restrict__ run, unsigned long long n, const __grid_constant__ PlaceMeta meta,
                                               const unsigned long long* __restrict__ pos0, const uint32_t* __restrict__ gt,
                                               unsigned long long seq, unsigned long long timeout_ns, volatile unsigned long long* err_slot) {
    __shared__ unsigned long long lo_s[kMaxWorld + 1];
    __shared__ FrzMatchDev* dst_s[kMaxWorld];
    __shared__ int last_s;
    const int world = meta.world, bins = meta.bins;
    for (int i = threadIdx.x; i <= meta.world; i += blockDim.x) lo_s[i] = meta.lo[i];
    for (int i = threadIdx.x; i < meta.world; i += blockDim.x) dst_s[i] = reinterpret_cast<FrzMatchDev*>(meta.peer[i] + kPlaceHeaderBytes);
    __syncthreads();
    const unsigned long long total = meta.total;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const FrzMatchDev m = run[i];
        const uint32_t s = bins > 1 ? min((uint32_t)m.score, (uint32_t)bins - 1) : 0u;
        const unsigned long long x = pos0[s] + (i - gt[s]);
        int p = (int)min((unsigned long long)(world - 1), x * (unsigned long long)world / total);   // lo[p] = floor(total * p / world): at most one off
        while (p > 0 && x < lo_s[p]) p--;
        while (p + 1 < world && x >= lo_s[p + 1]) p++;
        dst_s[p][x - lo_s[p]] = m;
    }
    __threadfence_system();   // this thread's peer stores are performed before the block signs off
    __syncthreads();
    PlaceHeader* mine = reinterpret_cast<PlaceHeader*>(meta.peer[meta.rank]);
    if (threadIdx.x == 0) last_s = atomicAdd(&mine->blocks_done, 1u) == gridDim.x - 1 ? 1 : 0;
    __syncthreads();
    if (!last_s) return;
    __threadfence_system();   // every block fenced its stores before its increment; order them before the flags below
    if (threadIdx.x == 0) mine->blocks_done = 0;   // ready for the next launch
    for (int q = threadIdx.x; q < world; q += blockDim.x) {
        volatile unsigned long long* f = &reinterpret_cast<PlaceHeader*>(meta.peer[q])->arrived[meta.parity][meta.rank];
        *f = seq;
    }
    __threadfence_system();
    unsigned long long t0 = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    for (int q = threadIdx.x; q < world; q += blockDim.x) {
        volatile unsigned long long* f = &mine->arrived[meta.parity][q];
        uint32_t spins = 0;
        while (*f != seq) {
            if ((++spins & 0x3ff) == 0) {
                unsigned long long t1;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                if (t1 - t0 > timeout_ns) { *err_slot = seq; break; }   // a peer never arrived: reported by the host, not a hang
            }
        }
    }
    __threadfence_system();   // acquire side: the peers' stores are visible to whatever follows this kernel on the stream
}

double now_s() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

double poll_timeout_s() {
    static double t = -1;
    if (t < 0) { const char* e = getenv("FRZ_PARALLEL_TIMEOUT_S"); t = e ? atof(e) : 120.0; if (t <= 0) t = 120.0; }
    return t;
}

// waits until every slot carries `seq` in its upper half; lower halves → vals (optional)
frz_status wait_slots(const volatile uint64_t* slots, int world, uint64_t seq, uint64_t* vals, const char* what) {
    const double t0 = now_s();
    for (int r = 0; r < world; r++) {
        uint32_t spins = 0;
        for (;;) {
            const uint64_t v = __atomic_load_n(const_cast<const uint64_t*>(slots + r), __ATOMIC_ACQUIRE);
            if ((v >> 32) == (seq & 0xFFFFFFFFull)) { if (vals) vals[r] = v & 0xFFFFFFFFull; break; }
            FRZ_CPU_RELAX();
            if ((++spins & 0x3FFF) == 0 && now_s() - t0 > poll_timeout_s())
                return frz_fail(FRZ_ERR_NCCL, "rank %d did not publish its %s within %.0f s (peer failed or ranks made different calls)", r, what,
                                poll_timeout_s());
        }
    }
    return FRZ_OK;
}

struct RankCtx {
    int rank = 0;        // global rank
    int device = 0;
    ncclComm_t nccl = nullptr;
    cudaStream_t side = nullptr;           // non-blocking: publishes the count while the main stream scores
    frz_matcher* clone = nullptr;
    uint64_t clone_epoch = 0;
    FrzMatchDev* run = nullptr;            // this rank's locally ordered run
    uint64_t run_cap = 0;
    unsigned long long* d_count = nullptr;
    FrzMatchDev* gathered = nullptr;
    uint64_t gathered_cap = 0;
    FrzMatchDev* merged = nullptr;
    uint64_t merged_cap = 0;
    FrzMergeScratch merge;
    // P2P placement (host-out calls): my run's pos0 and gt tables (pos0[0, bins) then gt[0, bins) in one allocation, staged in
    // one pinned block: they travel in ONE host→device copy); my slice buffer (header + elements), exported to the peers;
    // theirs mapped here
    unsigned long long* d_pos0 = nullptr;
    unsigned long long* h_pos0 = nullptr;
    unsigned char* place_raw = nullptr;
    uint64_t place_cap = 0;                 // elements
    unsigned char* peer_raw[kMaxWorld] = {};
    bool peer_ipc[kMaxWorld] = {};          // opened with cudaIpcOpenMemHandle (multi-process form)
    uint32_t* table_dev = nullptr;          // device-side address of the shared table block
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    bool ev_valid = false;
    uint64_t* ctrl_dev = nullptr;          // device-side address of the shared control block
};

struct Worker {
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::function<void()> job;
    bool has_job = false, done = false, quit = false;
};

}  // namespace

struct frz_comm {
    int world = 1;
    int rank = 0;                 // multi-process: this process's rank; local: 0
    bool local_form = true;
    bool force_nccl = false;      // test hook: FRZ_PARALLEL_FORCE_NCCL=1 runs the all-gather + merge even at world 1
    std::vector<RankCtx> ranks;   // the ranks this process drives (local: all; multi-process: one)
    std::vector<std::unique_ptr<Worker>> workers;   // local form, world > 1: one per GPU
    HostBlock ctrl;
    volatile uint64_t* ctrl_host = nullptr;
    HostBlock tables;             // [parity][rank][kTableBins] uint32: every rank's score table of the current step
    volatile uint32_t* tables_host = nullptr;
    bool p2p_exchange = true;     // host-out calls place matches straight into the peers' slice buffers (k_place); cleared by
                                  // FRZ_PARALLEL_EXCHANGE=allgather, or when peer access / cudaIpc is unavailable
    // local form: rendezvous of the worker threads (allgather_words)
    std::mutex tb_mu;
    std::condition_variable tb_cv;
    int tb_count = 0;
    uint64_t tb_gen = 0;
    std::vector<uint64_t> tb_words;
    uint64_t seq = 0;             // step sequence number (identical on all ranks as long as they make the same calls)
    uint64_t barrier_seq = 0;
    uint64_t alloc_seq = 0;
    std::vector<HostBlock> blocks;   // frz_comm_host_alloc
    std::mutex mu;
};

namespace {

frz_status set_device(int device) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return frz_fail(FRZ_ERR_NO_DEVICE, "no CUDA device available (%s); this library has no CPU fallback",
                        e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n) return frz_fail(FRZ_ERR_INVALID_ARG, "device %d out of range (have %d)", device, n);
    FRZ_CUDA_TRY(cudaSetDevice(device));
    return FRZ_OK;
}

void rank_release(RankCtx& r) {
    cudaSetDevice(r.device);
    if (r.clone) frz_matcher_destroy(r.clone);
    r.clone = nullptr;
    for (int q = 0; q < kMaxWorld; q++) {
        if (r.peer_ipc[q] && r.peer_raw[q]) cudaIpcCloseMemHandle(r.peer_raw[q]);
        r.peer_raw[q] = nullptr; r.peer_ipc[q] = false;
    }
    cudaFree(r.place_raw); r.place_raw = nullptr; r.place_cap = 0;
    cudaFree(r.run); cudaFree(r.d_count); cudaFree(r.gathered); cudaFree(r.merged); cudaFree(r.d_pos0);
    if (r.h_pos0) cudaFreeHost(r.h_pos0);
    r.run = nullptr; r.d_count = nullptr; r.gathered = nullptr; r.merged = nullptr; r.d_pos0 = nullptr; r.h_pos0 = nullptr;
    r.merge.release();
    for (auto& e : r.ev) { if (e) cudaEventDestroy(e); e = nullptr; }
    if (r.side) cudaStreamDestroy(r.side);
    r.side = nullptr;
    if (r.nccl) nccl_api().CommDestroy(r.nccl);
    r.nccl = nullptr;
}

frz_status rank_init(RankCtx& r) {
    FRZ_TRY(set_device(r.device));
    FRZ_CUDA_TRY(cudaStreamCreateWithFlags(&r.side, cudaStreamNonBlocking));
    FRZ_CUDA_TRY(cudaMalloc(&r.d_count, 2 * sizeof(unsigned long long)));
    FRZ_CUDA_TRY(cudaMemset(r.d_count, 0, 2 * sizeof(unsigned long long)));
    for (auto& e : r.ev) FRZ_CUDA_TRY(cudaEventCreate(&e));
    return FRZ_OK;
}

// ---- shared host blocks ----------------------------------------------------------------------------------
void host_block_release(HostBlock& b) {
    if (!b.ptr) return;
    if (b.registered) cudaHostUnregister(b.ptr);
    munmap(b.ptr, b.bytes);
    if (b.fd >= 0) close(b.fd);
    b = HostBlock();
}

// exchange of a few host words between the ranks of a multi-process communicator, over NCCL (set-up time only)
frz_status exchange_words(frz_comm* c, const uint64_t* mine, int n_words, uint64_t* all /* [world * n_words] */) {
    RankCtx& r = c->ranks[0];
    FRZ_TRY(set_device(r.device));
    unsigned long long *d_in = nullptr, *d_out = nullptr;
    frz_status st = [&]() -> frz_status {
        FRZ_CUDA_TRY(cudaMalloc(&d_in, n_words * sizeof(uint64_t)));
        FRZ_CUDA_TRY(cudaMalloc(&d_out, (size_t)c->world * n_words * sizeof(uint64_t)));
        FRZ_CUDA_TRY(cudaMemcpyAsync(d_in, mine, n_words * sizeof(uint64_t), cudaMemcpyHostToDevice, r.side));
        FRZ_NCCL_TRY(nccl_api().AllGather(d_in, d_out, (size_t)n_words, ncclUint64, r.nccl, r.side));
        FRZ_CUDA_TRY(cudaMemcpyAsync(all, d_out, (size_t)c->world * n_words * sizeof(uint64_t), cudaMemcpyDeviceToHost, r.side));
        FRZ_CUDA_TRY(cudaStreamSynchronize(r.side));
        return FRZ_OK;
    }();
    cudaFree(d_in); cudaFree(d_out);
    return st;
}

// every rank contributes n_words (<= 16) host words and receives everybody's: NCCL in the multi-process form, a
// rendezvous of the worker threads in the local form.  Collective; set-up paths only.
constexpr int kGatherWords = 16;
frz_status allgather_words(frz_comm* c, RankCtx& r, const uint64_t* mine, int n_words, uint64_t* all) {
    if (!c->local_form) return exchange_words(c, mine, n_words, all);
    if (c->world == 1) { memcpy(all, mine, n_words * sizeof(uint64_t)); return FRZ_OK; }
    auto rendezvous = [&]() -> bool {
        std::unique_lock<std::mutex> lk(c->tb_mu);
        const uint64_t gen = c->tb_gen;
        if (++c->tb_count == c->world) { c->tb_count = 0; c->tb_gen++; c->tb_cv.notify_all(); return true; }
        return c->tb_cv.wait_for(lk, std::chrono::duration<double>(poll_timeout_s()), [&] { return c->tb_gen != gen; });
    };
    {
        std::lock_guard<std::mutex> lk(c->tb_mu);
        if (c->tb_words.size() < (size_t)c->world * kGatherWords) c->tb_words.resize((size_t)c->world * kGatherWords);
        memcpy(&c->tb_words[(size_t)r.rank * kGatherWords], mine, n_words * sizeof(uint64_t));
    }
    if (!rendezvous()) return frz_fail(FRZ_ERR_NCCL, "a GPU worker did not reach the rendezvous within %.0f s", poll_timeout_s());
    for (int q = 0; q < c->world; q++) memcpy(all + (size_t)q * n_words, &c->tb_words[(size_t)q * kGatherWords], n_words * sizeof(uint64_t));
    if (!rendezvous()) return frz_fail(FRZ_ERR_NCCL, "a GPU worker did not reach the rendezvous within %.0f s", poll_timeout_s());
    return FRZ_OK;
}

// Slice buffers of the P2P placement: every rank owns `header + cap elements`, every other rank maps it (local form: peer
// access between the devices of one process; multi-process form: cudaIpc handles exchanged over the communicator).
// Grow-only and COLLECTIVE: `need` is derived from the step's total match count, which every rank knows, so all ranks
// take the same branch.  On any failure every rank clears c->p2p_exchange and the caller falls back to the all-gather.
frz_status ensure_place_buffers(frz_comm* c, RankCtx& r, uint64_t need, bool* ready) {
    *ready = false;
    if (r.place_cap >= need) { *ready = true; return FRZ_OK; }
    const int world = c->world;
    FRZ_CUDA_TRY(cudaDeviceSynchronize());   // nothing of mine may still read or write the old buffers
    for (int q = 0; q < world; q++) {
        if (r.peer_ipc[q] && r.peer_raw[q]) cudaIpcCloseMemHandle(r.peer_raw[q]);
        r.peer_raw[q] = nullptr; r.peer_ipc[q] = false;
    }
    uint64_t w[10], all[kMaxWorld * 10];
    memset(w, 0, sizeof w);
    FRZ_TRY(allgather_words(c, r, w, 1, all));   // everybody has dropped its mappings: the owners may free
    cudaFree(r.place_raw); r.place_raw = nullptr; r.place_cap = 0;
    const uint64_t want = need + need / 4 + 4096;
    bool ok = cudaMalloc(&r.place_raw, kPlaceHeaderBytes + want * sizeof(FrzMatchDev)) == cudaSuccess &&
              cudaMemset(r.place_raw, 0, kPlaceHeaderBytes) == cudaSuccess;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t size");
    if (ok && !c->local_form) {
        cudaIpcMemHandle_t h;
        ok = cudaIpcGetMemHandle(&h, r.place_raw) == cudaSuccess;
        if (ok) memcpy(&w[2], &h, sizeof h);
    }
    if (!ok) cudaGetLastError();
    w[0] = ok ? 1 : 0;
    w[1] = (uint64_t)reinterpret_cast<uintptr_t>(r.place_raw);
    FRZ_TRY(allgather_words(c, r, w, 10, all));
    for (int q = 0; q < world; q++) ok = ok && all[(size_t)q * 10] == 1;
    if (ok) {
        for (int q = 0; q < world && ok; q++) {
            if (q == r.rank) { r.peer_raw[q] = r.place_raw; continue; }
            if (c->local_form) { r.peer_raw[q] = reinterpret_cast<unsigned char*>((uintptr_t)all[(size_t)q * 10 + 1]); continue; }
            cudaIpcMemHandle_t h;
            memcpy(&h, &all[(size_t)q * 10 + 2], sizeof h);
            void* mapped = nullptr;
            if (cudaIpcOpenMemHandle(&mapped, h, cudaIpcMemLazyEnablePeerAccess) == cudaSuccess) {
                r.peer_raw[q] = static_cast<unsigned char*>(mapped);
                r.peer_ipc[q] = true;
            } else { cudaGetLastError(); ok = false; }
        }
    }
    uint64_t okw = ok ? 1 : 0;
    FRZ_TRY(allgather_words(c, r, &okw, 1, all));   // also: nobody stores into a buffer before its owner has zeroed the header
    for (int q = 0; q < world; q++) ok = ok && all[q] == 1;
    if (!ok) {   // every rank sees the same verdict: P2P placement is off for this communicator from now on
        for (int q = 0; q < world; q++) {
            if (r.peer_ipc[q] && r.peer_raw[q]) cudaIpcCloseMemHandle(r.peer_raw[q]);
            r.peer_raw[q] = nullptr; r.peer_ipc[q] = false;
        }
        cudaFree(r.place_raw); r.place_raw = nullptr; r.place_cap = 0;
        if (&r == &c->ranks[0]) c->p2p_exchange = false;   // one writer; the other workers read it at their next call
        return FRZ_OK;
    }
    r.place_cap = want;
    *ready = true;
    return FRZ_OK;
}

// ---- NUMA placement of the shared host buffer ------------------------------------------------------------------
// All G GPUs copy their slices into the buffer at the same moment: G x 52 GB/s of inbound DMA writes.  With every page on
// one memory node that node's DRAM write bandwidth and the socket interconnect are the limit (measured at 8 GPUs: the
// eight concurrent 6 MB slice copies took 0.28 ms instead of 0.11 ms, profiles/r02g_bench_n8.json; 0.21 ms with the
// first-touch placement below, whose parts only line up with the slices when the list fills the buffer,
// profiles/r02l_bench_n8.json).  See first_touch_near().
int gpu_numa_node(int device) {
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (char* p = bus; *p; p++) *p = (char)tolower(*p);
    char path[128];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = fopen(path, "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    return node;
}
bool node_cpus(int node, cpu_set_t* set) {   // parses /sys/devices/system/node/nodeN/cpulist ("0-31,64-95")
    char path[96];
    snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    FILE* f = fopen(path, "r");
    if (!f) return false;
    CPU_ZERO(set);
    int a = 0, b = 0, n = 0;
    for (;;) {
        if (fscanf(f, "%d", &a) != 1) break;
        b = a;
        int ch = fgetc(f);
        if (ch == '-') { if (fscanf(f, "%d", &b) != 1) break; ch = fgetc(f); }
        for (int cpu = a; cpu <= b && cpu < CPU_SETSIZE; cpu++) { CPU_SET(cpu, set); n++; }
        if (ch != ',') break;
    }
    fclose(f);
    return n > 0;
}
// Page placement of the shared host buffers: rank r first-touches the r-th part of the buffer from a CPU of its GPU's node
// (exact only when the list fills the buffer: slices are fractions of the USED part).  Measured at 8 GPUs (profiles/r02n_*,
// FRZ_PARALLEL_DEBUG=1 prints where the pages are): rank 0's 6 MB slice copy takes 0.19 ms with this placement against
// 0.26 ms with the pages interleaved over the memory nodes and 0.115 ms alone.  Leaving placement to the kernel tied only
// because the ranks happened to run on their GPU's node; in the one-process form it puts every page on one node.
bool numa_debug() { static int d = -1; if (d < 0) { const char* e = getenv("FRZ_PARALLEL_DEBUG"); d = e && atoi(e) ? 1 : 0; } return d == 1; }
// node of the page holding `addr` (move_pages with a null target = query), -1 when unknown
int page_node(void* addr) {
    void* page = reinterpret_cast<void*>(reinterpret_cast<uintptr_t>(addr) & ~4095ull);
    int status = -1;
    if (syscall(SYS_move_pages, 0, 1ul, &page, nullptr, &status, 0) != 0) return -1;
    return status;
}
// touches [lo, hi) of `ptr` (one byte per page, value preserved as zero) from a CPU near `device`, then restores the affinity
void first_touch_near(int device, unsigned char* ptr, uint64_t lo, uint64_t hi) {
    cpu_set_t old_set, near_set;
    const bool have_old = sched_getaffinity(0, sizeof old_set, &old_set) == 0;
    const int node = gpu_numa_node(device);
    bool moved = false;
    if (have_old && node >= 0 && node_cpus(node, &near_set)) {
        cpu_set_t both;
        CPU_AND(&both, &near_set, &old_set);   // stay inside whatever the launcher allowed
        if (CPU_COUNT(&both) > 0) moved = sched_setaffinity(0, sizeof both, &both) == 0;
    }
    for (uint64_t off = lo & ~4095ull; off < hi; off += 4096) ptr[off] = 0;
    if (moved) sched_setaffinity(0, sizeof old_set, &old_set);
    if (numa_debug() && hi > lo)
        fprintf(stderr, "[frz numa] device %d: sysfs node %d, affinity %s; pages of [%llu, %llu): first on node %d, middle %d, last %d\n",
                device, node, moved ? "moved" : "unchanged", (unsigned long long)lo, (unsigned long long)hi,
                page_node(ptr + lo), page_node(ptr + (lo + hi) / 2), page_node(ptr + hi - 1));
}

frz_status host_block_alloc(frz_comm* c, uint64_t bytes, HostBlock* out) {
    HostBlock b;
    bytes = (bytes + 4095) & ~4095ull;
    if (bytes == 0) bytes = 4096;
    b.bytes = bytes;
    if (c->local_form) {
        // one process: anonymous pages, part g touched near GPU g, then pinned for all devices
        b.ptr = mmap(nullptr, bytes, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
        if (b.ptr == MAP_FAILED) return frz_fail(FRZ_ERR_OOM, "cannot map %llu bytes of host memory", (unsigned long long)bytes);
        const int world = c->world;
        for (int g = 0; g < world; g++)
            first_touch_near(c->ranks[g].device, static_cast<unsigned char*>(b.ptr), bytes * (uint64_t)g / world, bytes * (uint64_t)(g + 1) / world);
        FRZ_TRY(set_device(c->ranks[0].device));
        if (cudaHostRegister(b.ptr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped) != cudaSuccess) {
            cudaGetLastError();
            munmap(b.ptr, bytes);
            return frz_fail(FRZ_ERR_OOM, "cannot pin %llu bytes of host memory", (unsigned long long)bytes);
        }
        b.registered = true;
        *out = b;
        return FRZ_OK;
    }
    // multi-process: rank 0 owns a memfd; every rank learns (pid, fd, status) from the exchange
    uint64_t mine[3] = {0, 0, 0};
    if (c->rank == 0) {
        b.fd = memfd_create("frz_comm", MFD_CLOEXEC);
        if (b.fd >= 0 && ftruncate(b.fd, (off_t)bytes) != 0) { close(b.fd); b.fd = -1; }
        mine[0] = (uint64_t)getpid(); mine[1] = (uint64_t)(int64_t)b.fd; mine[2] = b.fd >= 0 ? 1 : 0;
    }
    std::vector<uint64_t> all((size_t)c->world * 3);
    FRZ_TRY(exchange_words(c, mine, 3, all.data()));
    if (all[2] != 1) { if (b.fd >= 0) close(b.fd); return frz_fail(FRZ_ERR_OOM, "rank 0 could not create a %llu-byte shared memory segment", (unsigned long long)bytes); }
    if (c->rank != 0) {
        char path[64];
        snprintf(path, sizeof path, "/proc/%llu/fd/%lld", (unsigned long long)all[0], (long long)(int64_t)all[1]);
        b.fd = open(path, O_RDWR | O_CLOEXEC);
    }
    uint64_t ok = b.fd >= 0 ? 1 : 0;
    if (ok) {
        b.ptr = mmap(nullptr, bytes, PROT_READ | PROT_WRITE, MAP_SHARED, b.fd, 0);
        if (b.ptr == MAP_FAILED) { b.ptr = nullptr; ok = 0; }
    }
    // page placement (first_touch_near above): every rank touches ITS part of the segment, everybody waits, then everybody pins
    if (ok)
        first_touch_near(c->ranks[0].device, static_cast<unsigned char*>(b.ptr), bytes * (uint64_t)c->rank / c->world,
                         bytes * (uint64_t)(c->rank + 1) / c->world);
    std::vector<uint64_t> oks(c->world);
    FRZ_TRY(exchange_words(c, &ok, 1, oks.data()));
    if (ok) {
        FRZ_TRY(set_device(c->ranks[0].device));
        if (cudaHostRegister(b.ptr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped) == cudaSuccess) b.registered = true;
        else { cudaGetLastError(); ok = 0; }
    }
    // everybody must agree before anybody uses it (and before rank 0 could drop the fd)
    FRZ_TRY(exchange_words(c, &ok, 1, oks.data()));
    bool all_ok = true;
    for (uint64_t v : oks) all_ok = all_ok && v == 1;
    if (!all_ok) {
        if (b.ptr) { if (b.registered) cudaHostUnregister(b.ptr); munmap(b.ptr, bytes); }
        if (b.fd >= 0) close(b.fd);
        return frz_fail(FRZ_ERR_OOM, "could not map and pin the %llu-byte shared host segment on every rank", (unsigned long long)bytes);
    }
    // (a fresh memfd reads as zeros and first_touch_near only writes zeros: the control block starts clean)
    *out = b;
    return FRZ_OK;
}

frz_status comm_finish_setup(frz_comm* c) {
    { const char* e = getenv("FRZ_PARALLEL_FORCE_NCCL"); c->force_nccl = e && atoi(e) != 0; }
    FRZ_TRY(host_block_alloc(c, kCtrlBytes, &c->ctrl));
    c->ctrl_host = reinterpret_cast<volatile uint64_t*>(c->ctrl.ptr);
    {   // host-out exchange: p2p (default) → allgather
        const char* e = getenv("FRZ_PARALLEL_EXCHANGE");
        c->p2p_exchange = !(e && strcmp(e, "allgather") == 0) && c->world > 1;
    }
    if (c->p2p_exchange && c->local_form) {   // one process: plain peer access between every pair of devices
        for (RankCtx& a : c->ranks) {
            FRZ_TRY(set_device(a.device));
            for (RankCtx& b : c->ranks) {
                if (a.device == b.device) continue;
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, a.device, b.device) != cudaSuccess || !can) { cudaGetLastError(); c->p2p_exchange = false; continue; }
                const cudaError_t pe = cudaDeviceEnablePeerAccess(b.device, 0);
                if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) c->p2p_exchange = false;
                cudaGetLastError();
            }
        }
    }
    if (c->world > 1) {
        FRZ_TRY(host_block_alloc(c, (uint64_t)2 * c->world * kTableBins * sizeof(uint32_t), &c->tables));
        c->tables_host = reinterpret_cast<volatile uint32_t*>(c->tables.ptr);
    }
    for (RankCtx& r : c->ranks) {
        FRZ_TRY(set_device(r.device));
        void* dp = nullptr;
        FRZ_CUDA_TRY(cudaHostGetDevicePointer(&dp, c->ctrl.ptr, 0));
        r.ctrl_dev = reinterpret_cast<uint64_t*>(dp);
        if (c->world > 1) {
            FRZ_CUDA_TRY(cudaHostGetDevicePointer(&dp, c->tables.ptr, 0));
            r.table_dev = reinterpret_cast<uint32_t*>(dp);
            const size_t table_bytes = (size_t)kTableBins * (sizeof(unsigned long long) + sizeof(uint32_t));
            FRZ_CUDA_TRY(cudaMalloc(&r.d_pos0, table_bytes));
            FRZ_CUDA_TRY(cudaMallocHost(&r.h_pos0, table_bytes));
        }
    }
    return FRZ_OK;
}

void worker_main(Worker* w, int device) {
    cudaSetDevice(device);
    for (;;) {
        std::function<void()> job;
        {
            std::unique_lock<std::mutex> lk(w->mu);
            w->cv.wait(lk, [&] { return w->has_job || w->quit; });
            if (w->quit) return;
            job = std::move(w->job);
            w->has_job = false;
        }
        job();
        {
            std::lock_guard<std::mutex> lk(w->mu);
            w->done = true;
        }
        w->cv.notify_all();
    }
}

// ------------------------------------------------------------------------------------------ one rank's step
struct StepResult {
    frz_status status = FRZ_OK;
    std::string error;
    uint64_t total = 0;
    const FrzMatchDev* d_merged = nullptr;
};

// a shard that arrives as HOST Arrow buffers (end-to-end calls): matched while it streams in (host.cu: frz_match_shard_streamed)
struct HostShard {
    const uint8_t* bytes;
    const void* offsets;
    int offset_width;
    uint64_t n;
};

// Everything one GPU does for one match_list_parallel call.  `seq` is the step number shared by all ranks.
// `host_only`: the caller only needs the list in host memory (no device copy of the whole merged list): P2P placement allowed.
// Exactly one of `shard` (resident packed corpus) and `hs` (host buffers) is given.
frz_status rank_step(frz_comm* c, RankCtx& r, frz_matcher* m, const frz_corpus* shard, const HostShard* hs, uint32_t index_offset, uint64_t seq,
                     frz_match* out_host, uint64_t cap, bool want_host, bool host_only, StepResult* res) {
    FRZ_TRY(set_device(r.device));
    cudaStream_t main = nullptr;   // the device's legacy default stream: ordered with the caller's own default-stream work
    const int world = c->world;
    const int parity = (int)(seq & 1);
    if (!m || (!shard && !hs)) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    if (shard && frz_corpus_device(shard) != r.device)
        return frz_fail(FRZ_ERR_INVALID_ARG, "shard of rank %d lives on device %d, the communicator expects device %d", r.rank,
                        frz_corpus_device(shard), r.device);
    if (!r.clone || r.clone_epoch != frz_matcher_epoch(m)) {   // parallel.rs:46 — `matcher.clone()` per worker
        if (r.clone) frz_matcher_destroy(r.clone);
        r.clone = nullptr;
        FRZ_TRY(frz_matcher_clone(m, &r.clone));
        r.clone_epoch = frz_matcher_epoch(m);
    }
    const uint64_t n_local = hs ? hs->n : frz_corpus_len(shard);
    if (r.run_cap < std::max<uint64_t>(n_local, 1)) {
        cudaFree(r.run); r.run = nullptr; r.run_cap = 0;
        const uint64_t want = std::max<uint64_t>(n_local, 1);
        FRZ_CUDA_TRY(cudaMalloc(&r.run, want * sizeof(FrzMatchDev)));
        r.run_cap = want;
    }
    FRZ_CUDA_TRY(cudaEventRecord(r.ev[0], main));
    // ---- local pipeline (asynchronous): prefilter → count published → scoring → local order
    if (hs)
        FRZ_TRY(frz_match_shard_streamed(r.clone, hs->bytes, hs->offsets, hs->offset_width, hs->n, r.device, index_offset,
                                         reinterpret_cast<frz_match*>(r.run), r.run_cap, reinterpret_cast<uint64_t*>(r.d_count), main));
    else
        FRZ_TRY(frz_match_shard_device(r.clone, shard, index_offset, reinterpret_cast<frz_match*>(r.run), r.run_cap,
                                       reinterpret_cast<uint64_t*>(r.d_count), main));
    FRZ_TRY(frz_matcher_wait_count(r.clone, r.side));
    k_publish<<<1, 1, 0, r.side>>>(reinterpret_cast<volatile unsigned long long*>(r.ctrl_dev + kCtrlCount + parity * kMaxWorld + r.rank),
                                   r.d_count, seq);
    FRZ_CUDA_TRY(cudaGetLastError());
    FRZ_CUDA_TRY(cudaEventRecord(r.ev[1], main));
    // ---- the Vec lengths of all workers (k_merge.rs:96-104): polled from the shared block while the GPU scores
    uint64_t counts[kMaxWorld];
    FRZ_TRY(wait_slots(c->ctrl_host + kCtrlCount + parity * kMaxWorld, world, seq, counts, "match count"));
    uint64_t stride = 1, total = 0;
    for (int k = 0; k < world; k++) { stride = std::max(stride, counts[k]); total += counts[k]; }
    res->total = total;
    const bool collective = world > 1 || c->force_nccl;
    const FrzMatchDev* d_final = r.run;
    uint64_t d_final_first = 0;   // merged position of d_final[0] (non-zero in the P2P form)
    const uint8_t sort_mode = frz_matcher_sort(m);
    const bool by_score = (sort_mode == FRZ_SORT_SCORE_THEN_INDEX_ASC || sort_mode == FRZ_SORT_SCORE_THEN_INDEX_DESC) &&
                          frz_matcher_num_patterns(m) > 0;
    const bool reversed = sort_mode == FRZ_SORT_INDEX_DESC || sort_mode == FRZ_SORT_SCORE_THEN_INDEX_DESC;
    int bins = 1;
    const uint32_t* d_table = nullptr;
    if (by_score) d_table = frz_matcher_last_sort_table(r.clone, &bins);
    // ---- host-out calls: P2P PLACEMENT once the slice buffers are ready on every rank (collective, grow-only); otherwise the
    // all-gather below, whose merged list every rank then copies its slice from
    bool placed = false;          // the P2P placement runs this step
    if (want_host && host_only && world > 1 && r.nccl && c->p2p_exchange && (!by_score || bins > 0) && total > 0 && total <= 0xFFFFFFFFull) {
        if (total > cap) {
            FRZ_CUDA_TRY(cudaStreamSynchronize(main));
            return frz_fail(FRZ_ERR_CAPACITY, "output capacity %llu < %llu matches", (unsigned long long)cap, (unsigned long long)total);
        }
        if (!out_host) return frz_fail(FRZ_ERR_INVALID_ARG, "null out");
        FRZ_TRY(ensure_place_buffers(c, r, total / (uint64_t)world + 2, &placed));
    }
    if (placed) {
        // 1. my table → shared block (after the local pipeline on the main stream), everybody's tables ← shared block
        volatile uint32_t* tab_host = c->tables_host + ((size_t)parity * world) * kTableBins;
        if (by_score) {
            // the table is final one kernel before the run (after the sort's scan, before its scatter): publish it from the side
            // stream at that point, so the tables cross the host block — and the host prepares the exchange — while the scatter runs
            cudaStream_t pub = main;
            if (cudaEvent_t tev = frz_matcher_table_event(r.clone)) {
                FRZ_CUDA_TRY(cudaStreamWaitEvent(r.side, tev, 0));
                pub = r.side;
            }
            k_publish_table<<<1, 256, 0, pub>>>(r.table_dev + ((size_t)parity * world + r.rank) * kTableBins, d_table, bins,
                                                reinterpret_cast<volatile unsigned long long*>(r.ctrl_dev + kCtrlTable + parity * kMaxWorld + r.rank), seq);
            FRZ_CUDA_TRY(cudaGetLastError());
            FRZ_TRY(wait_slots(c->ctrl_host + kCtrlTable + parity * kMaxWorld, world, seq, nullptr, "score table"));
        }
        // 2. merged positions of MY run: pos0[s] = everything scoring higher than s in any run + the score-s blocks of the runs
        //    that precede mine in merge order, gt[s] = how many of my run score higher than s.  k_place stores every element
        //    of my run at its merged position inside the owning rank's slice buffer (peer memory over NVLink) and ends when
        //    all peers have done the same
        auto gt_at = [&](int q, int sc) -> uint64_t { return by_score ? (uint64_t)tab_host[(size_t)q * kTableBins + sc] : 0ull; };
        uint64_t* hp = reinterpret_cast<uint64_t*>(r.h_pos0);
        uint32_t* hg = reinterpret_cast<uint32_t*>(hp + bins);
        for (int sc = bins - 1; sc >= 0; sc--) {
            uint64_t acc = 0;
            for (int q = 0; q < world; q++) acc += gt_at(q, sc);
            for (int k = 0; k < world; k++) {
                const int q = reversed ? world - 1 - k : k;
                const uint64_t gtq = gt_at(q, sc);
                if (q == r.rank) { hp[sc] = acc; hg[sc] = (uint32_t)gtq; break; }
                acc += (sc == 0 ? counts[q] : gt_at(q, sc - 1)) - gtq;
            }
        }
        FRZ_CUDA_TRY(cudaMemcpyAsync(r.d_pos0, r.h_pos0, (size_t)bins * (sizeof(uint64_t) + sizeof(uint32_t)), cudaMemcpyHostToDevice, main));
        PlaceMeta meta;
        memset(&meta, 0, sizeof meta);
        for (int q = 0; q < world; q++) meta.peer[q] = r.peer_raw[q];
        for (int p = 0; p <= world; p++) meta.lo[p] = total * (uint64_t)p / (uint64_t)world;
        meta.total = total; meta.world = world; meta.rank = r.rank; meta.bins = bins; meta.parity = parity;
        const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((counts[r.rank] + 255) / 256, 148 * 4));
        k_place<<<grid, 256, 0, main>>>(r.run, counts[r.rank], meta, reinterpret_cast<const unsigned long long*>(r.d_pos0),
                                        reinterpret_cast<const uint32_t*>(r.d_pos0 + bins), seq, (unsigned long long)(poll_timeout_s() * 1e9),
                                        reinterpret_cast<volatile unsigned long long*>(r.ctrl_dev + kCtrlPlaceErr + r.rank));
        FRZ_CUDA_TRY(cudaGetLastError());
        d_final = reinterpret_cast<const FrzMatchDev*>(r.place_raw + kPlaceHeaderBytes);
        d_final_first = meta.lo[r.rank];
    } else if (collective) {
        if (r.run_cap < stride) {
            // another rank's run is longer than this rank's whole shard (ceil partitioning leaves the last shard short, or
            // empty): the all-gather reads `stride` elements from every rank, so move the run into a buffer that long
            FrzMatchDev* bigger = nullptr;
            FRZ_CUDA_TRY(cudaMalloc(&bigger, stride * sizeof(FrzMatchDev)));
            FRZ_CUDA_TRY(cudaMemcpyAsync(bigger, r.run, counts[r.rank] * sizeof(FrzMatchDev), cudaMemcpyDeviceToDevice, main));
            FRZ_CUDA_TRY(cudaStreamSynchronize(main));
            cudaFree(r.run);
            r.run = bigger;
            r.run_cap = stride;
        }
        const uint64_t need = (uint64_t)world * stride;
        if (r.gathered_cap < need) {
            cudaFree(r.gathered); r.gathered = nullptr; r.gathered_cap = 0;
            const uint64_t want = need + need / 4 + 1024;
            FRZ_CUDA_TRY(cudaMalloc(&r.gathered, want * sizeof(FrzMatchDev)));
            r.gathered_cap = want;
        }
        if (r.merged_cap < total) {
            cudaFree(r.merged); r.merged = nullptr; r.merged_cap = 0;
            const uint64_t want = total + total / 4 + 1024;
            FRZ_CUDA_TRY(cudaMalloc(&r.merged, want * sizeof(FrzMatchDev)));
            r.merged_cap = want;
        }
        // ---- THE collective: one all-gather of the per-shard (score, index) runs over NVLink
        if (r.nccl) {
            FRZ_NCCL_TRY(nccl_api().AllGather(r.run, r.gathered, (size_t)stride, ncclUint64, r.nccl, main));
        } else {   // world 1 without a communicator (local form + force flag): the gather of one run is a copy
            FRZ_CUDA_TRY(cudaMemcpyAsync(r.gathered, r.run, stride * sizeof(FrzMatchDev), cudaMemcpyDeviceToDevice, main));
        }
        // ---- k_merge_matches_by on this GPU
        FRZ_TRY(frz_merge_runs_ex(r.merge, r.gathered, stride, counts, world, frz_matcher_sort(m), frz_matcher_score_bound(m), r.merged, main));
        d_final = r.merged;
    }
    res->d_merged = placed ? nullptr : d_final;
    FRZ_CUDA_TRY(cudaEventRecord(r.ev[2], main));
    if (want_host) {
        if (total > cap) {   // every rank sees the same counts, so every rank takes this exit: no collective is left unbalanced
            FRZ_CUDA_TRY(cudaStreamSynchronize(main));
            return frz_fail(FRZ_ERR_CAPACITY, "output capacity %llu < %llu matches", (unsigned long long)cap, (unsigned long long)total);
        }
        if (total && !out_host) return frz_fail(FRZ_ERR_INVALID_ARG, "null out");
        // this rank's slice of the merged list → host (all ranks hold the whole list: the copy uses every PCIe link)
        const uint64_t lo = total * (uint64_t)r.rank / (uint64_t)world, hi = total * (uint64_t)(r.rank + 1) / (uint64_t)world;
        if (hi > lo)
            FRZ_CUDA_TRY(cudaMemcpyAsync(out_host + lo, d_final + (lo - d_final_first), (hi - lo) * sizeof(FrzMatchDev), cudaMemcpyDeviceToHost, main));
    }
    FRZ_CUDA_TRY(cudaEventRecord(r.ev[3], main));
    r.ev_valid = true;
    if (want_host && !c->local_form && world > 1) {
        // "my slice has landed", stream-ordered after the copy; the call returns once every rank has said so
        k_publish<<<1, 1, 0, main>>>(reinterpret_cast<volatile unsigned long long*>(r.ctrl_dev + kCtrlDone + parity * kMaxWorld + r.rank), nullptr, seq);
        FRZ_CUDA_TRY(cudaGetLastError());
    }
    FRZ_CUDA_TRY(cudaStreamSynchronize(main));
    if (placed && __atomic_load_n(const_cast<const uint64_t*>(c->ctrl_host + kCtrlPlaceErr + r.rank), __ATOMIC_ACQUIRE) == seq)
        return frz_fail(FRZ_ERR_NCCL, "rank %d: a peer GPU did not place its matches within %.0f s (peer failed or ranks made different calls)",
                        r.rank, poll_timeout_s());
    if (want_host && !c->local_form && world > 1)
        FRZ_TRY(wait_slots(c->ctrl_host + kCtrlDone + parity * kMaxWorld, world, seq, nullptr, "copy-out flag"));
    return FRZ_OK;
}

void run_job(frz_comm* c, RankCtx& r, frz_matcher* m, const frz_corpus* shard, uint32_t offset, uint64_t seq, frz_match* out,
             uint64_t cap, bool want_host, StepResult* res) {
    res->status = rank_step(c, r, m, shard, nullptr, offset, seq, out, cap, want_host, true, res);
    if (res->status != FRZ_OK) res->error = frz_last_error();
}

}  // namespace

// ================================================================================================ C ABI

extern "C" frz_status frz_comm_unique_id(uint8_t id[FRZ_UNIQUE_ID_BYTES]) {
    if (!id) return frz_fail(FRZ_ERR_INVALID_ARG, "null id");
    FRZ_TRY(nccl_ready());
    static_assert(sizeof(ncclUniqueId) == FRZ_UNIQUE_ID_BYTES, "ncclUniqueId size");
    ncclUniqueId u;
    FRZ_NCCL_TRY(nccl_api().GetUniqueId(&u));
    memcpy(id, &u, sizeof u);
    return FRZ_OK;
}

extern "C" void frz_comm_destroy(frz_comm* c) {
    if (!c) return;
    for (auto& w : c->workers) {
        { std::lock_guard<std::mutex> lk(w->mu); w->quit = true; }
        w->cv.notify_all();
        if (w->th.joinable()) w->th.join();
    }
    for (HostBlock& b : c->blocks) host_block_release(b);
    host_block_release(c->tables);
    host_block_release(c->ctrl);
    for (RankCtx& r : c->ranks) rank_release(r);
    delete c;
}

extern "C" frz_status frz_comm_create_local(int n_gpus, const int* devices, frz_comm** out) {
    if (!out) return frz_fail(FRZ_ERR_INVALID_ARG, "null out");
    if (n_gpus <= 0) return frz_fail(FRZ_ERR_THREADS_ZERO, "threads must be positive");   // parallel.rs:24
    if (n_gpus > kMaxWorld) return frz_fail(FRZ_ERR_INVALID_ARG, "at most %d GPUs per communicator", kMaxWorld);
    std::unique_ptr<frz_comm, void (*)(frz_comm*)> c(new frz_comm(), frz_comm_destroy);
    c->world = n_gpus;
    c->local_form = true;
    c->ranks.resize(n_gpus);
    std::vector<int> devs(n_gpus);
    for (int g = 0; g < n_gpus; g++) {
        devs[g] = devices ? devices[g] : g;
        for (int h = 0; h < g; h++)
            if (devs[h] == devs[g]) return frz_fail(FRZ_ERR_INVALID_ARG, "device %d listed twice", devs[g]);
        c->ranks[g].rank = g;
        c->ranks[g].device = devs[g];
        FRZ_TRY(rank_init(c->ranks[g]));
    }
    if (n_gpus > 1) {
        FRZ_TRY(nccl_ready());
        std::vector<ncclComm_t> comms(n_gpus);
        FRZ_NCCL_TRY(nccl_api().CommInitAll(comms.data(), n_gpus, devs.data()));
        for (int g = 0; g < n_gpus; g++) c->ranks[g].nccl = comms[g];
    }
    FRZ_TRY(comm_finish_setup(c.get()));
    if (n_gpus > 1) {
        for (int g = 0; g < n_gpus; g++) {
            c->workers.emplace_back(new Worker());
            Worker* w = c->workers.back().get();
            w->th = std::thread(worker_main, w, devs[g]);
        }
    }
    *out = c.release();
    return FRZ_OK;
}

extern "C" frz_status frz_comm_create_rank(const uint8_t id[FRZ_UNIQUE_ID_BYTES], int world, int rank, int device, frz_comm** out) {
    if (!out || !id) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    if (world <= 0) return frz_fail(FRZ_ERR_THREADS_ZERO, "threads must be positive");
    if (world > kMaxWorld || rank < 0 || rank >= world) return frz_fail(FRZ_ERR_INVALID_ARG, "bad world/rank %d/%d", rank, world);
    FRZ_TRY(nccl_ready());
    std::unique_ptr<frz_comm, void (*)(frz_comm*)> c(new frz_comm(), frz_comm_destroy);
    c->world = world;
    c->rank = rank;
    c->local_form = false;
    c->ranks.resize(1);
    c->ranks[0].rank = rank;
    c->ranks[0].device = device;
    FRZ_TRY(rank_init(c->ranks[0]));
    ncclUniqueId u;
    memcpy(&u, id, sizeof u);
    FRZ_NCCL_TRY(nccl_api().CommInitRank(&c->ranks[0].nccl, world, u, rank));
    FRZ_TRY(comm_finish_setup(c.get()));
    *out = c.release();
    return FRZ_OK;
}

extern "C" int frz_comm_world(const frz_comm* c) { return c ? c->world : 0; }
extern "C" int frz_comm_rank(const frz_comm* c) { return c ? c->rank : -1; }
extern "C" int frz_comm_device(const frz_comm* c, int i) { return (c && i >= 0 && i < (int)c->ranks.size()) ? c->ranks[i].device : -1; }

extern "C" int frz_comm_exchange_mode(const frz_comm* c) {
    return !c ? -1 : c->p2p_exchange ? 2 : 0;
}

extern "C" frz_status frz_comm_host_alloc(frz_comm* c, uint64_t bytes, void** out) {
    if (!c || !out) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    HostBlock b;
    FRZ_TRY(host_block_alloc(c, bytes, &b));
    c->blocks.push_back(b);
    *out = b.ptr;
    return FRZ_OK;
}

extern "C" frz_status frz_comm_host_free(frz_comm* c, void* p) {
    if (!c || !p) return FRZ_OK;
    for (size_t i = 0; i < c->blocks.size(); i++)
        if (c->blocks[i].ptr == p) {
            for (RankCtx& r : c->ranks) { cudaSetDevice(r.device); cudaDeviceSynchronize(); }
            host_block_release(c->blocks[i]);
            c->blocks.erase(c->blocks.begin() + (long)i);
            return FRZ_OK;
        }
    return frz_fail(FRZ_ERR_INVALID_ARG, "pointer was not allocated by frz_comm_host_alloc on this communicator");
}

extern "C" frz_status frz_comm_barrier(frz_comm* c) {
    if (!c) return frz_fail(FRZ_ERR_INVALID_ARG, "null communicator");
    if (c->local_form || c->world == 1) return FRZ_OK;
    const uint64_t seq = ++c->barrier_seq;
    const int parity = (int)(seq & 1);
    volatile uint64_t* slots = c->ctrl_host + kCtrlBarrier + parity * kMaxWorld;
    __atomic_store_n(const_cast<uint64_t*>(slots + c->rank), seq << 32, __ATOMIC_RELEASE);
    return wait_slots(slots, c->world, seq, nullptr, "barrier flag");
}

extern "C" frz_status frz_corpus_create_sharded(const uint8_t* bytes, const void* offsets, int offset_width, uint64_t n, frz_comm* c,
                                                frz_corpus** shards_out) {
    if (!c || !shards_out || !offsets) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    if (!c->local_form) return frz_fail(FRZ_ERR_INVALID_ARG, "frz_corpus_create_sharded needs a local (single-process) communicator");
    if (offset_width != 4 && offset_width != 8) return frz_fail(FRZ_ERR_INVALID_ARG, "offset_width must be 4 or 8");
    if (n > 0xFFFFFFFFull) return frz_fail(FRZ_ERR_TOO_MANY_ITEMS, "too many items in haystack, will overflow the u32 index: %llu", (unsigned long long)n);
    const int world = c->world;
    const uint64_t per = (n + world - 1) / world;   // shard g = [g * ceil(N/G), (g+1) * ceil(N/G))   (SURVEY.md §8(e))
    for (int g = 0; g < world; g++) shards_out[g] = nullptr;
    for (int g = 0; g < world; g++) {
        const uint64_t lo = std::min<uint64_t>((uint64_t)g * per, n), hi = std::min<uint64_t>((uint64_t)(g + 1) * per, n);
        // an Arrow slice: the offsets pointer moves, the value buffer does not (offsets stay absolute)
        const void* off_g = static_cast<const uint8_t*>(offsets) + lo * (uint64_t)offset_width;
        frz_status s = frz_corpus_create_arrow(bytes, off_g, offset_width, hi - lo, c->ranks[g].device, &shards_out[g]);
        if (s != FRZ_OK) {
            for (int h = 0; h < g; h++) { frz_corpus_destroy(shards_out[h]); shards_out[h] = nullptr; }
            return s;
        }
    }
    return FRZ_OK;
}

extern "C" frz_status frz_match_list_parallel(frz_matcher* m, const frz_corpus* const* shards, int n_shards, frz_comm* c, frz_match* out,
                                              uint64_t cap, uint64_t* n_out) {
    if (!m || !c || !shards) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    if (!c->local_form) return frz_fail(FRZ_ERR_INVALID_ARG, "multi-process communicator: call frz_match_list_parallel_rank on every rank");
    if (n_shards != c->world) return frz_fail(FRZ_ERR_INVALID_ARG, "%d shards for a communicator of %d GPUs", n_shards, c->world);
    std::lock_guard<std::mutex> lock(c->mu);
    uint64_t offs[kMaxWorld], total_items = 0;
    for (int g = 0; g < n_shards; g++) {
        if (!shards[g]) return frz_fail(FRZ_ERR_INVALID_ARG, "null shard %d", g);
        offs[g] = total_items;
        total_items += frz_corpus_len(shards[g]);
    }
    // Matcher::guard_against_haystack_overflow (src/matcher/mod.rs:438-446)
    if (total_items > 0xFFFFFFFFull)
        return frz_fail(FRZ_ERR_TOO_MANY_ITEMS, "too many items in haystack, will overflow the u32 index: %llu > %u (index offset: 0)",
                        (unsigned long long)total_items, 0xFFFFFFFFu);
    const uint64_t seq = ++c->seq;
    std::vector<StepResult> res(c->world);
    if (c->world == 1) {
        run_job(c, c->ranks[0], m, shards[0], 0, seq, out, cap, true, &res[0]);
    } else {
        for (int g = 0; g < c->world; g++) {
            Worker* w = c->workers[g].get();
            {
                std::lock_guard<std::mutex> lk(w->mu);
                w->job = [c, g, m, shards, &offs, seq, out, cap, &res] {
                    run_job(c, c->ranks[g], m, shards[g], (uint32_t)offs[g], seq, out, cap, true, &res[g]);
                };
                w->done = false;
                w->has_job = true;
            }
            w->cv.notify_all();
        }
        for (int g = 0; g < c->world; g++) {
            Worker* w = c->workers[g].get();
            std::unique_lock<std::mutex> lk(w->mu);
            w->cv.wait(lk, [&] { return w->done; });
        }
    }
    if (n_out) *n_out = res[0].total;
    for (int g = 0; g < c->world; g++)
        if (res[g].status != FRZ_OK) return frz_fail(res[g].status, "GPU %d: %s", c->ranks[g].device, res[g].error.c_str());
    return FRZ_OK;
}

extern "C" frz_status frz_match_list_parallel_rank(frz_matcher* m, const frz_corpus* shard, uint32_t index_offset, frz_comm* c, frz_match* out,
                                                   uint64_t cap, uint64_t* n_out, const frz_match** d_out) {
    if (!m || !c || !shard) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    if (c->local_form && c->world != 1) return frz_fail(FRZ_ERR_INVALID_ARG, "local communicator: call frz_match_list_parallel");
    if ((uint64_t)index_offset + frz_corpus_len(shard) > 0xFFFFFFFFull)
        return frz_fail(FRZ_ERR_TOO_MANY_ITEMS, "too many items in haystack, will overflow the u32 index: %llu > %u (index offset: %u)",
                        (unsigned long long)index_offset + frz_corpus_len(shard), 0xFFFFFFFFu, index_offset);
    std::lock_guard<std::mutex> lock(c->mu);
    const uint64_t seq = ++c->seq;
    StepResult res;
    const bool want_host = out != nullptr || cap != 0;
    const frz_status s = rank_step(c, c->ranks[0], m, shard, nullptr, index_offset, seq, out, cap, want_host, d_out == nullptr, &res);
    if (n_out) *n_out = res.total;
    if (d_out) *d_out = reinterpret_cast<const frz_match*>(res.d_merged);
    return s;
}

// End to end on one rank: the shard arrives as HOST Arrow buffers (streamed H2D + pack into the clone's reusable arena),
// then the collective match.  The ingest is asynchronous on the same stream as the local pipeline.
extern "C" frz_status frz_match_list_parallel_rank_host(frz_matcher* m, const uint8_t* bytes, const void* offsets, int offset_width, uint64_t n,
                                                        uint32_t index_offset, frz_comm* c, frz_match* out, uint64_t cap, uint64_t* n_out) {
    if (!m || !c || !offsets) return frz_fail(FRZ_ERR_INVALID_ARG, "null argument");
    if (c->local_form && c->world != 1) return frz_fail(FRZ_ERR_INVALID_ARG, "local communicator: shard with frz_corpus_create_sharded and call frz_match_list_parallel");
    if ((uint64_t)index_offset + n > 0xFFFFFFFFull)
        return frz_fail(FRZ_ERR_TOO_MANY_ITEMS, "too many items in haystack, will overflow the u32 index: %llu > %u (index offset: %u)",
                        (unsigned long long)index_offset + n, 0xFFFFFFFFu, index_offset);
    std::lock_guard<std::mutex> lock(c->mu);
    RankCtx& r = c->ranks[0];
    FRZ_TRY(set_device(r.device));
    if (!r.clone || r.clone_epoch != frz_matcher_epoch(m)) {
        if (r.clone) frz_matcher_destroy(r.clone);
        r.clone = nullptr;
        FRZ_TRY(frz_matcher_clone(m, &r.clone));
        r.clone_epoch = frz_matcher_epoch(m);
    }
    if (offset_width != 4 && offset_width != 8) return frz_fail(FRZ_ERR_INVALID_ARG, "offset_width must be 4 or 8");
    const HostShard hs{bytes, offsets, offset_width, n};
    const uint64_t seq = ++c->seq;
    StepResult res;
    const frz_status s = rank_step(c, r, m, nullptr, &hs, index_offset, seq, out, cap, true, true, &res);
    if (n_out) *n_out = res.total;
    return s;
}

extern "C" frz_status frz_comm_last_timings(frz_comm* c, int local_index, float* ms4, const frz_matcher** clone) {
    if (!c || local_index < 0 || local_index >= (int)c->ranks.size()) return frz_fail(FRZ_ERR_INVALID_ARG, "bad argument");
    RankCtx& r = c->ranks[local_index];
    if (clone) *clone = r.clone;
    if (ms4) {
        ms4[0] = ms4[1] = ms4[2] = ms4[3] = 0;
        if (r.ev_valid) {
            FRZ_TRY(set_device(r.device));
            FRZ_CUDA_TRY(cudaEventSynchronize(r.ev[3]));
            cudaEventElapsedTime(&ms4[0], r.ev[0], r.ev[1]);
            cudaEventElapsedTime(&ms4[1], r.ev[1], r.ev[2]);
            cudaEventElapsedTime(&ms4[2], r.ev[2], r.ev[3]);
            cudaEventElapsedTime(&ms4[3], r.ev[0], r.ev[3]);
            cudaGetLastError();
        }
    }
    return FRZ_OK;
}
