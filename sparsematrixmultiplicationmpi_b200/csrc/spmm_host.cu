// spmm_host.cu — the host-buffer half of the C-ABI: what the reference-shaped entry points call.
//
// The reference's operands are host objects: SparseMatrix (three std::vector) and FatVector =
// std::vector<std::vector<double>>, i.e. N separately allocated rows of k doubles
// ("Source Code/MatrixDefinitions.h":14-22). Crossing to the device therefore means
//   pack (N row buffers -> one row-major image, the reference's serialize(), utils.cpp:216-228)
//   -> H2D -> kernel -> D2H -> unpack (deserialize(), utils.cpp:237-253).
// Here pack and unpack run on a small host thread pool straight into / out of pinned staging
// memory owned by the handle, in row chunks, so the copy engine moves chunk c while the CPU packs
// chunk c+1; wide operands additionally travel in two k-slabs so that the upload of the second
// overlaps the download of the first (PCIe is full duplex). A flat pageable buffer (a C caller's
// malloc, numpy storage) takes the same route with "row i = base + i*k"; a flat pinned buffer is
// handed to the copy engine as it is.
//
// Multi-rank strategies inside one process (compat MPI rank-threads, one GPU per rank): helpers to
// stage only the B rows a shard reads, to let the kernel store C rows straight into the root
// rank's device buffer over NVLink (peer access), and to bring the finished C down once.
#include <algorithm>
#include <emmintrin.h>

#include <atomic>
#include <chrono>
#include <cstdio>
#include <condition_variable>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

#include "spmm_internal.h"

namespace spmm
{

// ---- host thread pool: parallel_for over chunk indices; the caller takes part ----------------------------------------
namespace
{
struct Job
{
    std::function<void(int)> fn;
    int n = 0;
    std::atomic<int> next{0}, done{0};
};

class Pool
{
  public:
    Pool()
    {
        int n = (int)std::thread::hardware_concurrency();
        if (const char *e = getenv("SPMM_HOST_THREADS"))
            n = atoi(e);
        n = std::max(1, std::min(n, 32));
        for (int i = 1; i < n; ++i) // the caller is the n-th
            th_.emplace_back([this] { worker(); });
    }
    ~Pool()
    {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto &t : th_)
            t.join();
    }
    int threads() const { return (int)th_.size() + 1; }
    void parallel_for(int n, const std::function<void(int)> &fn)
    {
        if (n <= 0)
            return;
        if (n == 1 || th_.empty())
        {
            for (int i = 0; i < n; ++i)
                fn(i);
            return;
        }
        auto job = std::make_shared<Job>();
        job->fn = fn;
        job->n = n;
        {
            std::lock_guard<std::mutex> lk(mu_);
            q_.push_back(job);
        }
        cv_.notify_all();
        run(job);
        while (job->done.load(std::memory_order_acquire) < n)
            std::this_thread::yield();
    }

  private:
    void run(const std::shared_ptr<Job> &j)
    {
        for (;;)
        {
            const int i = j->next.fetch_add(1);
            if (i >= j->n)
                break;
            j->fn(i);
            j->done.fetch_add(1, std::memory_order_release);
        }
        std::lock_guard<std::mutex> lk(mu_);
        for (auto it = q_.begin(); it != q_.end(); ++it)
            if (*it == j)
            {
                q_.erase(it);
                break;
            }
    }
    void worker()
    {
        for (;;)
        {
            std::shared_ptr<Job> j;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return stop_ || !q_.empty(); });
                if (stop_)
                    return;
                j = q_.front();
            }
            run(j);
        }
    }
    std::vector<std::thread> th_;
    std::mutex mu_;
    std::condition_variable cv_;
    std::deque<std::shared_ptr<Job>> q_;
    bool stop_ = false;
};

Pool &pool()
{
    static Pool p;
    return p;
}

} // namespace
void host_parallel_for(int n, const std::function<void(int)> &fn) { pool().parallel_for(n, fn); }
namespace
{

// A dense host operand: either N row pointers (the memory shape of a FatVector) or one flat row-major block.
struct HostRows
{
    const double *const *rows = nullptr; // rows[i] -> k doubles
    const double *flat = nullptr;        // row i at flat + i*ld
    long long ld = 0;
    const double *at(long long i) const { return rows ? rows[i] : flat + i * ld; }
};
struct HostRowsOut
{
    double *const *rows = nullptr;
    double *flat = nullptr;
    long long ld = 0;
    double *at(long long i) const { return rows ? rows[i] : flat + i * ld; }
};

bool is_pinned(const void *p)
{
    if (!p)
        return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess)
    {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost;
}

constexpr size_t CHUNK_BYTES = 1u << 20; // pipeline chunk: about 1 MB of rows, packed / unpacked by one host thread
constexpr int RING_WORKERS_MAX = 16;     // host threads that pack / unpack side by side, two ring slots each
constexpr int RING_SLOTS = 2 * RING_WORKERS_MAX;
int ring_workers()
{
    static const int w = [] {
        int v = 16; // measured on the B200 host (16 cores), cfg2 k=64 through the C++ entry point: 13.4 / 8.3 / 6.9 / 5.7 ms with 4 / 8 / 12 / 16 workers
        if (const char *e = getenv("SPMM_RING_WORKERS"))
            v = atoi(e);
        return std::max(1, std::min(v, RING_WORKERS_MAX));
    }();
    return w;
}

int ensure_device(double **buf, size_t *have, size_t want)
{
    if (*have >= want)
        return SPMM_OK;
    cudaFree(*buf);
    *buf = nullptr;
    *have = 0;
    SPMM_CUDA(cudaMalloc((void **)buf, sizeof(double) * std::max<size_t>(want, 1)));
    *have = want;
    return SPMM_OK;
}

int ensure_streams(spmm_csr_t A)
{
    if (!A->stream)
        SPMM_CUDA(cudaStreamCreateWithFlags(&A->stream, cudaStreamNonBlocking));
    if (!A->stream_up)
    {
        SPMM_CUDA(cudaStreamCreateWithFlags(&A->stream_up, cudaStreamNonBlocking));
        SPMM_CUDA(cudaStreamCreateWithFlags(&A->stream_down, cudaStreamNonBlocking));
    }
    while (A->events.size() < 16)
    {
        cudaEvent_t e;
        SPMM_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        A->events.push_back(e);
    }
    return SPMM_OK;
}

// Pinned staging rings: two slots per packing thread and direction, one event per slot. Small rings instead of full mirrors
// of B and C keep the first call on a new matrix cheap (page-locking 124 MB costs tens of milliseconds; the reference calls
// each function once per run). The slots are carved from one portable page-locked arena that spmm_devices_init allocates at
// program start (outside every timed call; 8 rank-threads that each page-locked their own ring inside their first row-wise
// call made that call 279 ms at -np 8); a lease that does not fit the arena page-locks its own memory and keeps it for later.
constexpr int ARENA_SLOTS = 128; // 1 MB each
struct Arena
{
    double *buf = nullptr;
    bool used[ARENA_SLOTS] = {};
};
std::mutex g_ring_mu;
Arena g_arena;

struct Ring
{
    int device = -1, n_slots = 0; // slots per direction
    double *buf = nullptr;
    int arena_first = -1;         // >= 0: carved from the arena
    cudaEvent_t ev[2 * RING_SLOTS] = {};
    double *slot(int dir, int i) const { return buf + ((size_t)(dir * n_slots + i) * CHUNK_BYTES) / sizeof(double); }
    cudaEvent_t event(int dir, int i) const { return ev[dir * RING_SLOTS + i]; }
};
std::vector<Ring *> g_rings_free; // private (non-arena) rings waiting for their next lease

int arena_init()
{
    std::lock_guard<std::mutex> lk(g_ring_mu);
    if (g_arena.buf)
        return SPMM_OK;
    SPMM_CUDA(cudaHostAlloc((void **)&g_arena.buf, (size_t)ARENA_SLOTS * CHUNK_BYTES, cudaHostAllocPortable));
    return SPMM_OK;
}

// a ring with `want` slots per direction for work on `device`
int borrow_ring(int device, int want, Ring **out)
{
    want = std::max(1, std::min(want, RING_SLOTS));
    Ring *r = nullptr;
    {
        std::lock_guard<std::mutex> lk(g_ring_mu);
        if (g_arena.buf)
        {
            int run = 0;
            for (int i = 0; i < ARENA_SLOTS && !r; ++i)
            {
                run = g_arena.used[i] ? 0 : run + 1;
                if (run == 2 * want)
                {
                    r = new Ring();
                    r->arena_first = i + 1 - run;
                    r->buf = g_arena.buf + ((size_t)r->arena_first * CHUNK_BYTES) / sizeof(double);
                    for (int j = r->arena_first; j <= i; ++j)
                        g_arena.used[j] = true;
                }
            }
        }
        for (size_t i = 0; !r && i < g_rings_free.size(); ++i)
            if (g_rings_free[i]->n_slots >= want)
            {
                r = g_rings_free[i];
                g_rings_free.erase(g_rings_free.begin() + (long)i);
            }
    }
    cudaError_t e = cudaSuccess;
    if (!r)
    {
        r = new Ring();
        e = cudaHostAlloc((void **)&r->buf, (size_t)2 * want * CHUNK_BYTES, cudaHostAllocPortable);
        r->n_slots = want;
    }
    if (r->arena_first >= 0)
        r->n_slots = want;
    if (e == cudaSuccess && r->device != device)
    {
        // events belong to a device: (re)create them for this lease's device
        for (int i = 0; i < 2 * RING_SLOTS; ++i)
            if (r->ev[i])
            {
                cudaEventDestroy(r->ev[i]);
                r->ev[i] = nullptr;
            }
        for (int d = 0; d < 2 && e == cudaSuccess; ++d)
            for (int i = 0; i < r->n_slots && e == cudaSuccess; ++i)
                e = cudaEventCreateWithFlags(&r->ev[d * RING_SLOTS + i], cudaEventDisableTiming);
        r->device = device;
    }
    if (e != cudaSuccess)
    {
        for (int i = 0; i < 2 * RING_SLOTS; ++i)
            if (r->ev[i])
                cudaEventDestroy(r->ev[i]);
        if (r->arena_first >= 0)
        {
            std::lock_guard<std::mutex> lk(g_ring_mu);
            for (int j = 0; j < 2 * r->n_slots; ++j)
                g_arena.used[r->arena_first + j] = false;
        }
        else if (r->buf)
            cudaFreeHost(r->buf);
        delete r;
        return cuda_fail(e, "pinned staging ring", __FILE__, __LINE__);
    }
    *out = r;
    return SPMM_OK;
}
void return_ring(Ring *r)
{
    if (!r)
        return;
    if (r->arena_first >= 0)
    {
        for (int i = 0; i < 2 * RING_SLOTS; ++i)
            if (r->ev[i])
                cudaEventDestroy(r->ev[i]);
        std::lock_guard<std::mutex> lk(g_ring_mu);
        for (int j = 0; j < 2 * r->n_slots; ++j)
            g_arena.used[r->arena_first + j] = false;
        delete r;
        return;
    }
    std::lock_guard<std::mutex> lk(g_ring_mu);
    g_rings_free.push_back(r);
}
struct RingLease
{
    Ring *r = nullptr;
    ~RingLease() { return_ring(r); }
};
int rows_per_chunk(int k);
// slots per direction a transfer of `rows` rows of k doubles can use: two per packing thread
int ring_want(long long rows, int k);

// One row into the pinned ring with streaming stores: the copy engine reads the chunk next, and lines left dirty in the packing
// core's cache would have to be snooped out one by one (measured: the H2D of chunks packed with plain memcpy ran at 14 GB/s).
inline void pack_row(double *dst, const double *src, size_t bytes)
{
    if ((((uintptr_t)dst | bytes) & 15u) == 0)
    {
        const char *s = reinterpret_cast<const char *>(src);
        char *d = reinterpret_cast<char *>(dst);
        for (size_t i = 0; i < bytes; i += 16)
            _mm_stream_si128(reinterpret_cast<__m128i *>(d + i), _mm_loadu_si128(reinterpret_cast<const __m128i *>(s + i)));
    }
    else
        std::memcpy(dst, src, bytes);
}

int rows_per_chunk(int k) { return (int)std::max<size_t>(1, CHUNK_BYTES / (sizeof(double) * (size_t)std::max(k, 1))); }
int ring_want(long long rows, int k)
{
    const long long chunks = (rows + rows_per_chunk(k) - 1) / rows_per_chunk(k);
    return 2 * (int)std::max<long long>(1, std::min<long long>({(long long)ring_workers(), (long long)pool().threads(), chunks}));
}

// Rows [r0, r1) of `src` (all k columns) -> the device image d (row r at d + r*k), enqueued on `s`. RING_WORKERS host threads
// each take every RING_WORKERS-th chunk: pack it into one of their two ring slots (serialize(), utils.cpp:216-228), hand it
// to the copy engine, go on packing the next while it travels.
int staged_upload(const Ring &ring, int device, const HostRows &src, double *d, int r0, int r1, int k, cudaStream_t s)
{
    if (r1 <= r0 || k <= 0)
        return SPMM_OK;
    const int rpc = rows_per_chunk(k), n_chunks = (r1 - r0 + rpc - 1) / rpc;
    const size_t width = sizeof(double) * (size_t)k;
    const int W = std::max(1, std::min({ring_workers(), pool().threads(), n_chunks, ring.n_slots / 2}));
    std::atomic<int> err{(int)cudaSuccess};
    static const bool timing = getenv("SPMM_HOST_TIMING") != nullptr;
    std::atomic<long long> ns_wait{0}, ns_pack{0}, ns_api{0}, ns_start{0};
    const auto t_begin = std::chrono::steady_clock::now();
    auto now_ns = [&] { return (long long)std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now() - t_begin).count(); };
    pool().parallel_for(W, [&](int w) {
        cudaError_t e = cudaSetDevice(device);
        if (timing)
            ns_start += now_ns();
        for (int i = 0, c = w; c < n_chunks && e == cudaSuccess; c += W, ++i)
        {
            const int c0 = r0 + c * rpc, c1 = std::min(r1, c0 + rpc), slot = 2 * w + (i & 1);
            const long long t0 = timing ? now_ns() : 0;
            if (i >= 2)
                e = cudaEventSynchronize(ring.event(0, slot)); // the chunk that used this slot has left the host
            const long long t1 = timing ? now_ns() : 0;
            double *stage = ring.slot(0, slot);
            for (int r = c0; r < c1; ++r)
                pack_row(stage + (size_t)(r - c0) * k, src.at(r), width);
            _mm_sfence(); // the streaming stores are globally visible before the copy engine is told to read them
            const long long t2 = timing ? now_ns() : 0;
            if (e == cudaSuccess)
                e = cudaMemcpyAsync(d + (size_t)c0 * k, stage, width * (size_t)(c1 - c0), cudaMemcpyHostToDevice, s);
            if (e == cudaSuccess)
                e = cudaEventRecord(ring.event(0, slot), s);
            if (timing)
            {
                ns_wait += t1 - t0;
                ns_pack += t2 - t1;
                ns_api += now_ns() - t2;
            }
        }
        if (e != cudaSuccess)
            err = (int)e;
    });
    if (timing)
        fprintf(stderr, "[spmm host] upload: %d chunks, %d workers; per worker: start %.3f ms, slot waits %.3f ms, packing %.3f ms, CUDA calls %.3f ms; all enqueued at %.3f ms\n",
                n_chunks, W, ns_start / 1e6 / W, ns_wait / 1e6 / W, ns_pack / 1e6 / W, ns_api / 1e6 / W, now_ns() / 1e6);
    SPMM_CUDA((cudaError_t)err.load());
    return SPMM_OK;
}

// n rows x k at d_c -> sink(row_begin, row_end, rows, ctx) chunk by chunk as they arrive (`rows` = row_begin's first double,
// leading dimension k); the sink runs on the host threads over disjoint row ranges (deserialize(), utils.cpp:237-253).
// Worker w owns chunks w, w+W, ...: its first two downloads are enqueued up front, each further one as soon as the slot it
// lands in has been handed to the sink.
typedef void (*RowsSink)(int, int, const double *, void *);
int staged_download(const Ring &ring, int device, const double *d_c, int n, int k, cudaStream_t s, RowsSink sink, void *ctx)
{
    if (n <= 0 || k <= 0)
        return SPMM_OK;
    const int rpc = rows_per_chunk(k), n_chunks = (n + rpc - 1) / rpc;
    const size_t width = sizeof(double) * (size_t)k;
    const int W = std::max(1, std::min({ring_workers(), pool().threads(), n_chunks, ring.n_slots / 2}));
    auto issue = [&](int c, int slot) -> cudaError_t {
        const int c0 = c * rpc, c1 = std::min(n, c0 + rpc);
        cudaError_t e = cudaMemcpyAsync(ring.slot(1, slot), d_c + (size_t)c0 * k, width * (size_t)(c1 - c0), cudaMemcpyDeviceToHost, s);
        return e == cudaSuccess ? cudaEventRecord(ring.event(1, slot), s) : e;
    };
    // in chunk order, so that the first chunks arrive first
    for (int c = 0; c < std::min(n_chunks, 2 * W); ++c)
        SPMM_CUDA(issue(c, 2 * (c % W) + ((c / W) & 1)));
    std::atomic<int> err{(int)cudaSuccess};
    pool().parallel_for(W, [&](int w) {
        cudaError_t e = cudaSetDevice(device);
        for (int i = 0, c = w; c < n_chunks && e == cudaSuccess; c += W, ++i)
        {
            const int c0 = c * rpc, c1 = std::min(n, c0 + rpc), slot = 2 * w + (i & 1);
            e = cudaEventSynchronize(ring.event(1, slot));
            if (e != cudaSuccess)
                break;
            sink(c0, c1, ring.slot(1, slot), ctx);
            if (c + 2 * W < n_chunks)
                e = issue(c + 2 * W, slot);
        }
        if (e != cudaSuccess)
            err = (int)e;
    });
    SPMM_CUDA((cudaError_t)err.load());
    return SPMM_OK;
}

struct CopySink
{
    HostRowsOut dst;
    int k;
};
void copy_sink(int r0, int r1, const double *rows, void *ctx)
{
    const CopySink &c = *static_cast<const CopySink *>(ctx);
    for (int r = r0; r < r1; ++r)
        std::memcpy(c.dst.at(r), rows + (size_t)(r - r0) * c.k, sizeof(double) * (size_t)c.k);
}

// The whole host-buffer call: rows [b0,b1) of B up (the other rows of the device image are not read by this launch),
// `launch(dB, dC, k0, kc, stream)`, c_rows rows of C down. Pinned flat buffers go to the copy engine as they are, wide ones
// in `slabs` k-slabs so that the upload of slab s+1 overlaps the download of slab s (PCIe is full duplex); everything else
// is staged through the ring in one pass (packing per slab would touch every source row once per slab: measured 3.3 ms with
// one slab against 4.3 / 5.2 ms with two / four on cfg2 k=64, gpurun_out/r2b_e2e.json).
template <typename Launch>
int host_multiply(spmm_csr_t A, const HostRows &B, int b0, int b1, int k, const HostRowsOut &C, RowsSink sink, void *sink_ctx,
                  int c_rows, int slabs, Launch launch)
{
    SPMM_CUDA(cudaSetDevice(A->device));
    std::lock_guard<std::mutex> guard(A->host_mu); // staging ring and streams of a handle serve one call at a time
    const size_t nb = (size_t)A->n_cols * (size_t)k, nc = (size_t)c_rows * (size_t)k;
    int rc = ensure_streams(A);
    if (!rc)
        rc = ensure_device(&A->d_B, &A->d_B_elems, nb);
    if (!rc)
        rc = ensure_device(&A->d_C, &A->d_C_elems, nc);
    const bool b_direct = !B.rows && is_pinned(B.flat), c_direct = !sink && !C.rows && is_pinned(C.flat);
    RingLease lease;
    if (!rc && !(b_direct && c_direct))
        rc = borrow_ring(A->device, ring_want(std::max<long long>(b1 - b0, c_rows), k), &lease.r);
    if (rc)
        return rc;
    if (!(b_direct && c_direct))
        slabs = 1;
    static const bool timing = getenv("SPMM_HOST_TIMING") != nullptr; // phase times of every call on stderr (diagnostics)
    const auto t_start = std::chrono::steady_clock::now();
    auto since = [&] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count(); };
    double t_up = 0, t_kernel = 0;
    while (slabs > 1 && (k % slabs != 0 || (k / slabs) % 2 != 0))
        --slabs;
    slabs = std::max(1, std::min(slabs, 8));
    const int ks = k / slabs;
    const size_t pitch = sizeof(double) * (size_t)k, width = sizeof(double) * (size_t)ks;
    for (int sidx = 0; sidx < slabs; ++sidx)
    {
        const int k0 = sidx * ks;
        cudaEvent_t up = A->events[2 * sidx], done = A->events[2 * sidx + 1];
        if (b_direct && b1 > b0)
        {
            const double *h = B.flat + (long long)b0 * B.ld + k0;
            if (slabs == 1 && B.ld == k)
                SPMM_CUDA(cudaMemcpyAsync(A->d_B + (size_t)b0 * k, h, pitch * (size_t)(b1 - b0), cudaMemcpyHostToDevice, A->stream_up));
            else
                SPMM_CUDA(cudaMemcpy2DAsync(A->d_B + (size_t)b0 * k + k0, pitch, h, sizeof(double) * (size_t)B.ld, width,
                                            (size_t)(b1 - b0), cudaMemcpyHostToDevice, A->stream_up));
        }
        else
        {
            rc = staged_upload(*lease.r, A->device, B, A->d_B, b0, b1, k, A->stream_up);
            if (rc)
                return rc;
        }
        SPMM_CUDA(cudaEventRecord(up, A->stream_up));
        SPMM_CUDA(cudaStreamWaitEvent(A->stream, up, 0));
        if (timing)
        {
            cudaStreamSynchronize(A->stream_up);
            t_up = since();
        }
        rc = launch(A->d_B, A->d_C, k0, ks, A->stream);
        if (rc)
            return rc;
        SPMM_CUDA(cudaEventRecord(done, A->stream));
        if (timing)
        {
            cudaStreamSynchronize(A->stream);
            t_kernel = since();
        }
        SPMM_CUDA(cudaStreamWaitEvent(A->stream_down, done, 0));
        if (c_direct)
        {
            if (slabs == 1 && C.ld == k)
                SPMM_CUDA(cudaMemcpyAsync(C.flat, A->d_C, pitch * (size_t)c_rows, cudaMemcpyDeviceToHost, A->stream_down));
            else
                SPMM_CUDA(cudaMemcpy2DAsync(C.flat + k0, sizeof(double) * (size_t)C.ld, A->d_C + k0, pitch, width, (size_t)c_rows,
                                            cudaMemcpyDeviceToHost, A->stream_down));
        }
        else
        {
            CopySink cs{C, k};
            rc = staged_download(*lease.r, A->device, A->d_C, c_rows, k, A->stream_down, sink ? sink : copy_sink, sink ? sink_ctx : &cs);
            if (rc)
                return rc;
        }
    }
    cudaError_t e = cudaStreamSynchronize(A->stream_down);
    if (e == cudaSuccess)
        e = cudaStreamSynchronize(A->stream);
    SPMM_CUDA(e);
    if (timing)
        fprintf(stderr, "[spmm host] upload done %.2f ms, kernel done %.2f ms, download done %.2f ms (last slab; %d slab%s, %s source, %s sink)\n",
                t_up, t_kernel, since(), slabs, slabs > 1 ? "s" : "", b_direct ? "pinned" : "staged", c_direct ? "pinned" : "staged");
    return rc;
}

int auto_slabs(size_t bytes, int k)
{
    int slabs = tuning().host_slabs;
    if (slabs <= 0)
        slabs = (bytes >= (16u << 20) && k >= 32) ? 2 : 1; // measured: 2.35 -> 1.90 ms at cfg2 k=64; 4 slabs of 128-byte rows copy slower
    return slabs;
}

// per-device scratch buffers (the root rank's C of a multi-rank strategy)
std::mutex g_scratch_mu;
std::map<std::pair<int, int>, std::pair<void *, size_t>> g_scratch;

} // namespace
} // namespace spmm

using namespace spmm;

extern "C"
{

int spmm_multiply_host(spmm_csr_t A, const double *B, int k, double *C, int kernel)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(k >= 0, "k is negative");
    const size_t nb = (size_t)A->n_cols * (size_t)k, nc = (size_t)A->n_rows * (size_t)k;
    if (nc == 0)
        return SPMM_OK;
    SPMM_REQUIRE(C != nullptr && (B != nullptr || nb == 0), "B/C is NULL");
    HostRows b;
    b.flat = B;
    b.ld = k;
    HostRowsOut c;
    c.flat = C;
    c.ld = k;
    return host_multiply(A, b, 0, A->n_cols, k, c, nullptr, nullptr, A->n_rows, auto_slabs((nb + nc) * sizeof(double), k),
                         [&](const double *dB, double *dC, int k0, int kc, cudaStream_t s) {
                             return spmm_multiply_strided_device(A, dB, k, dC, k, k0, kc, kernel, s);
                         });
}

int spmm_multiply_host_sink(spmm_csr_t A, const double *const *B_rows, int k, spmm_rows_sink sink, void *ctx, int kernel)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(k >= 0, "k is negative");
    const size_t nb = (size_t)A->n_cols * (size_t)k, nc = (size_t)A->n_rows * (size_t)k;
    if (nc == 0)
        return SPMM_OK;
    SPMM_REQUIRE(sink != nullptr && (B_rows != nullptr || nb == 0), "B_rows / sink is NULL");
    HostRows b;
    b.rows = B_rows;
    HostRowsOut none;
    return host_multiply(A, b, 0, A->n_cols, k, none, sink, ctx, A->n_rows, 1,
                         [&](const double *dB, double *dC, int k0, int kc, cudaStream_t s) {
                             return spmm_multiply_strided_device(A, dB, k, dC, k, k0, kc, kernel, s);
                         });
}

int spmm_multiply_host_rows(spmm_csr_t A, const double *const *B_rows, int k, double *const *C_rows, int kernel)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(k >= 0, "k is negative");
    const size_t nb = (size_t)A->n_cols * (size_t)k, nc = (size_t)A->n_rows * (size_t)k;
    if (nc == 0)
        return SPMM_OK;
    SPMM_REQUIRE(C_rows != nullptr && (B_rows != nullptr || nb == 0), "B_rows/C_rows is NULL");
    HostRows b;
    b.rows = B_rows;
    HostRowsOut c;
    c.rows = C_rows;
    return host_multiply(A, b, 0, A->n_cols, k, c, nullptr, nullptr, A->n_rows, 1,
                         [&](const double *dB, double *dC, int k0, int kc, cudaStream_t s) {
                             return spmm_multiply_strided_device(A, dB, k, dC, k, k0, kc, kernel, s);
                         });
}

int spmm_multiply_rows_host(spmm_csr_t A, int row_begin, int row_end, const double *B, int k, double *C_local,
                            int kernel)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(k >= 0, "k is negative");
    SPMM_REQUIRE(0 <= row_begin && row_begin <= row_end && row_end <= A->n_rows, "row range outside the matrix");
    const size_t nb = (size_t)A->n_cols * (size_t)k, nc = (size_t)(row_end - row_begin) * (size_t)k;
    if (nc == 0)
        return SPMM_OK;
    SPMM_REQUIRE(C_local != nullptr && (B != nullptr || nb == 0), "B/C is NULL");
    HostRows b;
    b.flat = B;
    b.ld = k;
    HostRowsOut c;
    c.flat = C_local;
    c.ld = k;
    return host_multiply(A, b, 0, A->n_cols, k, c, nullptr, nullptr, row_end - row_begin, 1,
                         [&](const double *dB, double *dC, int, int, cudaStream_t s) {
                             return spmm_multiply_rows_device(A, row_begin, row_end, dB, k, dC, kernel, s);
                         });
}

int spmm_multiply_nnz_range_host(spmm_csr_t A, long long nnz_begin, long long nnz_end, int first_row, int last_row,
                                 const double *B, int k, double *C_local, int kernel)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(k >= 0, "k is negative");
    if (last_row < first_row || k == 0 || nnz_begin == nnz_end)
        return SPMM_OK;
    SPMM_REQUIRE(C_local != nullptr && B != nullptr, "B/C is NULL");
    HostRows b;
    b.flat = B;
    b.ld = k;
    HostRowsOut c;
    c.flat = C_local;
    c.ld = k;
    return host_multiply(A, b, 0, A->n_cols, k, c, nullptr, nullptr, last_row - first_row + 1, 1,
                         [&](const double *dB, double *dC, int, int, cudaStream_t s) {
                             return spmm_multiply_nnz_range_device(A, nnz_begin, nnz_end, first_row, last_row, dB, k, dC,
                                                                   kernel, s);
                         });
}

// ---- pieces for strategies whose ranks share a process (one GPU per rank-thread) ----

int spmm_stage_b_rows(spmm_csr_t A, const double *const *B_rows, int row_begin, int row_end, int k, const double **d_B,
                      void **stream)
{
    SPMM_REQUIRE(A != nullptr && d_B != nullptr, "handle / output is NULL");
    SPMM_REQUIRE(k >= 0 && 0 <= row_begin && row_begin <= row_end && row_end <= A->n_cols, "row range outside B");
    SPMM_CUDA(cudaSetDevice(A->device));
    std::lock_guard<std::mutex> guard(A->host_mu);
    const size_t nb = (size_t)A->n_cols * (size_t)k;
    int rc = ensure_streams(A);
    if (!rc)
        rc = ensure_device(&A->d_B, &A->d_B_elems, nb);
    RingLease lease;
    if (!rc && row_end > row_begin)
        rc = borrow_ring(A->device, ring_want(row_end - row_begin, k), &lease.r);
    if (rc)
        return rc;
    SPMM_REQUIRE(B_rows != nullptr || row_end == row_begin, "B_rows is NULL");
    HostRows b;
    b.rows = B_rows;
    if (row_end > row_begin)
    {
        rc = staged_upload(*lease.r, A->device, b, A->d_B, row_begin, row_end, k, A->stream);
        if (rc)
            return rc;
        SPMM_CUDA(cudaStreamSynchronize(A->stream)); // the ring goes back to the free list: its chunks must have left the host
    }
    *d_B = A->d_B;
    if (stream)
        *stream = (void *)A->stream;
    return SPMM_OK;
}

int spmm_fetch_c_sink(spmm_csr_t A, const double *d_C, int n_rows, int k, spmm_rows_sink sink, void *ctx)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(n_rows >= 0 && k >= 0, "negative size");
    if (n_rows == 0 || k == 0)
        return SPMM_OK;
    SPMM_REQUIRE(d_C != nullptr && sink != nullptr, "d_C / sink is NULL");
    SPMM_CUDA(cudaSetDevice(A->device));
    std::lock_guard<std::mutex> guard(A->host_mu);
    RingLease lease;
    int rc = ensure_streams(A);
    if (!rc)
        rc = borrow_ring(A->device, ring_want(n_rows, k), &lease.r);
    if (rc)
        return rc;
    rc = staged_download(*lease.r, A->device, d_C, n_rows, k, A->stream_down, sink, ctx);
    SPMM_CUDA(cudaStreamSynchronize(A->stream_down));
    return rc;
}

int spmm_fetch_c_rows(spmm_csr_t A, const double *d_C, int n_rows, int k, double *const *C_rows)
{
    SPMM_REQUIRE(C_rows != nullptr || n_rows == 0 || k == 0, "C_rows is NULL");
    HostRowsOut c;
    c.rows = C_rows;
    CopySink cs{c, k};
    return spmm_fetch_c_sink(A, d_C, n_rows, k, copy_sink, &cs);
}

namespace
{
// spmm_upload_dense without the lock and the final wait (the caller holds A->host_mu); a staged upload has finished when it
// returns (its ring goes back to the free list)
int upload_block(spmm_csr_t A, const double *src, long long n_rows, int k, double *d_dst, cudaStream_t stream)
{
    if (is_pinned(src))
    {
        SPMM_CUDA(cudaMemcpyAsync(d_dst, src, sizeof(double) * (size_t)n_rows * (size_t)k, cudaMemcpyHostToDevice, stream));
        return SPMM_OK;
    }
    RingLease lease;
    int rc = borrow_ring(A->device, ring_want(n_rows, k), &lease.r);
    HostRows b;
    b.flat = src;
    b.ld = k;
    if (!rc)
        rc = staged_upload(*lease.r, A->device, b, d_dst, 0, (int)n_rows, k, stream);
    if (rc)
        return rc;
    SPMM_CUDA(cudaStreamSynchronize(stream)); // before the ring goes back to the free list
    return SPMM_OK;
}
} // namespace

int spmm_upload_dense(spmm_csr_t A, const double *src, long long n_rows, int k, double *d_dst, void *stream)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(n_rows >= 0 && k >= 0 && n_rows <= 2147483647LL, "bad size");
    if (n_rows == 0 || k == 0)
        return SPMM_OK;
    SPMM_REQUIRE(src != nullptr && d_dst != nullptr, "src / d_dst is NULL");
    SPMM_CUDA(cudaSetDevice(A->device));
    std::lock_guard<std::mutex> guard(A->host_mu);
    const int rc = upload_block(A, src, n_rows, k, d_dst, (cudaStream_t)stream);
    if (rc)
        return rc;
    SPMM_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return SPMM_OK;
}

int spmm_csr_update_values_host(spmm_csr_t A, const double *vals)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(A->owns, "a borrowed handle reads the caller's device array: edit it and call spmm_csr_update_values_device");
    if (A->nnz == 0)
        return SPMM_OK;
    SPMM_REQUIRE(vals != nullptr, "vals is NULL");
    SPMM_CUDA(cudaSetDevice(A->device));
    std::lock_guard<std::mutex> guard(A->host_mu);
    int rc = ensure_streams(A);
    // Straight into the handle's value array; a pageable source is staged as rows of 4 KB (the ring packs row by row) and
    // the last nnz % 512 values as one short row. Then the tile layout is refreshed from that array.
    constexpr int W = 512;
    const long long full = A->nnz / W, rest = A->nnz % W;
    if (!rc && full)
        rc = upload_block(A, vals, full, W, A->d_vals, A->stream);
    if (!rc && rest)
        rc = upload_block(A, vals + full * W, 1, (int)rest, A->d_vals + full * W, A->stream);
    if (!rc)
        rc = update_values(A, A->d_vals, A->stream);
    const cudaError_t e = cudaStreamSynchronize(A->stream);
    if (!rc)
        SPMM_CUDA(e);
    return rc;
}

int spmm_download_dense(spmm_csr_t A, const double *d_src, long long n_rows, int k, double *dst, void *stream)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_REQUIRE(n_rows >= 0 && k >= 0 && n_rows <= 2147483647LL, "bad size");
    if (n_rows == 0 || k == 0)
        return SPMM_OK;
    SPMM_REQUIRE(d_src != nullptr && dst != nullptr, "d_src / dst is NULL");
    SPMM_CUDA(cudaSetDevice(A->device));
    std::lock_guard<std::mutex> guard(A->host_mu);
    int rc = SPMM_OK;
    if (is_pinned(dst))
        SPMM_CUDA(cudaMemcpyAsync(dst, d_src, sizeof(double) * (size_t)n_rows * (size_t)k, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    else
    {
        RingLease lease;
        rc = borrow_ring(A->device, ring_want(n_rows, k), &lease.r);
        HostRowsOut c;
        c.flat = dst;
        c.ld = k;
        CopySink cs{c, k};
        if (!rc)
            rc = staged_download(*lease.r, A->device, d_src, (int)n_rows, k, (cudaStream_t)stream, copy_sink, &cs);
        const cudaError_t e = cudaStreamSynchronize((cudaStream_t)stream);
        if (!rc)
            SPMM_CUDA(e);
        return rc;
    }
    SPMM_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return rc;
}

int spmm_csr_stream_sync(spmm_csr_t A)
{
    SPMM_REQUIRE(A != nullptr, "handle is NULL");
    SPMM_CUDA(cudaSetDevice(A->device));
    if (A->stream)
        SPMM_CUDA(cudaStreamSynchronize(A->stream));
    return SPMM_OK;
}

int spmm_device_scratch(int device, int slot, long long bytes, void **out)
{
    SPMM_REQUIRE(out != nullptr && bytes >= 0 && slot >= 0, "bad scratch request");
    SPMM_CUDA(cudaSetDevice(device));
    std::lock_guard<std::mutex> lk(g_scratch_mu);
    auto &e = g_scratch[{device, slot}];
    if (e.second < (size_t)bytes)
    {
        cudaFree(e.first);
        e = {nullptr, 0};
        SPMM_CUDA(cudaMalloc(&e.first, std::max<size_t>((size_t)bytes, 16)));
        e.second = (size_t)bytes;
    }
    *out = e.first;
    return SPMM_OK;
}

int spmm_device_scratch_release(void)
{
    std::lock_guard<std::mutex> lk(g_scratch_mu);
    for (auto &kv : g_scratch)
    {
        cudaSetDevice(kv.first.first);
        cudaFree(kv.second.first);
    }
    g_scratch.clear();
    return SPMM_OK;
}

int spmm_peer_enable(int device, int peer)
{
    if (device == peer)
        return SPMM_OK;
    SPMM_CUDA(cudaSetDevice(device));
    int can = 0;
    SPMM_CUDA(cudaDeviceCanAccessPeer(&can, device, peer));
    if (!can)
    {
        set_error("device " + std::to_string(device) + " cannot access device " + std::to_string(peer) + " (no NVLink/PCIe peer path)");
        return SPMM_ERR_UNSUPPORTED;
    }
    const cudaError_t e = cudaDeviceEnablePeerAccess(peer, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled)
    {
        cudaGetLastError();
        return SPMM_OK;
    }
    SPMM_CUDA(e);
    return SPMM_OK;
}

namespace
{
bool warmup_wanted()
{
    const char *e = getenv("SPMM_NO_WARMUP");
    return !(e && *e == '1');
}
// one tiny multiply per kernel module on device d (see spmm_devices_init)
void warm_up_modules(int d)
{
    const int rp[3] = {0, 1, 2}, ci[2] = {0, 1};
    const double v[2] = {1.0, 1.0};
    spmm_csr_t A = nullptr;
    double *buf = nullptr;
    if (cudaSetDevice(d) != cudaSuccess || spmm_csr_create_host(d, 2, 2, 2, rp, ci, v, &A) != SPMM_OK)
        return;
    if (cudaMalloc((void **)&buf, sizeof(double) * 16) == cudaSuccess && cudaMemset(buf, 0, sizeof(double) * 16) == cudaSuccess)
    {
        int lo = 0, hi = 0;
        spmm_multiply_device(A, buf, 2, buf + 8, SPMM_KERNEL_ROWS, nullptr);  // even k: 16-byte accesses
        spmm_multiply_device(A, buf, 1, buf + 8, SPMM_KERNEL_ROWS, nullptr);  // odd k: 8-byte accesses
        spmm_multiply_device(A, buf, 2, buf + 8, SPMM_KERNEL_MERGE, nullptr);
        spmm_csr_column_span(A, &lo, &hi);                                     // the CSR build / shard unit
        spmm_csr_build_tiles(A, 8, 0);                                         // the tile-layout / tiled-kernel unit
        spmm_multiply_device(A, buf, 2, buf + 8, SPMM_KERNEL_AUTO, nullptr);
        cudaDeviceSynchronize();
    }
    cudaFree(buf);
    spmm_csr_destroy(A);
    cudaGetLastError();
}
} // namespace

int spmm_devices_init(int enable_peers)
{
    int count = 0;
    SPMM_CUDA(cudaGetDeviceCount(&count));
    for (int d = 0; d < count; ++d)
    {
        SPMM_CUDA(cudaSetDevice(d));
        SPMM_CUDA(cudaFree(nullptr)); // creates the primary context
    }
    for (int d = 0; enable_peers && d < count; ++d)
        for (int p = 0; p < count; ++p)
        {
            int can = 0;
            if (p == d || cudaDeviceCanAccessPeer(&can, d, p) != cudaSuccess || !can)
                continue;
            cudaSetDevice(d);
            const cudaError_t e = cudaDeviceEnablePeerAccess(p, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                return cuda_fail(e, "cudaDeviceEnablePeerAccess", __FILE__, __LINE__);
            cudaGetLastError();
        }
    if (count)
    {
        SPMM_CUDA(cudaSetDevice(0));
        const int rc = arena_init(); // page-locked staging arena, shared by the rank-threads of the process
        if (rc)
            return rc;
    }
    pool(); // host threads
    // CUDA loads a module when one of its kernels is first launched: 38 ms for the translation unit that holds the row and
    // merge kernels (measured: tools/first_launch_probe.py, first multiply of a process 38.1 ms, with any earlier launch from
    // the same unit 0.2 ms). A caller that times each function once (the reference's main.cpp:77-79) would pay that inside
    // its first call on every GPU; one tiny multiply per device and module here pays it at program start instead.
    if (warmup_wanted())
    {
        std::vector<std::thread> th;
        for (int d = 0; d < count; ++d)
            th.emplace_back([d] { warm_up_modules(d); });
        for (auto &t : th)
            t.join();
        SPMM_CUDA(cudaSetDevice(0));
    }
    return SPMM_OK;
}

int spmm_device_init(int device)
{
    int count = 0;
    SPMM_CUDA(cudaGetDeviceCount(&count));
    SPMM_REQUIRE(device >= 0 && device < count, "no such device");
    SPMM_CUDA(cudaSetDevice(device));
    SPMM_CUDA(cudaFree(nullptr)); // creates the primary context
    const int rc = arena_init();
    if (rc)
        return rc;
    pool();
    if (warmup_wanted())
        warm_up_modules(device);
    return SPMM_OK;
}

int spmm_host_threads(void) { return pool().threads(); }

void spmm_host_parallel_for(int n, void (*fn)(int, void *), void *ctx)
{
    if (fn)
        pool().parallel_for(n, [&](int i) { fn(i, ctx); });
}

} // extern "C"
