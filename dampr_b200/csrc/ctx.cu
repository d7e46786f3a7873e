// ctx.cu — context, streams, timings, pinned memory, text buffers and kv containers.
// Replaces the process pool / Queue plumbing of StageRunner.run (reference stagerunner.py:15-43)
// and the on-disk run files of dataset.py with device-resident buffers.
#include <cufile.h>
#include <dlfcn.h>
#include <fcntl.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <memory>
#include <mutex>
#include <thread>

#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#include "common.cuh"

int g_text_kernel = 2;
thread_local dampr_ctx *tl_ctx = nullptr;

static const size_t POOL_MAX_CACHED = 6ULL << 30;

void *pool_alloc(dampr_ctx *ctx, size_t bytes) {
    bytes = (bytes + 255) & ~(size_t)255;
    int best = -1;
    for (int i = 0; i < (int)ctx->pool_free_list.size(); ++i) {
        const PoolBlock &b = ctx->pool_free_list[i];
        if (b.bytes >= bytes && b.bytes <= 2 * bytes + (1 << 20) &&
            (best < 0 || b.bytes < ctx->pool_free_list[best].bytes))
            best = i;
    }
    if (best >= 0) {
        PoolBlock b = ctx->pool_free_list[best];
        ctx->pool_free_list.erase(ctx->pool_free_list.begin() + best);
        ctx->pool_cached_bytes -= b.bytes;
        // the previous user's work must be complete before anybody (either stream) touches it again
        cudaEventSynchronize(b.ev_compute);
        cudaEventSynchronize(b.ev_copy);
        cudaEventDestroy(b.ev_compute);
        cudaEventDestroy(b.ev_copy);
        ctx->pool_live[b.p] = b.bytes;
        return b.p;
    }
    void *p = nullptr;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        pool_trim(ctx, 0);
        e = cudaMalloc(&p, bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
    }
    ctx->pool_live[p] = bytes;
    return p;
}

void *host_pin(dampr_ctx *ctx, int which, size_t bytes) {
    if (ctx->h_pin_busy[which]) {
        cudaEventSynchronize(ctx->h_pin_ev[which]);
        ctx->h_pin_busy[which] = false;
    }
    if (ctx->h_pin_bytes[which] < bytes) {
        if (ctx->h_pin[which]) {
            cudaFreeHost(ctx->h_pin[which]);
            ctx->h_pin[which] = nullptr;
            ctx->h_pin_bytes[which] = 0;
        }
        size_t cap = std::max<size_t>(bytes + bytes / 4, 1 << 20);
        if (cudaMallocHost(&ctx->h_pin[which], cap) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        ctx->h_pin_bytes[which] = cap;
    }
    return ctx->h_pin[which];
}

void host_pin_used(dampr_ctx *ctx, int which) {
    if (!ctx->h_pin_ev[which] &&
        cudaEventCreateWithFlags(&ctx->h_pin_ev[which], cudaEventDisableTiming) != cudaSuccess) {
        cudaGetLastError();
        cudaStreamSynchronize(ctx->stream);  // no event: fall back to a full wait
        return;
    }
    cudaEventRecord(ctx->h_pin_ev[which], ctx->stream);
    ctx->h_pin_busy[which] = true;
}

void pool_free(dampr_ctx *ctx, void *p) {
    if (!p) return;
    auto it = ctx->pool_live.find(p);
    if (it == ctx->pool_live.end()) {
        cudaFree(p);
        return;
    }
    PoolBlock b;
    b.p = p;
    b.bytes = it->second;
    ctx->pool_live.erase(it);
    if (b.bytes > (2ULL << 30) ||
        cudaEventCreateWithFlags(&b.ev_compute, cudaEventDisableTiming) != cudaSuccess) {
        cudaFree(p);
        return;
    }
    if (cudaEventCreateWithFlags(&b.ev_copy, cudaEventDisableTiming) != cudaSuccess) {
        cudaEventDestroy(b.ev_compute);
        cudaFree(p);
        return;
    }
    cudaEventRecord(b.ev_compute, ctx->stream);
    cudaEventRecord(b.ev_copy, ctx->copy);
    ctx->pool_free_list.push_back(b);
    ctx->pool_cached_bytes += b.bytes;
    if (ctx->pool_cached_bytes > POOL_MAX_CACHED || ctx->pool_free_list.size() > 256) pool_trim(ctx, POOL_MAX_CACHED / 2);
}

void pool_trim(dampr_ctx *ctx, size_t keep_bytes) {
    while (!ctx->pool_free_list.empty() && (ctx->pool_cached_bytes > keep_bytes || ctx->pool_free_list.size() > 128)) {
        PoolBlock b = ctx->pool_free_list.front();
        ctx->pool_free_list.erase(ctx->pool_free_list.begin());
        ctx->pool_cached_bytes -= b.bytes;
        cudaEventDestroy(b.ev_compute);
        cudaEventDestroy(b.ev_copy);
        cudaFree(b.p);  // synchronises: safe regardless of the events
    }
}
int g_text_ctas = 4;
int g_file_cufile = 0;         // 1: file ingest through cuFile (GPUDirect Storage) instead of the page-locked ring
int g_cufile_threads = 8;
int g_host_threads_cap = 16;   // copy threads per staged transfer (dampr_set_option "host_threads")

// ---- staged transfers ---------------------------------------------------------------------------
namespace {

// Process-wide pool of copy threads (created on first use, parked on a condition variable).  One
// memcpy job at a time; the caller takes part in it.  A job is its own heap object, so a worker that
// wakes up late only ever sees a finished job (nothing left to claim), never a half-initialised one.
class CopyPool {
    static constexpr size_t PIECE = 1u << 20;
    struct Job {
        char *dst;
        const char *src;   // memory source, or nullptr: read from fd at file offset foff
        const char *src2 = nullptr;  // interleave mode: dst records = (src u64[i], src2 u64[i]); n = bytes of dst
        bool interleave = false;
        int fd = -1;
        size_t foff = 0;
        size_t n, pieces;
        std::atomic<size_t> next{0}, left{0};
        std::atomic<int> failed{0};
    };

  public:
    // two pools: uploads (0) and downloads (1) may run at the same time (spill.py overlaps them), each with its
    // own threads, so the host copies of the two PCIe directions do not queue behind each other
    static CopyPool &get(int which = 0) {
        static CopyPool p[2];
        return p[which & 1];
    }
    // returns false if a read from the file came up short
    bool run(void *dst, const void *src, size_t n, int threads, int fd = -1, size_t foff = 0, const void *src2 = nullptr,
             bool interleave = false) {
        if (src && !interleave && (threads <= 1 || n < 4 * PIECE)) {
            memcpy(dst, src, n);
            return true;
        }
        std::lock_guard<std::mutex> job_lock(job_mu_);
        auto job = std::make_shared<Job>();
        job->dst = (char *)dst;
        job->src = (const char *)src;
        job->src2 = (const char *)src2;
        job->interleave = interleave;
        job->fd = fd;
        job->foff = foff;
        job->n = n;
        job->pieces = (n + PIECE - 1) / PIECE;
        job->left.store(job->pieces);
        {
            std::lock_guard<std::mutex> lk(mu_);
            while ((int)workers_.size() < threads - 1) workers_.emplace_back([this] { loop(); });
            cur_ = job;
            ++gen_;
        }
        cv_.notify_all();
        work(*job);
        std::unique_lock<std::mutex> lk(mu_);
        done_cv_.wait(lk, [&] { return job->left.load() == 0; });
        return job->failed.load() == 0;
    }

  private:
    CopyPool() {}
    ~CopyPool() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto &t : workers_) t.join();
    }
    void work(Job &j) {
        for (;;) {
            const size_t i = j.next.fetch_add(1);
            if (i >= j.pieces) break;
            const size_t lo = i * PIECE, len = std::min(PIECE, j.n - lo);
            if (j.interleave) {
                // PIECE is a multiple of 16: records [lo / 16, (lo + len) / 16)
                u64 *__restrict d = reinterpret_cast<u64 *>(j.dst + lo);
                const u64 *__restrict k = reinterpret_cast<const u64 *>(j.src) + lo / 16;
                const size_t cnt = len / 16;
                if (j.src2) {
                    const u64 *__restrict v = reinterpret_cast<const u64 *>(j.src2) + lo / 16;
                    size_t i = 0;
#if defined(__SSE2__)
                    // two records per step; streaming stores: the slot is written once and read by the DMA engine,
                    // so no read-for-ownership of the destination lines (32 instead of 48 bytes of memory traffic
                    // per record). The slots are 4 KB aligned, the columns 8-byte aligned.
                    for (; i + 2 <= cnt; i += 2) {
                        const __m128i kk = _mm_loadu_si128(reinterpret_cast<const __m128i *>(k + i));
                        const __m128i vv = _mm_loadu_si128(reinterpret_cast<const __m128i *>(v + i));
                        _mm_stream_si128(reinterpret_cast<__m128i *>(d + 2 * i), _mm_unpacklo_epi64(kk, vv));
                        _mm_stream_si128(reinterpret_cast<__m128i *>(d + 2 * i + 2), _mm_unpackhi_epi64(kk, vv));
                    }
                    _mm_sfence();
#endif
                    for (; i < cnt; ++i) {
                        d[2 * i] = k[i];
                        d[2 * i + 1] = v[i];
                    }
                } else {
                    for (size_t i = 0; i < cnt; ++i) {
                        d[2 * i] = k[i];
                        d[2 * i + 1] = 0;
                    }
                }
            } else if (j.src) {
                memcpy(j.dst + lo, j.src + lo, len);
            } else {
                size_t got = 0;
                while (got < len) {
                    const ssize_t r = pread(j.fd, j.dst + lo + got, len - got, (off_t)(j.foff + lo + got));
                    if (r <= 0) {
                        j.failed.store(1);
                        break;
                    }
                    got += (size_t)r;
                }
            }
            if (j.left.fetch_sub(1) == 1) {
                std::lock_guard<std::mutex> lk(mu_);
                done_cv_.notify_all();
            }
        }
    }
    void loop() {
        u64 seen = 0;
        for (;;) {
            std::shared_ptr<Job> job;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return stop_ || gen_ != seen; });
                if (stop_) return;
                seen = gen_;
                job = cur_;
            }
            work(*job);
        }
    }
    std::mutex job_mu_, mu_;
    std::condition_variable cv_, done_cv_;
    std::vector<std::thread> workers_;
    std::shared_ptr<Job> cur_;
    u64 gen_ = 0;
    bool stop_ = false;
};

void par_memcpy(void *dst, const void *src, size_t n, int threads, int pool = 0) { CopyPool::get(pool).run(dst, src, n, threads); }
void par_interleave(void *dst_records, const void *keys, const void *vals, size_t count, int threads) {
    CopyPool::get().run(dst_records, keys, count * 16, std::max(threads, 1), -1, 0, vals, true);
}
bool par_pread(void *dst, int fd, size_t foff, size_t n, int threads) {
    return CopyPool::get().run(dst, nullptr, n, std::max(threads, 1), fd, foff);
}

bool is_pinned(const void *p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return a.type == cudaMemoryTypeHost || a.type == cudaMemoryTypeManaged;
}

int stage_init(dampr_ctx *ctx) {
    static std::mutex init_mu;   // (an uploading thread and the main thread may both arrive here first)
    std::lock_guard<std::mutex> lk(init_mu);
    if (ctx->dstage_ev[dampr_ctx::STAGE_SLOTS - 1]) return DAMPR_OK;
    for (int i = 0; i < dampr_ctx::STAGE_SLOTS; ++i) {
        if (ctx->stage_slot[i]) continue;
        CUDA_TRY(ctx, cudaHostAlloc(&ctx->stage_slot[i], dampr_ctx::STAGE_BYTES, cudaHostAllocDefault));
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->stage_ev[i], cudaEventDisableTiming));
        // downloads have a ring of their own: an upload (another host thread, the copy stream) and a download
        // (the compute stream) may be in flight together (spill.py overlaps the next batch's upload)
        CUDA_TRY(ctx, cudaHostAlloc(&ctx->dstage_slot[i], dampr_ctx::STAGE_BYTES, cudaHostAllocDefault));
        CUDA_TRY(ctx, cudaEventCreateWithFlags(&ctx->dstage_ev[i], cudaEventDisableTiming));
    }
    return DAMPR_OK;
}

// copy threads per staged transfer: a quarter of the hardware threads, at most the "host_threads" option
int copy_threads() {
    static const unsigned hw = std::max(4u, std::thread::hardware_concurrency());
    return (int)std::max(2u, std::min((unsigned)g_host_threads_cap, hw / 4));
}

}  // namespace

bool host_is_pinned(const void *p) { return is_pinned(p); }

int staged_h2d(dampr_ctx *ctx, void *dst, const void *src, size_t bytes, cudaStream_t st) {
    if (bytes == 0) return DAMPR_OK;
    if (bytes < (8u << 20) || is_pinned(src)) {
        // (a range that straddles two separately page-locked regions, or the end of one, is refused with
        // cudaErrorInvalidValue at enqueue time: such a copy goes through the ring like pageable memory)
        const cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) return DAMPR_OK;
        if (e != cudaErrorInvalidValue) CUDA_TRY(ctx, e);
        cudaGetLastError();
    }
    int rc = stage_init(ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> ring(ctx->stage_mu);
    const size_t B = dampr_ctx::STAGE_BYTES;
    for (size_t off = 0; off < bytes; off += B) {
        // the ring position carries over from call to call: a caller that uploads slot-sized chunks one call at
        // a time still fills the next slot while the previous one is on the wire
        const int slot = (int)(ctx->stage_next++ % dampr_ctx::STAGE_SLOTS);
        const size_t len = std::min(B, bytes - off);
        CUDA_TRY(ctx, cudaEventSynchronize(ctx->stage_ev[slot]));  // the DMA that last read this slot
        par_memcpy(ctx->stage_slot[slot], (const char *)src + off, len, copy_threads());
        CUDA_TRY(ctx, cudaMemcpyAsync((char *)dst + off, ctx->stage_slot[slot], len, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaEventRecord(ctx->stage_ev[slot], st));
    }
    return DAMPR_OK;
}

// (keys[i], vals[i]) columns in pageable host memory -> 16-byte records on the device: the copy threads interleave
// the two columns while they fill the page-locked ring (the same memory traffic as the plain staging copy), so no
// device staging block and no interleave kernel are needed
int staged_h2d_columns(dampr_ctx *ctx, void *dst_records, const u64 *keys, const u64 *vals, size_t count, cudaStream_t st) {
    if (count == 0) return DAMPR_OK;
    int rc = stage_init(ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> ring(ctx->stage_mu);
    const size_t R = dampr_ctx::STAGE_BYTES / 16;   // records per slot
    for (size_t off = 0; off < count; off += R) {
        const int slot = (int)(ctx->stage_next++ % dampr_ctx::STAGE_SLOTS);
        const size_t len = std::min(R, count - off);
        CUDA_TRY(ctx, cudaEventSynchronize(ctx->stage_ev[slot]));
        par_interleave(ctx->stage_slot[slot], keys + off, vals ? vals + off : nullptr, len, copy_threads());
        CUDA_TRY(ctx, cudaMemcpyAsync((char *)dst_records + off * 16, ctx->stage_slot[slot], len * 16, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaEventRecord(ctx->stage_ev[slot], st));
    }
    return DAMPR_OK;
}

// file (page cache) -> device: the copy threads pread() 1 MB pieces straight into the page-locked ring, the DMA of
// a slot overlaps the reads into the next ones
int staged_file_h2d(dampr_ctx *ctx, void *dst, int fd, size_t foff, size_t bytes, cudaStream_t st) {
    if (bytes == 0) return DAMPR_OK;
    int rc = stage_init(ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> ring(ctx->stage_mu);
    const size_t B = dampr_ctx::STAGE_BYTES;
    for (size_t off = 0; off < bytes; off += B) {
        const int slot = (int)(ctx->stage_next++ % dampr_ctx::STAGE_SLOTS);
        const size_t len = std::min(B, bytes - off);
        CUDA_TRY(ctx, cudaEventSynchronize(ctx->stage_ev[slot]));  // the DMA that last read this slot
        if (!par_pread(ctx->stage_slot[slot], fd, foff + off, len, copy_threads()))
            return set_err(ctx, DAMPR_ERR_ARG, "%s", "short read from the input file");
        CUDA_TRY(ctx, cudaMemcpyAsync((char *)dst + off, ctx->stage_slot[slot], len, cudaMemcpyHostToDevice, st));
        CUDA_TRY(ctx, cudaEventRecord(ctx->stage_ev[slot], st));
    }
    return DAMPR_OK;
}

int staged_d2h(dampr_ctx *ctx, void *dst, const void *src, size_t bytes, cudaStream_t st) {
    if (bytes == 0) return DAMPR_OK;
    if (bytes < (8u << 20) || is_pinned(dst)) {
        const cudaError_t e = cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st);
        if (e == cudaSuccess) {
            CUDA_TRY(ctx, cudaStreamSynchronize(st));
            return DAMPR_OK;
        }
        if (e != cudaErrorInvalidValue) CUDA_TRY(ctx, e);
        cudaGetLastError();   // straddles page-locked regions: through the ring
    }
    int rc = stage_init(ctx);
    if (rc) return rc;
    std::lock_guard<std::mutex> ring(ctx->dstage_mu);
    const size_t B = dampr_ctx::STAGE_BYTES;
    const size_t nchunks = (bytes + B - 1) / B;
    const size_t S = dampr_ctx::STAGE_SLOTS;
    // (the download ring is only ever used by this function, which drains every slot before it returns)
    for (size_t i = 0; i < nchunks + S - 1; ++i) {
        if (i >= S - 1) {  // drain chunk i-(S-1) before its slot is refilled by chunk i+1
            const size_t j = i - (S - 1);
            const size_t off = j * B, len = std::min(B, bytes - off);
            CUDA_TRY(ctx, cudaEventSynchronize(ctx->dstage_ev[j % S]));
            par_memcpy((char *)dst + off, ctx->dstage_slot[j % S], len, copy_threads(), 1);
        }
        if (i < nchunks) {
            const size_t off = i * B, len = std::min(B, bytes - off);
            CUDA_TRY(ctx, cudaMemcpyAsync(ctx->dstage_slot[i % S], (const char *)src + off, len, cudaMemcpyDeviceToHost, st));
            CUDA_TRY(ctx, cudaEventRecord(ctx->dstage_ev[i % S], st));
        }
    }
    return DAMPR_OK;
}

extern "C" {

int32_t dampr_abi_version(void) { return 1; }

int32_t dampr_device_count(int32_t *out_n) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *out_n = 0;
        return DAMPR_ERR_CUDA;
    }
    *out_n = n;
    return DAMPR_OK;
}

int32_t dampr_ctx_create(int32_t device, dampr_ctx **out) {
    if (!out) return DAMPR_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) return DAMPR_ERR_CUDA;
    if (device < 0 || device >= n) return DAMPR_ERR_ARG;
    if (cudaSetDevice(device) != cudaSuccess) return DAMPR_ERR_CUDA;
    dampr_ctx *c = new dampr_ctx();
    c->device = device;
    c->launches = 0;
    c->timing_enabled = true;
    c->upload_pending = false;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) {
        delete c;
        return DAMPR_ERR_CUDA;
    }
    c->num_sms = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&c->copy, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->upload_done, cudaEventDisableTiming) != cudaSuccess ||
        cudaMalloc(&c->d_scratch, 4096 * sizeof(u64)) != cudaSuccess ||
        cudaMallocHost(&c->h_scratch, 4096 * sizeof(u64)) != cudaSuccess) {
        delete c;
        return DAMPR_ERR_CUDA;
    }
    *out = c;
    return DAMPR_OK;
}

int32_t dampr_ctx_destroy(dampr_ctx *ctx) {
    if (!ctx) return DAMPR_ERR_ARG;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaStreamSynchronize(ctx->copy);
    for (auto &t : ctx->timings) {
        cudaEventDestroy(t.beg);
        cudaEventDestroy(t.end);
    }
    pool_trim(ctx, 0);
    for (auto &kv : ctx->pool_live) cudaFree(kv.first);
    ctx->pool_live.clear();
    cudaEventDestroy(ctx->upload_done);
    cudaFree(ctx->d_scratch);
    cudaFreeHost(ctx->h_scratch);
    for (int i = 0; i < 2; ++i) {
        if (ctx->h_pin[i]) cudaFreeHost(ctx->h_pin[i]);
        if (ctx->h_pin_ev[i]) cudaEventDestroy(ctx->h_pin_ev[i]);
        if (ctx->up_tmp[i]) cudaFree(ctx->up_tmp[i]);
        if (ctx->up_tmp_ev[i]) cudaEventDestroy(ctx->up_tmp_ev[i]);
    }
    for (int i = 0; i < dampr_ctx::STAGE_SLOTS; ++i) {
        if (ctx->stage_slot[i]) cudaFreeHost(ctx->stage_slot[i]);
        if (ctx->stage_ev[i]) cudaEventDestroy(ctx->stage_ev[i]);
        if (ctx->dstage_slot[i]) cudaFreeHost(ctx->dstage_slot[i]);
        if (ctx->dstage_ev[i]) cudaEventDestroy(ctx->dstage_ev[i]);
    }
    cudaStreamDestroy(ctx->stream);
    cudaStreamDestroy(ctx->copy);
    delete ctx;
    return DAMPR_OK;
}

int32_t dampr_ctx_sync(dampr_ctx *ctx) {
    if (!ctx) return DAMPR_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return DAMPR_OK;
}

int32_t dampr_ctx_sync_copy(dampr_ctx *ctx) {
    if (!ctx) return DAMPR_ERR_ARG;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy));
    return DAMPR_OK;
}

const char *dampr_last_error(dampr_ctx *ctx) { return ctx ? ctx->err.c_str() : "no context"; }

int32_t dampr_ctx_timings(dampr_ctx *ctx, double *out_ms, int32_t *out_ids, int32_t cap,
                          int32_t *n) {
    if (!ctx || !n) return DAMPR_ERR_ARG;
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    int k = 0;
    for (auto &t : ctx->timings) {
        if (k >= cap) break;
        float ms = 0.f;
        CUDA_TRY(ctx, cudaEventElapsedTime(&ms, t.beg, t.end));
        out_ms[k] = (double)ms;
        out_ids[k] = t.id;
        k++;
    }
    *n = k;
    return DAMPR_OK;
}

int32_t dampr_ctx_timings_reset(dampr_ctx *ctx) {
    if (!ctx) return DAMPR_ERR_ARG;
    cudaStreamSynchronize(ctx->stream);
    for (auto &t : ctx->timings) {
        cudaEventDestroy(t.beg);
        cudaEventDestroy(t.end);
    }
    ctx->timings.clear();
    return DAMPR_OK;
}

int32_t dampr_ctx_timing_enable(dampr_ctx *ctx, int32_t on) {
    if (!ctx) return DAMPR_ERR_ARG;
    ctx->timing_enabled = on != 0;
    return DAMPR_OK;
}

int32_t dampr_ctx_launches(dampr_ctx *ctx, uint64_t *out) {
    if (!ctx || !out) return DAMPR_ERR_ARG;
    *out = ctx->launches;
    return DAMPR_OK;
}

int32_t dampr_ctx_stream(dampr_ctx *ctx, uint64_t *out_stream) {
    if (!ctx || !out_stream) return DAMPR_ERR_ARG;
    *out_stream = (uint64_t)(uintptr_t)ctx->stream;
    return DAMPR_OK;
}

int32_t dampr_ctx_mem_info(dampr_ctx *ctx, uint64_t *free_bytes, uint64_t *total_bytes) {
    if (!ctx || !free_bytes || !total_bytes) return DAMPR_ERR_ARG;
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    size_t f = 0, t = 0;
    CUDA_TRY(ctx, cudaMemGetInfo(&f, &t));
    *free_bytes = f;
    *total_bytes = t;
    return DAMPR_OK;
}

int32_t dampr_ctx_num_sms(dampr_ctx *ctx, int32_t *out) {
    if (!ctx || !out) return DAMPR_ERR_ARG;
    *out = ctx->num_sms;
    return DAMPR_OK;
}

int32_t dampr_host_alloc(uint64_t nbytes, void **out) {
    if (!out) return DAMPR_ERR_ARG;
    *out = nullptr;
    cudaError_t e = cudaMallocHost(out, nbytes ? nbytes : 1);
    return e == cudaSuccess ? DAMPR_OK : DAMPR_ERR_NOMEM;
}

int32_t dampr_host_free(void *p) {
    if (!p) return DAMPR_OK;
    return cudaFreeHost(p) == cudaSuccess ? DAMPR_OK : DAMPR_ERR_CUDA;
}

// Page-lock memory the caller owns (the spill run buffer, spill.py): transfers from / to it then go straight over
// PCIe instead of through the staging ring and the copy threads.
int32_t dampr_host_register(void *p, uint64_t nbytes) {
    if (!p || !nbytes) return DAMPR_ERR_ARG;
    cudaError_t e = cudaHostRegister(p, nbytes, cudaHostRegisterDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return e == cudaErrorMemoryAllocation ? DAMPR_ERR_NOMEM : DAMPR_ERR_CUDA;
    }
    return DAMPR_OK;
}

int32_t dampr_host_unregister(void *p) {
    if (!p) return DAMPR_OK;
    cudaError_t e = cudaHostUnregister(p);
    if (e != cudaSuccess) cudaGetLastError();
    return e == cudaSuccess ? DAMPR_OK : DAMPR_ERR_CUDA;
}

// ---- text buffers -------------------------------------------------------------------------
int32_t dampr_textbuf_create(dampr_ctx *ctx, uint64_t capacity, dampr_textbuf **out) {
    ARG_CHECK(ctx, ctx && out, "null");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    dampr_textbuf *tb = new dampr_textbuf();
    u64 cap16 = (capacity + 15) & ~15ULL;
    tb->alloc_bytes = TEXT_LEAD + cap16 + TEXT_TAIL_PAD;
    tb->capacity = capacity;
    tb->n = 0;
    tb->uploaded_hi = 0;
    cudaError_t e = cudaMalloc(&tb->alloc, tb->alloc_bytes);
    if (e != cudaSuccess) {
        delete tb;
        ctx->err = std::string("cudaMalloc(textbuf) failed: ") + cudaGetErrorString(e);
        return DAMPR_ERR_NOMEM;
    }
    tb->text = tb->alloc + TEXT_LEAD;
    // lead-in reads as '\n' so offset 0 is a line start
    CUDA_TRY(ctx, cudaMemsetAsync(tb->alloc, '\n', TEXT_LEAD, ctx->copy));
    *out = tb;
    return DAMPR_OK;
}

int32_t dampr_textbuf_destroy(dampr_ctx *ctx, dampr_textbuf *tb) {
    if (!tb) return DAMPR_OK;
    if (ctx) {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        cudaStreamSynchronize(ctx->copy);
    }
    cudaFree(tb->alloc);
    delete tb;
    return DAMPR_OK;
}

int32_t dampr_textbuf_set_length(dampr_ctx *ctx, dampr_textbuf *tb, uint64_t n) {
    ARG_CHECK(ctx, ctx && tb, "null");
    ARG_CHECK(ctx, n <= tb->capacity, "length exceeds textbuf capacity");
    tb->n = n;
    // everything after the text reads as '\n' (virtual terminator of an unterminated last line)
    u64 pad = tb->alloc_bytes - TEXT_LEAD - n;
    CUDA_TRY(ctx, cudaMemsetAsync(tb->text + n, '\n', pad, ctx->copy));
    CUDA_TRY(ctx, cudaEventRecord(ctx->upload_done, ctx->copy));
    ctx->upload_pending = true;
    return DAMPR_OK;
}

int32_t dampr_textbuf_upload(dampr_ctx *ctx, dampr_textbuf *tb, uint64_t off, const void *host,
                             uint64_t len) {
    ARG_CHECK(ctx, ctx && tb && (host || len == 0), "null");
    ARG_CHECK(ctx, off + len <= tb->capacity, "upload exceeds textbuf capacity");
    if (len) {
        int rc = staged_h2d(ctx, tb->text + off, host, len, ctx->copy);
        if (rc) return rc;
        if (off + len > tb->uploaded_hi) tb->uploaded_hi = off + len;
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->upload_done, ctx->copy));
    ctx->upload_pending = true;
    return DAMPR_OK;
}

// ---- GPUDirect Storage ingest (cuFile), opt-in: dampr_set_option("file_cufile", 1) ---------------------------
// libcufile is bound at run time. cuFileRead moves file bytes to device memory without the page-locked ring, by
// DMA from the NVMe controller, where the nvidia-fs driver and an O_DIRECT-capable file system are present. Without
// the driver the path is refused before libcufile is touched: cuFile's "compatibility mode" only copies through its
// own bounce buffers, which the ring does too, and on B200 machines without the driver its cuFileRead blocked for
// good. Several host threads issue disjoint 16 MB reads.
namespace {

struct CuFileApi {
    void *lib = nullptr;
    CUfileError_t (*DriverOpen)() = nullptr;
    CUfileError_t (*HandleRegister)(CUfileHandle_t *, CUfileDescr_t *) = nullptr;
    void (*HandleDeregister)(CUfileHandle_t) = nullptr;
    ssize_t (*Read)(CUfileHandle_t, void *, size_t, off_t, off_t) = nullptr;
    bool driver_open = false;
    std::string why;
};

CuFileApi *cufile_api() {
    static CuFileApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        if (access("/proc/driver/nvidia-fs/version", F_OK) != 0) {
            api.why = "the nvidia-fs (GPUDirect Storage) driver is not loaded";
            return;
        }
        const char *names[] = {"libcufile.so.0", "libcufile.so", "/usr/local/cuda/targets/x86_64-linux/lib/libcufile.so.0"};
        for (const char *n : names) {
            api.lib = dlopen(n, RTLD_NOW);
            if (api.lib) break;
        }
        if (!api.lib) {
            api.why = "libcufile.so.0 not found";
            return;
        }
        api.DriverOpen = reinterpret_cast<decltype(api.DriverOpen)>(dlsym(api.lib, "cuFileDriverOpen"));
        api.HandleRegister = reinterpret_cast<decltype(api.HandleRegister)>(dlsym(api.lib, "cuFileHandleRegister"));
        api.HandleDeregister = reinterpret_cast<decltype(api.HandleDeregister)>(dlsym(api.lib, "cuFileHandleDeregister"));
        api.Read = reinterpret_cast<decltype(api.Read)>(dlsym(api.lib, "cuFileRead"));
        if (!api.DriverOpen || !api.HandleRegister || !api.HandleDeregister || !api.Read) {
            api.why = "cuFile symbols missing";
            api.lib = nullptr;
            return;
        }
        const CUfileError_t e = api.DriverOpen();
        if (e.err != CU_FILE_SUCCESS) {
            api.why = "cuFileDriverOpen failed (" + std::to_string((int)e.err) + ")";
            api.lib = nullptr;
            return;
        }
        api.driver_open = true;
    });
    return &api;
}

int cufile_h2d(dampr_ctx *ctx, void *dst, const char *path, size_t foff, size_t bytes) {
    CuFileApi *a = cufile_api();
    if (!a->driver_open) {
        return set_err(ctx, DAMPR_ERR_CUDA, "cuFile is not available: %s", a->why.c_str());
    }
    // O_DIRECT first (what GPUDirect Storage wants); a file system that refuses it, or whose registration fails
    // with it, gets a second try with a plain descriptor (cuFile's compatibility mode)
    int fd = -1;
    CUfileHandle_t fh;
    int last_err = 0;
    bool registered = false;
    for (int attempt = 0; attempt < 2 && !registered; ++attempt) {
        fd = open(path, attempt == 0 ? (O_RDONLY | O_DIRECT) : O_RDONLY);
        if (fd < 0) continue;
        CUfileDescr_t descr;
        memset(&descr, 0, sizeof descr);
        descr.handle.fd = fd;
        descr.type = CU_FILE_HANDLE_TYPE_OPAQUE_FD;
        const CUfileError_t e = a->HandleRegister(&fh, &descr);
        if (e.err == CU_FILE_SUCCESS) {
            registered = true;
        } else {
            last_err = (int)e.err;
            close(fd);
            fd = -1;
        }
    }
    if (!registered) {
        char b[64];
        snprintf(b, sizeof b, "CUfileOpError %d", last_err);
        return set_err(ctx, DAMPR_ERR_CUDA, "cuFileHandleRegister failed (%s): this file system is not served by cuFile", b);
    }
    const size_t PIECE = 16u << 20;
    const size_t pieces = (bytes + PIECE - 1) / PIECE;
    const int nthreads = (int)std::max<size_t>(1, std::min<size_t>(pieces, (size_t)g_cufile_threads));
    std::atomic<size_t> next{0};
    std::atomic<int> failed{0};
    const int device = ctx->device;
    auto work = [&] {
        cudaSetDevice(device);
        for (;;) {
            const size_t i = next.fetch_add(1);
            if (i >= pieces || failed.load()) break;
            const size_t lo = i * PIECE, len = std::min(PIECE, bytes - lo);
            size_t got = 0;
            while (got < len) {
                const ssize_t r = a->Read(fh, dst, len - got, (off_t)(foff + lo + got), (off_t)(lo + got));
                if (r <= 0) {
                    failed.store(1);
                    break;
                }
                got += (size_t)r;
            }
        }
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nthreads; ++t) th.emplace_back(work);
    work();
    for (auto &t : th) t.join();
    a->HandleDeregister(fh);
    close(fd);
    if (failed.load()) return set_err(ctx, DAMPR_ERR_CUDA, "cuFileRead failed on %s", path);
    return DAMPR_OK;
}

}  // namespace

int32_t dampr_textbuf_upload_file(dampr_ctx *ctx, dampr_textbuf *tb, uint64_t off, const char *path,
                                  uint64_t file_off, uint64_t len) {
    ARG_CHECK(ctx, ctx && tb && path, "null");
    ARG_CHECK(ctx, off + len <= tb->capacity, "upload exceeds textbuf capacity");
    if (len && g_file_cufile) {
        CUDA_TRY(ctx, cudaSetDevice(ctx->device));
        // earlier uploads into this buffer travel on the copy stream; cuFileRead is not stream-ordered
        CUDA_TRY(ctx, cudaStreamSynchronize(ctx->copy));
        const int rc = cufile_h2d(ctx, tb->text + off, path, file_off, len);
        if (rc) return rc;
        if (off + len > tb->uploaded_hi) tb->uploaded_hi = off + len;
    } else if (len) {
        const int fd = open(path, O_RDONLY);
        if (fd < 0) return set_err(ctx, DAMPR_ERR_ARG, "cannot open %s", path);
        const int rc = staged_file_h2d(ctx, tb->text + off, fd, file_off, len, ctx->copy);
        close(fd);
        if (rc) return rc;
        if (off + len > tb->uploaded_hi) tb->uploaded_hi = off + len;
    }
    CUDA_TRY(ctx, cudaEventRecord(ctx->upload_done, ctx->copy));
    ctx->upload_pending = true;
    return DAMPR_OK;
}

int32_t dampr_textbuf_devptr(dampr_ctx *ctx, dampr_textbuf *tb, uint64_t *out_ptr) {
    ARG_CHECK(ctx, ctx && tb && out_ptr, "null");
    *out_ptr = (uint64_t)(uintptr_t)tb->text;
    return DAMPR_OK;
}

// ---- kv containers ------------------------------------------------------------------------
int32_t dampr_kv_create(dampr_ctx *ctx, uint64_t capacity, dampr_kv **out) {
    ARG_CHECK(ctx, ctx && out, "null");
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    dampr_kv *kv = new dampr_kv();
    kv->capacity = capacity;
    kv->n = 0;
    kv->alt = nullptr;
    kv->rec = nullptr;
    u64 bytes = (capacity ? capacity : 1) * sizeof(ulonglong2);
    kv->rec = (ulonglong2 *)pool_alloc(ctx, bytes);
    if (!kv->rec) {
        delete kv;
        ctx->err = "device allocation (kv) failed";
        return DAMPR_ERR_NOMEM;
    }
    *out = kv;
    return DAMPR_OK;
}

int32_t dampr_kv_destroy(dampr_ctx *ctx, dampr_kv *kv) {
    if (!kv) return DAMPR_OK;
    if (ctx) {
        cudaSetDevice(ctx->device);
        pool_free(ctx, kv->rec);  // recycled once the work recorded on both streams has finished
        if (kv->alt) pool_free(ctx, kv->alt);
    } else {
        cudaFree(kv->rec);
        if (kv->alt) cudaFree(kv->alt);
    }
    delete kv;
    return DAMPR_OK;
}

int32_t dampr_kv_size(dampr_ctx *ctx, dampr_kv *kv, uint64_t *n) {
    ARG_CHECK(ctx, ctx && kv && n, "null");
    *n = kv->n;
    return DAMPR_OK;
}

int32_t dampr_kv_set_size(dampr_ctx *ctx, dampr_kv *kv, uint64_t n) {
    ARG_CHECK(ctx, ctx && kv, "null");
    ARG_CHECK(ctx, n <= kv->capacity, "size exceeds kv capacity");
    kv->n = n;
    return DAMPR_OK;
}

int32_t dampr_kv_devptr(dampr_ctx *ctx, dampr_kv *kv, uint64_t *out_ptr) {
    ARG_CHECK(ctx, ctx && kv && out_ptr, "null");
    *out_ptr = (uint64_t)(uintptr_t)kv->rec;
    return DAMPR_OK;
}

int32_t dampr_kv_upload(dampr_ctx *ctx, dampr_kv *kv, uint64_t off, const void *host_records,
                        uint64_t count) {
    ARG_CHECK(ctx, ctx && kv && (host_records || count == 0), "null");
    ARG_CHECK(ctx, off + count <= kv->capacity, "upload exceeds kv capacity");
    // uploads must not overtake compute that still reads the buffer
    if (count) {
        int rc = staged_h2d(ctx, kv->rec + off, host_records, count * sizeof(ulonglong2), ctx->copy);
        if (rc) return rc;
    }
    if (off + count > kv->n) kv->n = off + count;
    CUDA_TRY(ctx, cudaEventRecord(ctx->upload_done, ctx->copy));
    ctx->upload_pending = true;
    return DAMPR_OK;
}

int32_t dampr_kv_download(dampr_ctx *ctx, dampr_kv *kv, uint64_t off, void *host_records,
                          uint64_t count) {
    ARG_CHECK(ctx, ctx && kv && (host_records || count == 0), "null");
    ARG_CHECK(ctx, off + count <= kv->n, "download exceeds kv size");
    wait_uploads(ctx);
    if (count) return staged_d2h(ctx, host_records, kv->rec + off, count * sizeof(ulonglong2), ctx->stream);
    return DAMPR_OK;
}

}  // extern "C"
