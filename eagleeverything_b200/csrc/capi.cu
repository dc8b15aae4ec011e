// Host side of libeaglegpu.so: per-GPU contexts, resident genotype stores + path cache, the multi-GPU set, and the C
// entry points of include/eagle_gpu.h (the reference-facing exports, the store API, device-level pieces and ingest).
// No CPU compute path exists here: every entry point either runs the CUDA kernels or fails with an error code.
#include <cublas_v2.h>
#include <dlfcn.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cmath>
#include <cstdarg>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <string>
#include <vector>

#include "common.cuh"
#include "hostio.cuh"

struct eg_store {
    int8_t* d = nullptr;
    int64_t rows = 0, cols = 0;
    int64_t pitch = 0;  // row-major stores (Mt orientation): bytes per row.  0: K-blocked store (M orientation),
                        // [ceil(cols/128)][rows][128] bytes -- the layout the SYRK streams (syrk_i8.cu)
    size_t bytes() const { return pitch ? (size_t)rows * (size_t)pitch : (size_t)((cols + 127) / 128) * (size_t)rows * 128; }
    // M stores uploaded from a host image: rows x rows int32, M * M^T over all columns of the store, accumulated chunk
    // by chunk UNDER the host-to-device copy (store_from_image); eg_store_mmt then only finalizes.  nullptr otherwise.
    int32_t* C32 = nullptr;
    int pins = 0;   // > 0 while an entry point works on the store: cache eviction under memory pressure skips it
    // Marker-sharded stores (eg_init_multi with more than one GPU): nparts > 1, part[r] lives on GPU slot r and holds the
    // markers [off[r], off[r+1]) -- columns of an M store, rows of an Mt store; d == nullptr, rows / cols are the totals.
    int nparts = 0;
    eg_store* part[16] = {};
    int64_t off[17] = {};
    bool mt_orientation = false;   // composite stores: which axis is sharded (row-major parts: rows)
};

namespace eg {

// ------------------------------------------------------------------ errors
static thread_local char g_err[1024] = "";

int set_error(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}
int check_cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return EG_OK;
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        return set_error(EG_ERR_ALLOC, "CUDA out of memory in %s", what);
    }
    return set_error(EG_ERR_CUDA, "CUDA error in %s: %s", what, cudaGetErrorString(e));
}
static std::atomic<long long> g_launches{0};  // kernels launched by this library (bench.py reports the count)
int check_launch(const char* kernel) {
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return check_cuda(cudaGetLastError(), kernel);
}

// ------------------------------------------------------------------ context
struct CacheEntry {
    std::string key;
    eg_store* store;
    uint64_t stamp;
};
struct FreeBlock {
    void* p;
    size_t bytes;
};
// One context per GPU.  Slot 0 is the device of eg_init(); eg_init_multi(ngpu, devs) fills slots 0 .. ngpu-1 and starts one
// host thread per slot.  Every thread works on the slot its thread-local pointer names (the calling thread: slot 0).
struct Context {
    bool ready = false;
    int device = -1;
    int sms = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;
    cublasHandle_t cublas = nullptr;
    std::vector<CacheEntry> cache;
    uint64_t clock = 0;
    int32_t* d_err = nullptr;
    double timing[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    // exact-size recycling list on top of the stream-ordered pool (see pool_alloc)
    std::mutex pool_mu;
    std::vector<FreeBlock> free_blocks;
    std::unordered_map<void*, size_t> live_blocks;
    size_t free_bytes = 0, recycle_limit = 0;
    cudaEvent_t scan_ev[2] = {nullptr, nullptr};   // around the dominant scan kernel of the last eg_dev_scan on this GPU
    double scan_ops = 0.0;
    void reset() {
        ready = false; device = -1; sms = 0; stream = copy_stream = nullptr; cublas = nullptr; cache.clear(); clock = 0;
        d_err = nullptr; for (double& t : timing) t = 0; free_blocks.clear(); live_blocks.clear(); free_bytes = 0; recycle_limit = 0; scan_ev[0] = scan_ev[1] = nullptr; scan_ops = 0.0;
    }
};
constexpr int EG_MAX_GPUS = 16;
static Context g_ctxs[EG_MAX_GPUS];
static thread_local Context* t_ctx = &g_ctxs[0];
#define g_ctx (*t_ctx)

int num_sms() {
    if (g_ctx.sms > 0) return g_ctx.sms;
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0)
        return sms;
    return 148;
}

static int ensure_init() {
    if (g_ctx.ready) return check_cuda(cudaSetDevice(g_ctx.device), "cudaSetDevice");
    const char* env = getenv("EAGLE_GPU_DEVICE");
    return eg_init(env ? atoi(env) : 0);
}

// accessors for the other translation units of the library (algebra.cu)
int ensure_init_pub() { return ensure_init(); }
cudaStream_t ctx_stream() { return g_ctx.stream; }
cublasHandle_t ctx_cublas() { return g_ctx.cublas; }

void syrk_release_cache();
void scan_i8_release();
void algebra_release();
void eigbasis_release();
void prep_i8_release();
int launch_prepare_i8(const double* d_S, const double* d_V, int64_t n, int64_t col0, int64_t col1, double* d_tmp,
                      double* d_Wp, int64_t Kpad, cudaStream_t st, bool* done);
static int g_scan_mode = -1;
int scan_mode() {
    if (g_scan_mode < 0) {
        const char* e = getenv("EAGLE_SCAN_MODE");  // default: exact int8 slices; "f64" / "dmma" / "0" selects DMMA
        g_scan_mode = (e && (e[0] == 'f' || e[0] == 'd' || e[0] == '0')) ? 0 : 1;
    }
    return g_scan_mode;
}
int launch_scan(const int8_t* d_Mt, int64_t L, int64_t n, int64_t pitch, const double* d_Wp,
                const int64_t* d_zero_rows, int n_zero, double* d_a, double* d_vara, cudaStream_t st);

// Stream-ordered allocations from the device's default memory pool (release threshold raised in eg_init), with an
// exact-size recycling list on top: every forward step asks for the same handful of multi-GB sizes (two 10 GB stores,
// n x n workspaces, staging buffers), and handing a freed block straight back to the next request of the same size keeps
// the driver pool from splitting a 10 GB block for an 800 MB request and then having to map 10 GB of fresh memory for
// the next store -- measured as random 0.2 - 0.9 s stalls inside eg_store_from_host_ascii / eg_store_a_and_vara
// (scripts/e2e_probe.py: steps of 540 ms turning into 1,200 - 1,400 ms).  Everything here is ordered on g_ctx.stream.
static void pool_flush_locked() {
    for (auto& b : g_ctx.free_blocks) cudaFreeAsync(b.p, g_ctx.stream);
    g_ctx.free_blocks.clear();
    g_ctx.free_bytes = 0;
}
static cudaError_t pool_alloc(void** p, size_t bytes) {
    if (!bytes) bytes = 16;
    std::lock_guard<std::mutex> lk(g_ctx.pool_mu);
    for (size_t i = 0; i < g_ctx.free_blocks.size(); i++)
        if (g_ctx.free_blocks[i].bytes == bytes) {
            *p = g_ctx.free_blocks[i].p;
            g_ctx.free_bytes -= bytes;
            g_ctx.free_blocks.erase(g_ctx.free_blocks.begin() + i);
            g_ctx.live_blocks[*p] = bytes;
            return cudaSuccess;
        }
    cudaError_t e = cudaMallocAsync(p, bytes, g_ctx.stream);
    if (e != cudaSuccess && !g_ctx.free_blocks.empty()) {  // make room: give the recycled blocks back and try once more
        cudaGetLastError();
        pool_flush_locked();
        cudaStreamSynchronize(g_ctx.stream);
        e = cudaMallocAsync(p, bytes, g_ctx.stream);
    }
    if (e == cudaSuccess) g_ctx.live_blocks[*p] = bytes;
    return e;
}
static void pool_free(void* p) {
    if (!p) return;
    std::lock_guard<std::mutex> lk(g_ctx.pool_mu);
    auto it = g_ctx.live_blocks.find(p);
    const size_t bytes = it == g_ctx.live_blocks.end() ? 0 : it->second;
    if (it != g_ctx.live_blocks.end()) g_ctx.live_blocks.erase(it);
    if (bytes >= ((size_t)1 << 20) && g_ctx.free_bytes + bytes <= g_ctx.recycle_limit) {
        g_ctx.free_blocks.push_back({p, bytes});
        g_ctx.free_bytes += bytes;
    } else {
        cudaFreeAsync(p, g_ctx.stream);
    }
}
static void pool_flush() {
    std::lock_guard<std::mutex> lk(g_ctx.pool_mu);
    pool_flush_locked();
}
// For the plain cudaMalloc users of the library (LAPACK workspace, digit slices, host-level algebra buffers): when the
// device is out of memory, hand the recycled blocks and the cached part of the stream-ordered pool back to the driver --
// those bytes are invisible to cudaMalloc -- so that the caller can retry once.  eg_cache_clear() uses it, too.
void pool_give_back() {
    if (!g_ctx.ready) return;
    pool_flush();
    cudaStreamSynchronize(g_ctx.stream);
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, g_ctx.device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
}

// Scratch for work queued on `st` by another translation unit (syrk_i8.cu: the E2M1 copy of a store).  The pool orders
// everything on g_ctx.stream, so `st` waits for the allocation and g_ctx.stream for the work on `st` before the block
// can be handed out again.
static void stream_after(cudaStream_t waiter, cudaStream_t st) {
    if (waiter == st) return;
    cudaEvent_t ev;
    if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) {
        cudaGetLastError();
        cudaStreamSynchronize(st);
        return;
    }
    cudaEventRecord(ev, st);
    cudaStreamWaitEvent(waiter, ev, 0);
    cudaEventDestroy(ev);
}
cudaError_t scratch_alloc(void** p, size_t bytes, cudaStream_t st) {
    cudaError_t e = pool_alloc(p, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        *p = nullptr;
        return e;
    }
    stream_after(st, g_ctx.stream);
    return cudaSuccess;
}
void scratch_free(void* p, cudaStream_t st) {
    stream_after(g_ctx.stream, st);
    pool_free(p);
}

// RAII device buffer (valid on g_ctx.stream)
struct DevBuf {
    void* p = nullptr;
    ~DevBuf() { pool_free(p); }
    int alloc(size_t bytes, const char* what) {
        pool_free(p);
        p = nullptr;
        cudaError_t e = pool_alloc(&p, bytes);
        if (e != cudaSuccess) {
            cudaGetLastError();
            p = nullptr;
            return set_error(EG_ERR_ALLOC, "out of device memory allocating %zu bytes for %s", bytes, what);
        }
        return EG_OK;
    }
    template <class T>
    T* as() { return reinterpret_cast<T*>(p); }
};

struct Timer {
    cudaEvent_t a, b;
    cudaStream_t st;
    Timer(cudaStream_t s) : st(s) {
        cudaEventCreate(&a);
        cudaEventCreate(&b);
        cudaEventRecord(a, st);
    }
    double stop() {
        float ms = 0;
        cudaEventRecord(b, st);
        cudaEventSynchronize(b);
        cudaEventElapsedTime(&ms, a, b);
        return ms;
    }
    ~Timer() {
        cudaEventDestroy(a);
        cudaEventDestroy(b);
    }
};

static bool is_na(double x) { return std::isnan(x); }  // NA_real_ is a NaN; see header

// selected_loci (doubles, NA sentinel) -> validated 0-based index list
static int parse_selected(const double* sel, int64_t nsel, int64_t limit, std::vector<int64_t>& out, const char* who) {
    out.clear();
    if (!sel || nsel <= 0 || is_na(sel[0])) return EG_OK;
    for (int64_t i = 0; i < nsel; i++) {
        if (is_na(sel[i]) || sel[i] < 0 || sel[i] >= (double)limit)
            return set_error(EG_ERR_ARG, "%s: selected_loci[%lld] = %g is outside [0, %lld)", who, (long long)i,
                             sel[i], (long long)limit);
        out.push_back((int64_t)sel[i]);
    }
    return EG_OK;
}

// ------------------------------------------------------------------ stores
static thread_local bool t_is_worker = false;   // a GPU slot's worker thread (eg_init_multi): never evicts, never fans out
struct Pin {   // RAII: a store an entry point is working on is not evictable (nor are the parts of a sharded store)
    eg_store* s;
    explicit Pin(const eg_store* st) : s(const_cast<eg_store*>(st)) { if (s) s->pins++; }
    ~Pin() { if (s) s->pins--; }
    Pin(const Pin&) = delete;
    Pin& operator=(const Pin&) = delete;
};
static void free_store_tree(eg_store* s);
// Drops the least recently used cached store of this slot that no entry point holds; false when none is left.
static bool cache_evict_one() {
    size_t lru = g_ctx.cache.size();
    for (size_t i = 0; i < g_ctx.cache.size(); i++)
        if (g_ctx.cache[i].store->pins == 0 && (lru == g_ctx.cache.size() || g_ctx.cache[i].stamp < g_ctx.cache[lru].stamp)) lru = i;
    if (lru == g_ctx.cache.size()) return false;
    eg_store* victim = g_ctx.cache[lru].store;
    g_ctx.cache.erase(g_ctx.cache.begin() + lru);
    free_store_tree(victim);
    cudaStreamSynchronize(g_ctx.stream);
    return true;
}
static int store_alloc(int64_t rows, int64_t cols, bool kblocked, eg_store** out) {
    eg_store* s = new eg_store();
    s->rows = rows;
    s->cols = cols;
    s->pitch = kblocked ? 0 : store_pitch(cols);
    const char* inject = getenv("EAGLE_TEST_FAIL_ALLOC");   // tests: every allocation attempt of a store fails
    const bool fail = inject && inject[0] == '1';
    cudaError_t e = fail ? cudaErrorMemoryAllocation : pool_alloc((void**)&s->d, s->bytes() + 256);
    if (e != cudaSuccess) {
        cudaGetLastError();
        // evict cached stores (least recently used first, never one that a caller still holds) and retry once per
        // eviction; worker threads of a multi-GPU set leave eviction to the orchestrating thread (store_from_image_any)
        while (e != cudaSuccess && !t_is_worker && cache_evict_one()) {
            e = fail ? cudaErrorMemoryAllocation : pool_alloc((void**)&s->d, s->bytes() + 256);
            if (e != cudaSuccess) cudaGetLastError();
        }
        if (e != cudaSuccess) {
            delete s;
            return set_error(EG_ERR_ALLOC, "out of device memory for a %lld x %lld genotype store", (long long)rows,
                             (long long)cols);
        }
    }
    *out = s;
    return EG_OK;
}
// The end of every store built in this file: hand s out when rc is EG_OK, otherwise free it and pass rc on.
static int finish_store(int rc, eg_store* s, eg_store** out) {
    if (rc != EG_OK) {
        free_store_tree(s);
        return rc;
    }
    *out = s;
    return EG_OK;
}
// The ASCII decoders' 4-int status (flag, row bits 0-30, column, row bits 31-) -> EG_ERR_FORMAT; row0 / col0: where the
// decoded range starts in the image.
static int decode_status(const int32_t* h_err, int64_t row0, int64_t col0) {
    if (!h_err[0]) return EG_OK;
    const int64_t brow = ((int64_t)h_err[3] << 31) | (int64_t)h_err[1];
    return set_error(EG_ERR_FORMAT,
                     "genotype file is not in no-space ASCII format: byte outside {'0','1','2'} near row %lld, column %lld "
                     "(wrong dims / line pitch?)",
                     (long long)(row0 + brow), (long long)(col0 + h_err[2]));
}

// K-blocked (M orientation) stores: the image is uploaded in COLUMN chunks (2-D copies, ~256 MB each, two staging
// buffers); every chunk is decoded into its 128-marker blocks and its contribution to M * M^T is accumulated right
// away (int32, exact, order-free), so that decode and the whole SYRK hide under the PCIe transfer -- at config 3 the
// upload takes 181 ms and the SYRK 34.  The product stays with the store (eg_store::C32).
static int store_from_image_kb(const uint8_t* image, int64_t src_pitch_host, int64_t row0, int64_t rows, int64_t col0,
                               int64_t w, eg_store* s, eg_store** out) {
    int64_t cw = ((int64_t)(256LL << 20) / rows) / 128 * 128;
    if (cw < 128) cw = 128;
    if (cw > round_up(w, 128)) cw = round_up(w, 128);
    const int64_t nchunks = (w + cw - 1) / cw;
    DevBuf stg[2], errs;
    cudaEvent_t copied[2], decoded[2];
    int rc = EG_OK;
    for (int i = 0; i < 2 && rc == EG_OK; i++) rc = stg[i].alloc((size_t)rows * cw + 64, "ASCII staging");
    if (rc == EG_OK) rc = errs.alloc((size_t)nchunks * 4 * sizeof(int32_t), "decode status");
    bool eager = rc == EG_OK && rows >= 2;
    if (eager && pool_alloc((void**)&s->C32, (size_t)rows * rows * sizeof(int32_t)) != cudaSuccess) {
        cudaGetLastError();
        s->C32 = nullptr;   // no room for the product: upload only
        eager = false;
    }
    if (rc != EG_OK) return finish_store(rc, s, out);
    for (int i = 0; i < 2; i++) {
        cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&decoded[i], cudaEventDisableTiming);
    }
    cudaMemsetAsync(errs.p, 0, (size_t)nchunks * 4 * sizeof(int32_t), g_ctx.stream);
    if (eager) cudaMemsetAsync(s->C32, 0, (size_t)rows * rows * sizeof(int32_t), g_ctx.stream);
    cudaEventRecord(decoded[0], g_ctx.stream);
    cudaStreamWaitEvent(g_ctx.copy_stream, decoded[0], 0);  // staging buffers were allocated in g_ctx.stream order
    Timer total(g_ctx.stream);
    for (int64_t k = 0; k < nchunks && rc == EG_OK; k++) {
        const int b = (int)(k & 1);
        const int64_t c = k * cw, wk = (c + cw <= w) ? cw : w - c;
        if (k >= 2) cudaStreamWaitEvent(g_ctx.copy_stream, decoded[b], 0);
        const uint8_t* src = image + row0 * src_pitch_host + col0 + c;
        rc = check_cuda(cudaMemcpy2DAsync(stg[b].p, cw, src, src_pitch_host, wk, rows, cudaMemcpyHostToDevice, g_ctx.copy_stream),
                        "H2D copy of the ASCII genotype image");
        if (rc != EG_OK) break;
        cudaEventRecord(copied[b], g_ctx.copy_stream);
        cudaStreamWaitEvent(g_ctx.stream, copied[b], 0);
        int8_t* blocks = s->d + (c / 128) * rows * 128;     // first 128-marker block of this chunk
        rc = eg_dev_decode_kb(stg[b].as<uint8_t>(), cw, (int64_t)rows * cw + 64, rows, wk, blocks, rows, 0,
                              errs.as<int32_t>() + 4 * k, g_ctx.stream);
        cudaEventRecord(decoded[b], g_ctx.stream);
        if (rc == EG_OK && eager) rc = eg_dev_syrk_i8_kb(blocks, rows, wk, s->C32, rows, g_ctx.stream);
    }
    std::vector<int32_t> h_err((size_t)nchunks * 4, 0);
    if (rc == EG_OK)
        rc = check_cuda(cudaMemcpyAsync(h_err.data(), errs.p, h_err.size() * sizeof(int32_t), cudaMemcpyDeviceToHost, g_ctx.stream),
                        "decode status D2H");
    if (rc == EG_OK) rc = check_cuda(cudaStreamSynchronize(g_ctx.stream), "genotype decode");
    cudaStreamSynchronize(g_ctx.copy_stream);
    g_ctx.timing[0] = total.stop();  // H2D + decode + M.Mt (overlapped)
    for (int i = 0; i < 2; i++) {
        cudaEventDestroy(copied[i]);
        cudaEventDestroy(decoded[i]);
    }
    for (int64_t k = 0; k < nchunks && rc == EG_OK; k++) rc = decode_status(&h_err[4 * k], row0, col0 + k * cw);
    return finish_store(rc, s, out);
}

// Host ASCII image -> store.  Rows [row0,row1), columns [col0,col1) of an image with `cols_total`
// characters per line.  Row blocks are staged through two device buffers so that the H2D copy of
// block k+1 overlaps the decode of block k.
static int store_from_image(const uint8_t* image, int64_t cols_total, int64_t row0, int64_t row1, int64_t col0,
                            int64_t col1, bool kblocked, eg_store** out, int fd = -1) {
    EG_TRY(ensure_init());
    const int64_t rows = row1 - row0, w = col1 - col0, src_pitch_host = cols_total + 1;
    if (!image || rows <= 0 || w <= 0 || col0 < 0 || col1 > cols_total || row0 < 0)
        return set_error(EG_ERR_ARG, "genotype store: bad image range");
    eg_store* s = nullptr;
    EG_TRY(store_alloc(rows, w, kblocked, &s));
    if (kblocked) {
        // column-chunk pipeline with the M.Mt accumulation under the copy: for page-locked images (2-D copies out of
        // pageable / mmap'ed memory are staged by the driver and slower than the row-block path below)
        const char* env = getenv("EAGLE_EAGER_MMT");
        cudaPointerAttributes at;
        const bool pinned = cudaPointerGetAttributes(&at, image) == cudaSuccess && at.type == cudaMemoryTypeHost;
        cudaGetLastError();
        if (pinned && !(env && env[0] == '0')) return store_from_image_kb(image, src_pitch_host, row0, rows, col0, w, s, out);
    }
    const bool full_width = (w == cols_total);
    const int64_t dev_pitch = full_width ? src_pitch_host : round_up(w, 16);
    int64_t block_rows = (int64_t)(256LL << 20) / dev_pitch;
    if (block_rows < 1) block_rows = 1;
    if (block_rows > rows) block_rows = rows;
    DevBuf stg[2];
    cudaEvent_t copied[2], decoded[2];
    int rc = EG_OK;
    for (int i = 0; i < 2 && rc == EG_OK; i++) rc = stg[i].alloc((size_t)block_rows * dev_pitch + 64, "ASCII staging");
    if (rc != EG_OK) return finish_store(rc, s, out);
    for (int i = 0; i < 2; i++) {
        cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&decoded[i], cudaEventDisableTiming);
    }
    // the staging buffers were allocated in g_ctx.stream order: the copy stream must not run ahead of that
    cudaEventRecord(decoded[0], g_ctx.stream);
    cudaStreamWaitEvent(g_ctx.copy_stream, decoded[0], 0);
    cudaMemsetAsync(g_ctx.d_err, 0, 4 * sizeof(int32_t), g_ctx.stream);
    double t_h2d = 0;
    Timer total(g_ctx.stream);
    int k = 0;
    for (int64_t r = 0; r < rows && rc == EG_OK; r += block_rows, k++) {
        const int b = k & 1;
        const int64_t nr = (r + block_rows <= rows) ? block_rows : rows - r;
        if (k >= 2) cudaStreamWaitEvent(g_ctx.copy_stream, decoded[b], 0);  // staging buffer free again
        // pageable memory and files go through the page-locked ring with parallel copier threads (hostio.cu); the
        // decode of this block then overlaps the staging of the next one
        HostSrc hs;
        hs.p = image;
        hs.fd = fd;
        const size_t soff = (size_t)(row0 + r) * (size_t)src_pitch_host + (size_t)col0;
        if (full_width) {
            // the very last line of a file may lack its '\n': never read past row1*pitch - 1
            size_t bytes = (size_t)nr * src_pitch_host;
            if (r + nr == rows) bytes -= 1;
            rc = h2d_staged_2d(stg[b].p, bytes, hs, soff, bytes, bytes, 1, g_ctx.copy_stream);
        } else {
            rc = h2d_staged_2d(stg[b].p, (size_t)dev_pitch, hs, soff, (size_t)src_pitch_host, (size_t)w, (size_t)nr, g_ctx.copy_stream);
        }
        if (rc != EG_OK) break;
        cudaEventRecord(copied[b], g_ctx.copy_stream);
        cudaStreamWaitEvent(g_ctx.stream, copied[b], 0);
        rc = kblocked ? eg_dev_decode_kb(stg[b].as<uint8_t>(), dev_pitch, (int64_t)block_rows * dev_pitch + 64, nr, w, s->d,
                                         rows, r, g_ctx.d_err, g_ctx.stream)
                      : eg_dev_decode(stg[b].as<uint8_t>(), dev_pitch, (int64_t)block_rows * dev_pitch + 64, nr, w,
                                      s->d + r * s->pitch, s->pitch, g_ctx.d_err, g_ctx.stream);
        cudaEventRecord(decoded[b], g_ctx.stream);
    }
    int32_t h_err[4] = {0, 0, 0, 0};
    if (rc == EG_OK)
        rc = check_cuda(cudaMemcpyAsync(h_err, g_ctx.d_err, sizeof(h_err), cudaMemcpyDeviceToHost, g_ctx.stream),
                        "decode status D2H");
    if (rc == EG_OK) rc = check_cuda(cudaStreamSynchronize(g_ctx.stream), "genotype decode");
    cudaStreamSynchronize(g_ctx.copy_stream);
    t_h2d = total.stop();
    g_ctx.timing[0] = t_h2d;  // H2D + decode (overlapped)
    for (int i = 0; i < 2; i++) {
        cudaEventDestroy(copied[i]);
        cudaEventDestroy(decoded[i]);
    }
    if (rc == EG_OK) rc = decode_status(h_err, row0, col0);
    return finish_store(rc, s, out);
}

struct MappedFile {
    int fd = -1;
    const uint8_t* p = nullptr;
    size_t size = 0;
    struct stat st;
    ~MappedFile() {
        if (p) munmap(const_cast<uint8_t*>(p), size);
        if (fd >= 0) close(fd);
    }
    int open_ro(const char* path) {
        fd = ::open(path, O_RDONLY);
        if (fd < 0) return set_error(EG_ERR_OPEN, "ERROR: Could not open  %s", path);  // ReadBlock.cpp:43
        if (fstat(fd, &st) != 0) return set_error(EG_ERR_OPEN, "ERROR: Could not open  %s", path);
        size = (size_t)st.st_size;
        if (size == 0) return set_error(EG_ERR_FORMAT, "%s is empty", path);
        void* m = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
        if (m == MAP_FAILED) return set_error(EG_ERR_OPEN, "could not map %s", path);
        p = static_cast<const uint8_t*>(m);
        madvise(m, size, MADV_SEQUENTIAL);
        return EG_OK;
    }
};

static int check_image_size(const MappedFile& f, const char* path, int64_t rows, int64_t cols) {
    const size_t want = (size_t)rows * (size_t)(cols + 1);
    if (f.size != want && f.size + 1 != want)
        return set_error(EG_ERR_FORMAT, "%s has %zu bytes; %lld rows x %lld columns of no-space ASCII need %zu", path,
                         f.size, (long long)rows, (long long)cols, want);
    if (rows > 1 && f.p[cols] != '\n')
        return set_error(EG_ERR_FORMAT, "%s: first line is not %lld characters long", path, (long long)cols);
    return EG_OK;
}

static int store_from_image_any(const uint8_t* image, int64_t cols_total, int64_t row0, int64_t row1, int64_t col0,
                                int64_t col1, bool kblocked, eg_store** out, bool allow_multi, int fd = -1);
// cache key: (realpath, size, mtime, hash of the first and last 4 KB, dims, layout)
static int cache_key(const char* path, int64_t rows, int64_t cols, bool kblocked, std::string& key) {
    struct stat st;
    if (stat(path, &st) != 0) return set_error(EG_ERR_OPEN, "ERROR: Could not open  %s", path);
    // FNV-1a over the first and the last 4 KB: a file rewritten with the same size inside one timestamp tick of the file
    // system (coarse mtime) must not be served from the stale store
    uint64_t h = 1469598103934665603ull;
    {
        const int fd = ::open(path, O_RDONLY);
        if (fd < 0) return set_error(EG_ERR_OPEN, "ERROR: Could not open  %s", path);
        unsigned char blk[4096];
        const off_t offs[2] = {0, st.st_size > 4096 ? st.st_size - 4096 : 0};
        for (int k = 0; k < (st.st_size > 4096 ? 2 : 1); k++) {
            const ssize_t got = pread(fd, blk, sizeof(blk), offs[k]);
            for (ssize_t i = 0; i < got; i++) h = (h ^ blk[i]) * 1099511628211ull;
        }
        close(fd);
    }
    char* rp = realpath(path, nullptr);
    char buf[4400];
    // inode and ctime as well: a file replaced by rename(), or rewritten in place inside one mtime tick, changes them
    snprintf(buf, sizeof(buf), "%s|%lld|%lld.%09ld|%llu|%lld.%09ld|%016llx|%lldx%lld|%c", rp ? rp : path, (long long)st.st_size,
             (long long)st.st_mtim.tv_sec, (long)st.st_mtim.tv_nsec, (unsigned long long)st.st_ino, (long long)st.st_ctim.tv_sec,
             (long)st.st_ctim.tv_nsec, (unsigned long long)h, (long long)rows, (long long)cols, kblocked ? 'K' : 'R');
    free(rp);
    key = buf;
    return EG_OK;
}
static void cache_insert(const std::string& key, eg_store* s) {
    const char* envmax = getenv("EAGLE_GPU_CACHE_ENTRIES");
    const size_t maxe = envmax ? (size_t)atoi(envmax) : 4;
    // entries of the same file (same path, dims, layout) under an older stamp are stale: a rewritten file must not keep
    // 10 GB resident until the LRU rule reaches it
    auto same_file = [](const std::string& a, const std::string& b) {
        const size_t pa = a.find('|'), pb = b.find('|');
        if (pa == std::string::npos || pa != pb || a.compare(0, pa, b, 0, pb) != 0) return false;
        const size_t ta = a.rfind('|', a.rfind('|') - 1), tb = b.rfind('|', b.rfind('|') - 1);   // "|rowsxcols|layout"
        return a.substr(ta) == b.substr(tb);
    };
    for (size_t i = 0; i < g_ctx.cache.size();)
        if (same_file(g_ctx.cache[i].key, key) && g_ctx.cache[i].store->pins == 0) {
            free_store_tree(g_ctx.cache[i].store);
            g_ctx.cache.erase(g_ctx.cache.begin() + i);
        } else i++;
    while (g_ctx.cache.size() >= (maxe ? maxe : 1))
        if (!cache_evict_one()) break;   // everything left is held by a caller
    g_ctx.cache.push_back({key, s, ++g_ctx.clock});
}
// allow_multi: with a multi-GPU set the store may be marker-sharded over the GPUs (the hot-path exports); callers that
// need one plain store (ingest, ReshapeM, the packed container) pass false and get it on the first GPU.
static int cached_store(const char* path, int64_t rows, int64_t cols, bool kblocked, eg_store** out, bool allow_multi = true) {
    EG_TRY(ensure_init());
    if (!path) return set_error(EG_ERR_ARG, "null file name");
    if (rows <= 0 || cols <= 0) return set_error(EG_ERR_ARG, "dims must be positive");
    std::string key;
    EG_TRY(cache_key(path, rows, cols, kblocked, key));
    for (auto& e : g_ctx.cache)
        if (e.key == key && (allow_multi || e.store->nparts <= 1)) {
            e.stamp = ++g_ctx.clock;
            *out = e.store;
            return EG_OK;
        }
    MappedFile f;
    EG_TRY(f.open_ro(path));
    EG_TRY(check_image_size(f, path, rows, cols));
    eg_store* s = nullptr;
    EG_TRY(store_from_image_any(f.p, cols, 0, rows, 0, cols, kblocked, &s, allow_multi, f.fd));
    cache_insert(key, s);
    *out = s;
    return EG_OK;
}

// ------------------------------------------------------------------ small conversion kernel for eg_ReadBlock
__global__ void __launch_bounds__(256) i8_to_f64_colmajor_kernel(const int8_t* __restrict__ in, int64_t rows,
                                                                 int64_t cols, int64_t pitch,
                                                                 double* __restrict__ out) {
    __shared__ int8_t tile[32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t r0 = (int64_t)blockIdx.y * 32, c0 = (int64_t)blockIdx.x * 32;
    for (int i = ty; i < 32; i += 8) {
        const int64_t r = r0 + i, c = c0 + tx;
        tile[i][tx] = (r < rows && c < cols) ? in[r * pitch + c] : (int8_t)0;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int64_t c = c0 + i, r = r0 + tx;
        if (r < rows && c < cols) out[r + c * rows] = -(double)tile[tx][i];  // stores hold the negated value (decode.cu)
    }
}

// ------------------------------------------------------------------ W -> U (symmetric half) for the scan
// In place on the packed Wp (column-major, ld = Kpad): for i < k  U[i][k] = W[i][k] + W[k][i], U[k][i] = 0.
// w_is_upper != 0: only the upper triangle of W was computed (W known symmetric): U[i][k] = 2 W[i][k].
__global__ void __launch_bounds__(256) symmetrize_upper_kernel(double* __restrict__ Wp, int64_t n, int64_t ld,
                                                               int w_is_upper) {
    __shared__ double tile[32][33];
    const int bx = blockIdx.x, by = blockIdx.y;  // tile (rows by*32.., cols bx*32..) with bx >= by
    if (bx < by) return;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int64_t r0 = (int64_t)by * 32, c0 = (int64_t)bx * 32;
    // stage the mirrored tile W[c0.., r0..] (rows of the lower part) through shared memory
    for (int i = ty; i < 32; i += 8) {
        const int64_t r = c0 + tx, c = r0 + i;  // element (r, c) of the lower tile, r fastest (coalesced)
        tile[i][tx] = (r < n && c < n) ? Wp[r + c * ld] : 0.0;
    }
    __syncthreads();
    for (int i = ty; i < 32; i += 8) {
        const int64_t r = r0 + tx, c = c0 + i;  // element (r, c) of the upper tile
        if (r < n && c < n) {
            if (r < c) Wp[r + c * ld] = Wp[r + c * ld] + (w_is_upper ? Wp[r + c * ld] : tile[tx][i]);  // W[r][c] + W[c][r]
            else if (r > c) Wp[r + c * ld] = 0.0;                        // inside a diagonal tile
        }
    }
    if (bx != by) {
        __syncthreads();
        for (int i = ty; i < 32; i += 8) {
            const int64_t r = c0 + tx, c = r0 + i;
            if (r < n && c < n) Wp[r + c * ld] = 0.0;  // strictly lower tile
        }
    }
}

// max |A_ij| and max |A_ij - A_ji| of a column-major n x n matrix (non-negative doubles order like uint64).
// 64 x 64 tiles, 16 independent 8-byte loads per thread and phase (the 32 x 32 version ran at 0.9 TB/s).
__global__ void __launch_bounds__(256) symmetry_kernel(const double* __restrict__ A, int64_t n,
                                                       unsigned long long* __restrict__ out) {
    __shared__ double tile[64][65];
    const int bx = blockIdx.x, by = blockIdx.y;
    if (bx < by) return;
    const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;  // 64 x 4
    const int64_t r0 = (int64_t)by * 64, c0 = (int64_t)bx * 64;
    double v[16];
#pragma unroll
    for (int k = 0; k < 16; k++) {  // mirrored tile: element (c0 + tx, r0 + i), first index fastest (coalesced)
        const int i = ty + 4 * k;
        const int64_t r = c0 + tx, c = r0 + i;
        v[k] = (r < n && c < n) ? A[r + c * n] : 0.0;
    }
#pragma unroll
    for (int k = 0; k < 16; k++) tile[ty + 4 * k][tx] = v[k];
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; k++) {
        const int i = ty + 4 * k;
        const int64_t r = r0 + tx, c = c0 + i;
        v[k] = (r < n && c < n) ? A[r + c * n] : 0.0;
    }
    double mabs = 0.0, masym = 0.0;
#pragma unroll
    for (int k = 0; k < 16; k++) {
        const int i = ty + 4 * k;
        if (r0 + tx < n && c0 + i < n) {
            const double a = v[k], b = tile[tx][i];
            mabs = fmax(mabs, fmax(fabs(a), fabs(b)));
            const double d = fabs(a - b);
            masym = fmax(masym, d == d ? d : 1.0e300);  // NaN counts as asymmetric
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mabs = fmax(mabs, __shfl_xor_sync(0xffffffffu, mabs, o));
        masym = fmax(masym, __shfl_xor_sync(0xffffffffu, masym, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(out, (unsigned long long)__double_as_longlong(mabs));
        atomicMax(out + 1, (unsigned long long)__double_as_longlong(masym));
    }
}

static void say(eg_message_fn message, void* ctx, const char* fmt, ...) {
    if (!message) return;
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    message(ctx, buf);
}

}  // namespace eg

using namespace eg;

// ================================================================== lifecycle
extern "C" int eg_abi_version(void) { return 1; }

extern "C" const char* eg_last_error(void) { return g_err; }

extern "C" int eg_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

// ------------------------------------------------------------------ multi-GPU plumbing (SURVEY.md section 8(b), 8(e))
// One process, one host thread per GPU (the reference's user calls AM(..., ngpu = ) from a single R session:
// R/AM.R:185-196).  NCCL is bound at run time (dlopen of libnccl.so.2, re-using a copy that is already loaded in the
// process, e.g. the one torch bundles) so that single-GPU users carry no dependency on it.
namespace eg {
typedef struct ncclComm* ncclComm_t;
struct NcclApi {
    void* h = nullptr;
    int (*CommInitAll)(ncclComm_t*, int, const int*) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*Broadcast)(const void*, void*, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;
constexpr int NCCL_INT32 = 2, NCCL_FLOAT64 = 8, NCCL_SUM = 0;   // ncclInt32, ncclFloat64, ncclSum (nccl.h, stable ABI values)

struct WorkerPool {
    std::vector<std::thread> th;
    std::mutex mu;
    std::condition_variable cv, cv_done;
    std::function<int(int)> job;
    uint64_t gen = 0;
    int pending = 0;
    bool stop = false;
    std::vector<int> rc;
    std::vector<std::string> err;
    // agree(): host-side barrier of the GPU threads that ORs their status -- called before every collective so that a
    // failure on one GPU makes all of them skip the exchange instead of leaving the others waiting inside NCCL forever
    int bar_count = 0, bar_gen = 0, bar_rc = EG_OK, bar_result = EG_OK;
};
struct Multi {
    int n = 0;  // 0 / 1: single GPU
    int devs[EG_MAX_GPUS] = {};
    ncclComm_t comm[EG_MAX_GPUS] = {};
    WorkerPool* pool = nullptr;
};
static Multi g_multi;

static void worker_main(int r) {
    t_ctx = &g_ctxs[r];
    t_is_worker = true;
    cudaSetDevice(g_ctxs[r].device);
    WorkerPool& P = *g_multi.pool;
    uint64_t seen = 0;
    for (;;) {
        std::function<int(int)> job;
        {
            std::unique_lock<std::mutex> lk(P.mu);
            P.cv.wait(lk, [&] { return P.stop || P.gen != seen; });
            if (P.stop) return;
            seen = P.gen;
            job = P.job;
        }
        g_err[0] = 0;
        const int rc = job(r);
        {
            std::lock_guard<std::mutex> lk(P.mu);
            P.rc[r] = rc;
            P.err[r] = g_err;
            if (--P.pending == 0) P.cv_done.notify_all();
        }
    }
}
// run fn(r) on the thread of every GPU slot; the first failure (lowest slot) becomes the caller's error
static int run_all(const std::function<int(int)>& fn) {
    WorkerPool& P = *g_multi.pool;
    {
        std::unique_lock<std::mutex> lk(P.mu);
        P.job = fn;
        P.pending = g_multi.n;
        for (int r = 0; r < g_multi.n; r++) P.rc[r] = EG_OK;
        P.gen++;
        P.cv.notify_all();
        P.cv_done.wait(lk, [&] { return P.pending == 0; });
    }
    for (int r = 0; r < g_multi.n; r++)
        if (P.rc[r] != EG_OK) return set_error(P.rc[r], "GPU %d: %s", g_multi.devs[r], P.err[r].c_str());
    return EG_OK;
}
static bool multi_trace() {
    static int on = -1;
    if (on < 0) { const char* e = getenv("EAGLE_MULTI_TRACE"); on = e && e[0] == '1'; }
    return on == 1;
}
#define MTRACE(...) do { if (t_is_worker && multi_trace()) { fprintf(stderr, "[eagle gpu %d] ", g_ctx.device); fprintf(stderr, __VA_ARGS__); fputc('\n', stderr); fflush(stderr); } } while (0)
// Every GPU thread calls agree(my status so far); all return the same value: EG_OK, or the first failure's code.  The
// thread that failed keeps its own message; the others get a short note.  Off the worker threads (a plain store worked on
// by the calling thread as slot 0 of 1, also while a multi-GPU set exists) there is nobody to agree with: rc comes back.
static int agree(int rc) {
    if (!t_is_worker) return rc;
    WorkerPool& P = *g_multi.pool;
    std::unique_lock<std::mutex> lk(P.mu);
    if (rc != EG_OK && P.bar_rc == EG_OK) P.bar_rc = rc;
    const int gen = P.bar_gen;
    if (++P.bar_count == g_multi.n) {
        P.bar_result = P.bar_rc;
        P.bar_rc = EG_OK;
        P.bar_count = 0;
        P.bar_gen++;
        P.cv_done.notify_all();
    } else {
        P.cv_done.wait(lk, [&] { return P.bar_gen != gen; });
    }
    const int res = P.bar_result;
    lk.unlock();
    if (res != EG_OK && rc == EG_OK) return set_error(res, "another GPU of the set failed");
    return rc != EG_OK ? rc : EG_OK;
}
static int check_nccl(int rc, const char* what) {
    if (rc == 0) return EG_OK;
    return set_error(EG_ERR_CUDA, "NCCL error in %s: %s", what, g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
}
#define EG_NCCL(expr) EG_TRY(::eg::check_nccl((expr), #expr))

// contiguous, `align`-aligned split of [0, total) over nparts (the same rule as eagleeverything_b200/dist.py::shard_range)
static void shard_range(int64_t total, int nparts, int r, int64_t align, int64_t* a, int64_t* b) {
    const int64_t blocks = (total + align - 1) / align, base = blocks / nparts, extra = blocks % nparts;
    const int64_t b0 = r * base + (r < extra ? r : extra), b1 = b0 + base + (r < extra ? 1 : 0);
    *a = b0 * align < total ? b0 * align : total;
    *b = b1 * align < total ? b1 * align : total;
}

static int init_slot(Context& c, int device) {
    EG_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    EG_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return set_error(EG_ERR_CUDA, "device %d is sm_%d%d; this library contains sm_100a code only", device,
                         prop.major, prop.minor);
    c.sms = prop.multiProcessorCount;
    EG_CUDA(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    EG_CUDA(cudaStreamCreateWithFlags(&c.copy_stream, cudaStreamNonBlocking));
    if (cublasCreate(&c.cublas) != CUBLAS_STATUS_SUCCESS) return set_error(EG_ERR_CUDA, "cublasCreate failed");
    EG_CUDA(cudaMalloc(&c.d_err, 4 * sizeof(int32_t)));
    {   // keep freed blocks in the pool instead of returning them to the driver at every synchronisation
        cudaMemPool_t pool;
        EG_CUDA(cudaDeviceGetDefaultMemPool(&pool, device));
        uint64_t keep = UINT64_MAX;
        EG_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    }
    {   // recycle at most half of the device memory (EAGLE_GPU_RECYCLE_GB overrides; 0 switches the list off)
        size_t free_b = 0, total_b = 0;
        EG_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const char* env = getenv("EAGLE_GPU_RECYCLE_GB");
        c.recycle_limit = env ? (size_t)(atof(env) * 1e9) : total_b / 2;
    }
    c.device = device;
    c.ready = true;
    return EG_OK;
}
// the calling thread's workspaces of the other translation units (thread-local: each thread releases its own)
static void release_workspaces() {
    syrk_release_cache();
    scan_i8_release();
    prep_i8_release();
    algebra_release();
    eigbasis_release();
    hostio_release();
}
// runs on the thread that owns the slot (its thread-local workspaces are released with it)
static void shutdown_slot() {
    if (!g_ctx.ready) return;
    cudaSetDevice(g_ctx.device);
    cudaDeviceSynchronize();
    eg_cache_clear();
    release_workspaces();
    if (g_ctx.scan_ev[0]) { cudaEventDestroy(g_ctx.scan_ev[0]); cudaEventDestroy(g_ctx.scan_ev[1]); }
    if (g_ctx.cublas) cublasDestroy(g_ctx.cublas);
    if (g_ctx.stream) cudaStreamDestroy(g_ctx.stream);
    if (g_ctx.copy_stream) cudaStreamDestroy(g_ctx.copy_stream);
    if (g_ctx.d_err) cudaFree(g_ctx.d_err);
    g_ctx.reset();
}
static int check_devices(int* ndev_out) {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_error(EG_ERR_CUDA, "no usable CUDA device (%s); libeaglegpu has no CPU fallback",
                         e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    *ndev_out = ndev;
    return EG_OK;
}

// ------------------------------------------------------------------ marker-sharded (composite) stores
// part r of a composite store; runs on the thread of GPU slot r (the part's memory belongs to that slot's pool)
static void free_part(eg_store* S, int r) {
    eg_store* p = S->part[r];
    if (!p) return;
    pool_free(p->C32);
    pool_free(p->d);
    delete p;
    S->part[r] = nullptr;
}
static void free_store_tree(eg_store* s) {
    if (!s) return;
    if (s->nparts > 1) {
        if (g_multi.n > 1 && g_multi.pool && !t_is_worker) run_all([s](int r) { free_part(s, r); return EG_OK; });
        delete s;
        return;
    }
    pool_free(s->C32);
    pool_free(s->d);
    delete s;
}
static eg_store* new_composite(int64_t rows, int64_t cols, bool kblocked) {
    eg_store* S = new eg_store();
    S->rows = rows;
    S->cols = cols;
    S->pitch = kblocked ? 0 : store_pitch(cols);
    S->nparts = g_multi.n;
    S->mt_orientation = !kblocked;
    const int64_t markers = kblocked ? cols : rows;
    for (int r = 0; r < g_multi.n; r++) {
        int64_t a, b;
        shard_range(markers, g_multi.n, r, 128, &a, &b);
        S->off[r] = a;
        S->off[r + 1] = b;
    }
    return S;
}
// run_all with eviction on the orchestrating thread: when a GPU runs out of memory, drop one unheld cached store and retry
static int run_all_evicting(const std::function<int(int)>& fn, const std::function<void()>& undo) {
    for (;;) {
        const int rc = run_all(fn);
        if (rc != EG_ERR_ALLOC) return rc;
        const std::string msg = g_err;
        if (undo) undo();
        if (!cache_evict_one()) return set_error(EG_ERR_ALLOC, "%s", msg.c_str());
    }
}
// Rows [row0,row1) x columns [col0,col1) of a host image -> a store; with a multi-GPU set (and allow_multi) a composite
// whose parts are the marker shards, every GPU pulling and decoding its own byte ranges concurrently.
static int store_from_image_any(const uint8_t* image, int64_t cols_total, int64_t row0, int64_t row1, int64_t col0,
                                int64_t col1, bool kblocked, eg_store** out, bool allow_multi, int fd) {
    if (g_multi.n <= 1 || !allow_multi || t_is_worker) return store_from_image(image, cols_total, row0, row1, col0, col1, kblocked, out, fd);
    EG_TRY(ensure_init());
    if (!image || row1 <= row0 || col1 <= col0 || col0 < 0 || col1 > cols_total || row0 < 0)
        return set_error(EG_ERR_ARG, "genotype store: bad image range");
    eg_store* S = new_composite(row1 - row0, col1 - col0, kblocked);
    auto undo = [S]() { run_all([S](int r) { free_part(S, r); return EG_OK; }); };
    const int rc = run_all_evicting([&](int r) -> int {
        const int64_t a = S->off[r], b = S->off[r + 1];
        if (a == b) return EG_OK;
        return kblocked ? store_from_image(image, cols_total, row0, row1, col0 + a, col0 + b, true, &S->part[r], fd)
                        : store_from_image(image, cols_total, row0 + a, row0 + b, col0, col1, false, &S->part[r], fd);
    }, undo);
    if (rc != EG_OK) {
        const std::string msg = g_err;
        undo();
        delete S;
        return set_error(rc, "%s", msg.c_str());
    }
    g_ctx.timing[0] = 0;
    for (int r = 0; r < g_multi.n; r++) g_ctx.timing[0] = std::max(g_ctx.timing[0], g_ctxs[r].timing[0]);
    *out = S;
    return EG_OK;
}

// ------------------------------------------------------------------ compute helpers on stores
// A plain store is worked on as slot 0 of 1 on the calling thread, a composite one by every GPU slot on its own thread.
static const eg_store* slot_part(const eg_store* S, int r) { return S->nparts > 1 ? S->part[r] : S; }
static int on_each_slot(const eg_store* S, const std::function<int(int)>& fn) { return S->nparts > 1 ? run_all(fn) : fn(0); }
// the entries of `idx` (markers of the whole store) that slot r holds, relative to its first marker
static std::vector<int64_t> slot_indices(const eg_store* S, int r, const std::vector<int64_t>& idx) {
    if (S->nparts <= 1) return idx;
    std::vector<int64_t> z;
    for (int64_t c : idx)
        if (c >= S->off[r] && c < S->off[r + 1]) z.push_back(c - S->off[r]);
    return z;
}

// Partial product of one plain store into C (n x n int32, zeroed / overwritten here), zeroed columns corrected.
// keep_product: cache the int32 product with the store (stores of the path cache: calculateMMt_rcpp is called again by
// SummaryAM with other selected loci, R/summary_am.R:142 -- the repeat then costs a copy, the rank-k correction and the
// finalize pass instead of a second contraction)
static int partial_product(const eg_store* M, const std::vector<int64_t>& zero_cols, DevBuf& C, bool keep_product) {
    const int64_t n = M->rows;
    cudaStream_t st = g_ctx.stream;
    EG_TRY(C.alloc((size_t)n * n * sizeof(int32_t), "MMt int32 accumulator"));
    const char* envk = getenv("EAGLE_KEEP_PRODUCT");   // "0": contract again on every call (bench.py's steady-state leg)
    const bool reuse = !(envk && envk[0] == '0');
    if (M->C32 && reuse) {  // accumulated under the upload (store_from_image_kb): keep it intact for later calls
        EG_CUDA(cudaMemcpyAsync(C.p, M->C32, (size_t)n * n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
        g_ctx.timing[1] = 0.0;
    } else {
        EG_CUDA(cudaMemsetAsync(C.p, 0, (size_t)n * n * sizeof(int32_t), st));
        Timer t(st);
        EG_TRY(M->pitch ? eg_dev_syrk_i8(M->d, n, M->cols, M->pitch, C.as<int32_t>(), n, st)
                        : eg_dev_syrk_i8_kb(M->d, n, M->cols, C.as<int32_t>(), n, st));
        g_ctx.timing[1] = t.stop();
        if (keep_product && reuse && !M->C32) {
            int32_t* keep = nullptr;
            if (pool_alloc((void**)&keep, (size_t)n * n * sizeof(int32_t)) == cudaSuccess) {
                EG_CUDA(cudaMemcpyAsync(keep, C.p, (size_t)n * n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
                const_cast<eg_store*>(M)->C32 = keep;
            } else {
                cudaGetLastError();  // no room: contract again next time
            }
        }
    }
    if (!zero_cols.empty())
        EG_TRY(eg_dev_syrk_zero_cols(M->d, n, M->pitch, zero_cols.data(), (int64_t)zero_cols.size(), C.as<int32_t>(), n, st));
    return EG_OK;
}

// M.Mt, slot r of N: the slot contracts its marker shard; with several GPUs ONE int32 all-reduce (exact, order-free) over
// NVLink follows; every slot finalizes and returns its own block of rows of K to the host (the n x n result crosses PCIe
// once, in parallel).
static int mmt_slot(const eg_store* M, int r, const std::vector<int64_t>& zero_cols, double* out_host, bool keep_product) {
    const int64_t n = M->rows;
    const int N = M->nparts > 1 ? M->nparts : 1;
    cudaStream_t st = g_ctx.stream;
    DevBuf C, D;
    const eg_store* part = slot_part(M, r);
    auto local = [&]() -> int {
        if (part) {
            EG_TRY(partial_product(part, slot_indices(M, r, zero_cols), C, keep_product));
        } else {   // no markers on this GPU: zeros into the all-reduce
            EG_TRY(C.alloc((size_t)n * n * sizeof(int32_t), "MMt int32 accumulator"));
            EG_CUDA(cudaMemsetAsync(C.p, 0, (size_t)n * n * sizeof(int32_t), st));
        }
        return D.alloc((size_t)n * n * sizeof(double), "MMt output");
    };
    MTRACE("mmt: partial product of markers [%lld, %lld)", (long long)M->off[r], (long long)M->off[r + 1]);
    EG_TRY(agree(local()));
    {   // timing slot 2: the all-reduce with several GPUs, the finalize with one
        Timer t(st);
        if (N > 1) {
            MTRACE("mmt: all-reduce of %lld x %lld int32", (long long)n, (long long)n);
            EG_NCCL(g_nccl.AllReduce(C.p, C.p, (size_t)n * n, NCCL_INT32, NCCL_SUM, g_multi.comm[r], st));
        } else {
            EG_TRY(eg_dev_mmt_finalize(C.as<int32_t>(), n, n, D.as<double>(), st));
        }
        g_ctx.timing[2] = t.stop();
    }
    if (N > 1) EG_TRY(eg_dev_mmt_finalize(C.as<int32_t>(), n, n, D.as<double>(), st));
    int64_t i0, i1;
    shard_range(n, N, r, 1, &i0, &i1);
    Timer t(st);
    if (i1 > i0) EG_TRY(d2h_staged(out_host + i0 * n, D.as<double>() + i0 * n, (size_t)(i1 - i0) * n * sizeof(double), st));
    EG_CUDA(cudaStreamSynchronize(st));
    g_ctx.timing[3] = t.stop();
    MTRACE("mmt: done");
    return EG_OK;
}
static int mmt_of_store(const eg_store* M, const std::vector<int64_t>& zero_cols, double* out_host, bool keep_product = false) {
    Pin pin(M);
    return on_each_slot(M, [&](int r) { return mmt_slot(M, r, zero_cols, out_host, keep_product); });
}

// The scan, slot r of N.  S and V cross PCIe once: slot r uploads columns [k0_r, k1_r) of each and, with several GPUs, the
// blocks are exchanged over NVLink (one grouped broadcast); when the pre-products take the digit-slice path the columns of
// W = S (V S) are split over the GPUs at equal cost and exchanged the same way; every slot scans its own markers and writes
// its slice of a / var(a) straight into the caller's vectors.  With one slot the cuts are [0, n) and the steps are those of
// eg_dev_scan_prepare: symmetry check, zeroed Wp, all columns of W, fold.
static int scan_slot(const eg_store* Mt, int r, const std::vector<int64_t>& zero_rows, const double* S, const double* V,
                     const double* a, double* out_a, double* out_vara) {
    const int64_t n = Mt->cols;
    const int N = Mt->nparts > 1 ? Mt->nparts : 1;
    const int64_t Kpad = round_up(n, 32);
    cudaStream_t st = g_ctx.stream;
    const eg_store* part = slot_part(Mt, r);
    const int64_t L = part ? part->rows : 0;
    DevBuf dS, dV, da, dT, dW, oa, ov;
    auto alloc = [&]() -> int {
        EG_TRY(dS.alloc((size_t)n * n * 8, "inv_MMt_sqrt"));
        EG_TRY(dV.alloc((size_t)n * n * 8, "dim_reduced_vara"));
        EG_TRY(da.alloc((size_t)n * 8, "a"));
        EG_TRY(dW.alloc((size_t)eg_scan_wp_elems(n) * 8, "packed W"));
        EG_TRY(oa.alloc((size_t)(L ? L : 1) * 8, "a out"));
        return ov.alloc((size_t)(L ? L : 1) * 8, "vara out");
    };
    const int rc_alloc = alloc();
    Timer t_up(st);
    auto upload = [&]() -> int {
        EG_TRY(rc_alloc);
        int64_t k0, k1;
        shard_range(n, N, r, 1, &k0, &k1);
        if (k1 > k0) {   // R-owned (pageable) matrices: page-locked ring, parallel copiers
            EG_TRY(h2d_staged(dS.as<double>() + k0 * n, S + k0 * n, (size_t)(k1 - k0) * n * 8, st));
            EG_TRY(h2d_staged(dV.as<double>() + k0 * n, V + k0 * n, (size_t)(k1 - k0) * n * 8, st));
        }
        EG_CUDA(cudaMemcpyAsync(da.p, a, (size_t)n * 8, cudaMemcpyHostToDevice, st));
        return EG_OK;
    };
    MTRACE("scan: upload of 1/%d of S and V", N);
    EG_TRY(agree(upload()));
    if (N > 1) {
        EG_NCCL(g_nccl.GroupStart());
        for (int q = 0; q < N; q++) {
            int64_t q0, q1;
            shard_range(n, N, q, 1, &q0, &q1);
            if (q1 == q0) continue;
            EG_NCCL(g_nccl.Broadcast(dS.as<double>() + q0 * n, dS.as<double>() + q0 * n, (size_t)(q1 - q0) * n, NCCL_FLOAT64, q, g_multi.comm[r], st));
            EG_NCCL(g_nccl.Broadcast(dV.as<double>() + q0 * n, dV.as<double>() + q0 * n, (size_t)(q1 - q0) * n, NCCL_FLOAT64, q, g_multi.comm[r], st));
        }
        EG_NCCL(g_nccl.GroupEnd());
    }
    g_ctx.timing[4] = t_up.stop();
    Timer t_prep(st);
    int sym = 0;
    bool split = false;
    std::vector<int64_t> cuts(N + 1, n);
    auto products = [&]() -> int {
        EG_TRY(eg_dev_inputs_symmetric(dS.as<double>(), dV.as<double>(), n, &sym, st));
        split = sym && eg_prep_uses_i8(n);   // otherwise every GPU computes all of W itself (bit-identical to one GPU)
        for (int q = 0; q < N; q++) {
            if (split) {   // cost of columns [0,c): n c (V S) + c^2 / 2 (upper part of S X)  ->  equal-cost cuts
                int64_t c = (int64_t)llround((double)n * (sqrt(1.0 + 3.0 * q / N) - 1.0) / 32.0) * 32;
                cuts[q] = c < n ? c : n;
            } else {
                cuts[q] = q == 0 ? 0 : n;
            }
        }
        int64_t widest = 1;
        for (int q = 0; q < N; q++) widest = std::max(widest, cuts[q + 1] - cuts[q]);
        EG_TRY(dT.alloc((size_t)n * (split ? widest : n) * 8, "scan scratch"));
        EG_CUDA(cudaMemsetAsync(dW.p, 0, (size_t)eg_scan_wp_elems(n) * 8, st));
        return eg_dev_scan_prepare_cols(dS.as<double>(), dV.as<double>(), n, split ? cuts[r] : 0, split ? cuts[r + 1] : n, sym,
                                        dT.as<double>(), dW.as<double>(), st);
    };
    MTRACE("scan: pre-products of my columns of W");
    EG_TRY(agree(products()));
    if (N > 1) {
        EG_NCCL(g_nccl.GroupStart());
        for (int q = 0; q < N && split; q++)
            if (cuts[q + 1] > cuts[q])
                EG_NCCL(g_nccl.Broadcast(dW.as<double>() + cuts[q] * Kpad, dW.as<double>() + cuts[q] * Kpad,
                                         (size_t)(cuts[q + 1] - cuts[q]) * Kpad, NCCL_FLOAT64, q, g_multi.comm[r], st));
        EG_NCCL(g_nccl.GroupEnd());
    }
    EG_TRY(eg_dev_scan_fold(dS.as<double>(), da.as<double>(), n, sym, dW.as<double>(), st));
    g_ctx.timing[5] = t_prep.stop();
    MTRACE("scan: %lld markers", (long long)L);
    if (L > 0) {
        const std::vector<int64_t> z = slot_indices(Mt, r, zero_rows);
        {
            Timer t(st);
            EG_TRY(eg_dev_scan(part->d, L, n, part->pitch, dW.as<double>(), z.empty() ? nullptr : z.data(), (int64_t)z.size(),
                               oa.as<double>(), ov.as<double>(), st));
            g_ctx.timing[6] = t.stop();
        }
        Timer t(st);   // off[0] is 0 for every store, so a plain store's results start at out_a[0]
        EG_CUDA(cudaMemcpyAsync(out_a + Mt->off[r], oa.p, (size_t)L * 8, cudaMemcpyDeviceToHost, st));
        EG_CUDA(cudaMemcpyAsync(out_vara + Mt->off[r], ov.p, (size_t)L * 8, cudaMemcpyDeviceToHost, st));
        EG_CUDA(cudaStreamSynchronize(st));
        g_ctx.timing[7] = t.stop();
    } else {
        EG_CUDA(cudaStreamSynchronize(st));
    }
    MTRACE("scan: done");
    return EG_OK;
}
static int scan_of_store(const eg_store* Mt, const std::vector<int64_t>& zero_rows, const double* S, const double* V,
                         const double* a, double* out_a, double* out_vara) {
    if (!Mt->pitch)
        return set_error(EG_ERR_ARG, "the scan needs an Mt store (markers as rows); transpose the M store first");
    Pin pin(Mt);
    return on_each_slot(Mt, [&](int r) { return scan_slot(Mt, r, zero_rows, S, V, a, out_a, out_vara); });
}
}  // namespace eg

extern "C" int eg_init(int device) {
    if (g_multi.n <= 1 && g_ctxs[0].ready && g_ctxs[0].device == device) return check_cuda(cudaSetDevice(device), "cudaSetDevice");
    if (g_ctxs[0].ready || g_multi.n > 1) eg_shutdown();
    int ndev = 0;
    EG_TRY(check_devices(&ndev));
    if (device < 0 || device >= ndev) return set_error(EG_ERR_ARG, "eg_init: device %d of %d", device, ndev);
    t_ctx = &g_ctxs[0];
    return init_slot(g_ctxs[0], device);
}

// eg_init_multi(ngpu, devs): the marker-sharded form.  devs == NULL: devices 0 .. ngpu-1.
extern "C" int eg_init_multi(int ngpu, const int* devs) {
    if (ngpu < 1 || ngpu > EG_MAX_GPUS) return set_error(EG_ERR_ARG, "eg_init_multi: ngpu = %d (1 .. %d)", ngpu, EG_MAX_GPUS);
    if (ngpu == 1) return eg_init(devs ? devs[0] : 0);
    bool same = g_multi.n == ngpu;
    for (int r = 0; same && r < ngpu; r++) same = g_multi.devs[r] == (devs ? devs[r] : r);
    if (same) return check_cuda(cudaSetDevice(g_multi.devs[0]), "cudaSetDevice");
    if (g_ctxs[0].ready || g_multi.n > 1) eg_shutdown();
    int ndev = 0;
    EG_TRY(check_devices(&ndev));
    for (int r = 0; r < ngpu; r++) {
        const int d = devs ? devs[r] : r;
        if (d < 0 || d >= ndev) return set_error(EG_ERR_ARG, "eg_init_multi: device %d of %d", d, ndev);
        for (int q = 0; q < r; q++)
            if ((devs ? devs[q] : q) == d) return set_error(EG_ERR_ARG, "eg_init_multi: device %d listed twice", d);
    }
    if (!g_nccl.h) {
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);   // a copy already in the process (torch's) wins
        if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
        if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
        if (!h) return set_error(EG_ERR_CUDA, "eg_init_multi: libnccl.so.2 not found (%s)", dlerror());
        g_nccl.h = h;
        *(void**)&g_nccl.CommInitAll = dlsym(h, "ncclCommInitAll");
        *(void**)&g_nccl.CommDestroy = dlsym(h, "ncclCommDestroy");
        *(void**)&g_nccl.AllReduce = dlsym(h, "ncclAllReduce");
        *(void**)&g_nccl.Broadcast = dlsym(h, "ncclBroadcast");
        *(void**)&g_nccl.GroupStart = dlsym(h, "ncclGroupStart");
        *(void**)&g_nccl.GroupEnd = dlsym(h, "ncclGroupEnd");
        *(void**)&g_nccl.GetErrorString = dlsym(h, "ncclGetErrorString");
        if (!g_nccl.CommInitAll || !g_nccl.CommDestroy || !g_nccl.AllReduce || !g_nccl.Broadcast || !g_nccl.GroupStart || !g_nccl.GroupEnd)
            return set_error(EG_ERR_CUDA, "eg_init_multi: libnccl.so.2 lacks a required symbol");
    }
    for (int r = 0; r < ngpu; r++) {
        g_multi.devs[r] = devs ? devs[r] : r;
        int rc = init_slot(g_ctxs[r], g_multi.devs[r]);
        if (rc != EG_OK) {
            g_multi.n = 0;
            return rc;
        }
    }
    {
        const int nrc = g_nccl.CommInitAll(g_multi.comm, ngpu, g_multi.devs);
        if (nrc != 0) {   // leave nothing half-built behind
            const int rc = check_nccl(nrc, "ncclCommInitAll");
            const std::string msg = g_err;
            for (int r = 0; r < ngpu; r++) {
                t_ctx = &g_ctxs[r];
                shutdown_slot();
            }
            t_ctx = &g_ctxs[0];
            return set_error(rc, "%s", msg.c_str());
        }
    }
    g_multi.n = ngpu;
    g_multi.pool = new WorkerPool();
    g_multi.pool->rc.assign(ngpu, EG_OK);
    g_multi.pool->err.assign(ngpu, std::string());
    for (int r = 0; r < ngpu; r++) g_multi.pool->th.emplace_back(worker_main, r);
    t_ctx = &g_ctxs[0];
    return check_cuda(cudaSetDevice(g_multi.devs[0]), "cudaSetDevice");
}
extern "C" int eg_gpu_count(void) { return g_multi.n > 1 ? g_multi.n : (g_ctxs[0].ready ? 1 : 0); }

extern "C" void eg_cache_clear(void) {
    for (auto& e : g_ctx.cache) free_store_tree(e.store);
    g_ctx.cache.clear();
    // hand the recycled memory back to the driver; called by the user with a multi-GPU set: the parts' pools live on the workers
    if (g_multi.n > 1 && !t_is_worker && g_multi.pool)
        run_all([](int) { pool_give_back(); return EG_OK; });
    else
        pool_give_back();
}

extern "C" int eg_shutdown(void) {
    if (g_multi.n > 1) {
        t_ctx = &g_ctxs[0];
        eg_cache_clear();   // composite stores: parts are freed on their own threads
        // the calling thread's own workspaces on device 0 (single-GPU entry points it ran itself)
        cudaSetDevice(g_ctxs[0].device);
        release_workspaces();
        run_all([](int r) {
            if (g_multi.comm[r]) g_nccl.CommDestroy(g_multi.comm[r]);
            g_multi.comm[r] = nullptr;
            shutdown_slot();
            return EG_OK;
        });
        {
            std::lock_guard<std::mutex> lk(g_multi.pool->mu);
            g_multi.pool->stop = true;
            g_multi.pool->cv.notify_all();
        }
        for (auto& t : g_multi.pool->th) t.join();
        delete g_multi.pool;
        g_multi.pool = nullptr;
        g_multi.n = 0;
        return EG_OK;
    }
    t_ctx = &g_ctxs[0];
    shutdown_slot();
    return EG_OK;
}

extern "C" int eg_set_scan_mode(int mode) {
    if (mode != 0 && mode != 1) return set_error(EG_ERR_ARG, "eg_set_scan_mode: 0 (FP64 DMMA) or 1 (exact int8 slices)");
    g_scan_mode = mode;
    return EG_OK;
}
extern "C" int eg_get_scan_mode(void) { return scan_mode(); }
namespace eg {
int scan_i8_digits();
void scan_i8_set_digits(int d);
}
extern "C" int eg_set_scan_digits(int digits) {
    if (digits != 6 && digits != 7) return set_error(EG_ERR_ARG, "eg_set_scan_digits: 6 or 7 balanced base-256 digits per column");
    scan_i8_set_digits(digits);
    return EG_OK;
}
extern "C" int eg_get_scan_digits(void) { return scan_i8_digits(); }

namespace eg {
// CUDA events around the dominant scan kernel of the last eg_dev_scan call (for roofline reporting)
void scan_kernel_mark(int which, cudaStream_t st, double ops) {
    if (!g_ctx.scan_ev[0]) {
        cudaEventCreate(&g_ctx.scan_ev[0]);
        cudaEventCreate(&g_ctx.scan_ev[1]);
    }
    cudaEventRecord(g_ctx.scan_ev[which], st);
    if (which == 0) g_ctx.scan_ops = ops;
}
}  // namespace eg
extern "C" int eg_last_scan_kernel(double* ms, double* ops) {
    if (!g_ctx.scan_ev[0] || !ms || !ops) return set_error(EG_ERR_ARG, "eg_last_scan_kernel: no scan has run");
    EG_CUDA(cudaEventSynchronize(g_ctx.scan_ev[1]));
    float f = 0;
    EG_CUDA(cudaEventElapsedTime(&f, g_ctx.scan_ev[0], g_ctx.scan_ev[1]));
    *ms = f;
    *ops = g_ctx.scan_ops;
    return EG_OK;
}

extern "C" long long eg_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

namespace eg {
void prep_kernel_times(double* ms, double* ops);
}
extern "C" int eg_last_prep_kernels(double* ms, double* ops) {
    if (!ms || !ops) return set_error(EG_ERR_ARG, "eg_last_prep_kernels: null");
    prep_kernel_times(ms, ops);
    return EG_OK;
}

extern "C" int eg_last_timing(double* out_ms, int n_out) {
    if (!out_ms) return set_error(EG_ERR_ARG, "eg_last_timing: null");
    for (int i = 0; i < n_out && i < 8; i++) out_ms[i] = g_ctx.timing[i];
    return EG_OK;
}

// ================================================================== stores
extern "C" int eg_store_from_host_ascii(const uint8_t* image, int64_t rows, int64_t cols, int64_t col0, int64_t col1,
                                        eg_store_t** out) {
    if (!out) return set_error(EG_ERR_ARG, "null out");
    return store_from_image_any(image, cols, 0, rows, col0, col1, true, out, true);  // M orientation: K-blocked
}
extern "C" int eg_store_from_host_ascii_rows(const uint8_t* image, int64_t rows, int64_t cols, int64_t row0,
                                             int64_t row1, eg_store_t** out) {
    if (!out || row1 > rows) return set_error(EG_ERR_ARG, "bad row range");
    return store_from_image_any(image, cols, row0, row1, 0, cols, false, out, true);  // Mt orientation: row-major
}
// ------------------------------------------------------------------ packed 2-bit container (pack2.cu)
// Host words in, K-blocked (M orientation) or row-major (Mt orientation) store out: one H2D copy of the whole (4x smaller
// than the store) rows*wpr*8 bytes, then the unpack kernel writes the store in its layout.
extern "C" int eg_store_from_host_packed(const uint64_t* words, int64_t rows, int64_t cols, int kblocked, eg_store_t** out) {
    if (!words || !out || rows <= 0 || cols <= 0) return set_error(EG_ERR_ARG, "eg_store_from_host_packed: bad argument");
    EG_TRY(ensure_init());
    const int64_t wpr = eg_packed_words_per_row(cols);
    eg_store* s = nullptr;
    EG_TRY(store_alloc(rows, cols, kblocked != 0, &s));
    DevBuf w;
    int rc = w.alloc((size_t)rows * wpr * 8, "packed genotype words");
    Timer total(g_ctx.stream);
    if (rc == EG_OK) rc = check_cuda(cudaMemcpyAsync(w.p, words, (size_t)rows * wpr * 8, cudaMemcpyHostToDevice, g_ctx.stream), "H2D of the packed genotypes");
    if (rc == EG_OK) rc = check_cuda(cudaMemsetAsync(g_ctx.d_err, 0, 4 * sizeof(int32_t), g_ctx.stream), "memset");
    if (rc == EG_OK) rc = eg_dev_unpack_2bit(w.as<uint64_t>(), rows, cols, s->d, s->pitch, g_ctx.d_err, g_ctx.stream);  // pitch 0: K-blocked
    int32_t h_err[4] = {0, 0, 0, 0};
    if (rc == EG_OK) rc = check_cuda(cudaMemcpyAsync(h_err, g_ctx.d_err, sizeof(h_err), cudaMemcpyDeviceToHost, g_ctx.stream), "status D2H");
    if (rc == EG_OK) rc = check_cuda(cudaStreamSynchronize(g_ctx.stream), "unpack");
    g_ctx.timing[0] = total.stop();
    if (rc == EG_OK && h_err[0])
        rc = set_error(EG_ERR_FORMAT, "packed genotype container: code 3 or stray bits near row %lld, column %lld",
                       (long long)(((int64_t)h_err[3] << 31) | h_err[1]), (long long)h_err[2]);
    return finish_store(rc, s, out);
}
// store -> host words (rows * eg_packed_words_per_row(cols) uint64): what an ingest step writes to disk once
extern "C" int eg_store_to_host_packed(const eg_store_t* s, uint64_t* out_words) {
    if (!s || !out_words) return set_error(EG_ERR_ARG, "eg_store_to_host_packed: bad argument");
    if (s->nparts > 1) return set_error(EG_ERR_ARG, "eg_store_to_host_packed: the store is sharded over several GPUs");
    EG_TRY(ensure_init());
    const int64_t wpr = eg_packed_words_per_row(s->cols);
    DevBuf w;
    EG_TRY(w.alloc((size_t)s->rows * wpr * 8, "packed genotype words"));
    EG_TRY(eg_dev_pack_2bit(s->d, s->rows, s->cols, s->pitch, w.as<uint64_t>(), g_ctx.stream));
    EG_CUDA(cudaMemcpyAsync(out_words, w.p, (size_t)s->rows * wpr * 8, cudaMemcpyDeviceToHost, g_ctx.stream));
    return check_cuda(cudaStreamSynchronize(g_ctx.stream), "pack D2H");
}

// ------------------------------------------------------------------ ReshapeM on resident stores
// Drops the individuals `idx` (0-based, any order, duplicates ignored): rows of an M store (individuals_are_rows != 0)
// or columns of an Mt store.  reference: src/ReshapeM_rcpp.cpp:59-109 (which rewrites both ASCII files).
extern "C" int eg_store_drop_individuals(const eg_store_t* in, const int64_t* idx, int64_t k, int individuals_are_rows,
                                         eg_store_t** out) {
    if (!in || !out || k < 0 || (k > 0 && !idx)) return set_error(EG_ERR_ARG, "eg_store_drop_individuals: bad argument");
    if (in->nparts > 1) return set_error(EG_ERR_ARG, "eg_store_drop_individuals: the store is sharded over several GPUs");
    Pin pin_in(in);
    EG_TRY(ensure_init());
    const int64_t n_in = individuals_are_rows ? in->rows : in->cols;
    std::vector<char> drop((size_t)n_in, 0);
    for (int64_t i = 0; i < k; i++) {
        if (idx[i] < 0 || idx[i] >= n_in)
            return set_error(EG_ERR_ARG, "ReshapeM: individual %lld is outside 0..%lld", (long long)idx[i], (long long)n_in - 1);
        drop[(size_t)idx[i]] = 1;
    }
    std::vector<int64_t> map;
    for (int64_t i = 0; i < n_in; i++)
        if (!drop[(size_t)i]) map.push_back(i);
    if (map.empty()) return set_error(EG_ERR_ARG, "ReshapeM: no individual left");
    if (!individuals_are_rows && in->pitch == 0)
        return set_error(EG_ERR_ARG, "ReshapeM: dropping columns needs a row-major (Mt orientation) store");
    DevBuf dm;
    EG_TRY(dm.alloc(map.size() * sizeof(int64_t), "ReshapeM index map"));
    EG_CUDA(cudaMemcpyAsync(dm.p, map.data(), map.size() * sizeof(int64_t), cudaMemcpyHostToDevice, g_ctx.stream));
    eg_store* s = nullptr;
    const int64_t n_out = (int64_t)map.size();
    int rc;
    if (individuals_are_rows) {
        EG_TRY(store_alloc(n_out, in->cols, in->pitch == 0, &s));
        rc = eg_dev_gather_rows(in->d, in->rows, in->cols, in->pitch, dm.as<int64_t>(), n_out, s->d, s->pitch, g_ctx.stream);
    } else {
        EG_TRY(store_alloc(in->rows, n_out, false, &s));
        rc = eg_dev_gather_cols(in->d, in->rows, in->pitch, dm.as<int64_t>(), n_out, s->d, s->pitch, g_ctx.stream);
    }
    if (rc == EG_OK) rc = check_cuda(cudaStreamSynchronize(g_ctx.stream), "ReshapeM gather");  // `map` goes out of scope
    return finish_store(rc, s, out);
}

extern "C" int eg_store_from_file(const char* path, int64_t rows, int64_t cols, int64_t col0, int64_t col1,
                                  eg_store_t** out) {
    if (!out || !path) return set_error(EG_ERR_ARG, "null argument");
    MappedFile f;
    EG_TRY(f.open_ro(path));
    EG_TRY(check_image_size(f, path, rows, cols));
    return store_from_image_any(f.p, cols, 0, rows, col0, col1, true, out, true, f.fd);
}
extern "C" int eg_store_transpose(const eg_store_t* in, eg_store_t** out) {
    if (!in || !out) return set_error(EG_ERR_ARG, "null argument");
    EG_TRY(ensure_init());
    Pin pin(in);
    if (in->nparts > 1) {   // marker shards transpose in place: part r (n x L_r) -> (L_r x n), no exchange
        if (in->mt_orientation) return set_error(EG_ERR_ARG, "eg_store_transpose: sharded Mt stores are not transposed back");
        eg_store* S = new_composite(in->cols, in->rows, false);
        for (int r = 0; r <= in->nparts; r++) S->off[r] = in->off[r];
        auto undo = [S]() { run_all([S](int r) { free_part(S, r); return EG_OK; }); };
        const int rc = run_all_evicting([&](int r) -> int {
            const eg_store* p = in->part[r];
            if (!p) return EG_OK;
            EG_TRY(store_alloc(p->cols, p->rows, false, &S->part[r]));
            EG_TRY(eg_dev_transpose_kb_i8(p->d, p->rows, p->cols, S->part[r]->d, S->part[r]->pitch, g_ctx.stream));
            return check_cuda(cudaStreamSynchronize(g_ctx.stream), "transpose");
        }, undo);
        if (rc != EG_OK) {
            const std::string msg = g_err;
            undo();
            delete S;
            return set_error(rc, "%s", msg.c_str());
        }
        *out = S;
        return EG_OK;
    }
    eg_store* s = nullptr;
    EG_TRY(store_alloc(in->cols, in->rows, false, &s));  // the transpose is always a row-major (Mt-type) store
    int rc = in->pitch ? eg_dev_transpose_i8(in->d, in->rows, in->cols, in->pitch, s->d, s->pitch, g_ctx.stream)
                       : eg_dev_transpose_kb_i8(in->d, in->rows, in->cols, s->d, s->pitch, g_ctx.stream);
    if (rc == EG_OK) rc = check_cuda(cudaStreamSynchronize(g_ctx.stream), "transpose");
    return finish_store(rc, s, out);
}
extern "C" int eg_store_free(eg_store_t* s) {
    if (!s) return EG_OK;
    free_store_tree(s);
    return EG_OK;
}
extern "C" int eg_store_info(const eg_store_t* s, int64_t* rows, int64_t* cols, int64_t* pitch, void** device_ptr) {
    if (!s) return set_error(EG_ERR_ARG, "null store");
    if (rows) *rows = s->rows;
    if (cols) *cols = s->cols;
    if (pitch) *pitch = s->pitch;
    if (device_ptr) *device_ptr = s->d;   // NULL for a store sharded over several GPUs
    return EG_OK;
}
extern "C" int eg_store_mmt(const eg_store_t* M, const int64_t* zero_cols, int64_t n_zero, double* out_MMt_host) {
    if (!M || !out_MMt_host || n_zero < 0) return set_error(EG_ERR_ARG, "eg_store_mmt: bad argument");
    EG_TRY(ensure_init());
    std::vector<int64_t> z;
    for (int64_t i = 0; i < n_zero; i++) {
        if (zero_cols[i] < 0 || zero_cols[i] >= M->cols) return set_error(EG_ERR_ARG, "zero column out of range");
        z.push_back(zero_cols[i]);
    }
    return mmt_of_store(M, z, out_MMt_host);
}
extern "C" int eg_store_a_and_vara(const eg_store_t* Mt, const int64_t* zero_rows, int64_t n_zero,
                                   const double* inv_MMt_sqrt, const double* dim_reduced_vara, const double* a,
                                   double* out_a, double* out_vara) {
    if (!Mt || !inv_MMt_sqrt || !dim_reduced_vara || !a || !out_a || !out_vara || n_zero < 0)
        return set_error(EG_ERR_ARG, "eg_store_a_and_vara: bad argument");
    EG_TRY(ensure_init());
    std::vector<int64_t> z;
    for (int64_t i = 0; i < n_zero; i++) {
        if (zero_rows[i] < 0 || zero_rows[i] >= Mt->rows) return set_error(EG_ERR_ARG, "zero row out of range");
        z.push_back(zero_rows[i]);
    }
    return scan_of_store(Mt, z, inv_MMt_sqrt, dim_reduced_vara, a, out_a, out_vara);
}
extern "C" int eg_store_extract_col(const eg_store_t* M, int64_t col, int32_t* out) {
    if (!M || !out || col < 0 || col >= M->cols) return set_error(EG_ERR_ARG, "eg_store_extract_col: bad argument");
    EG_TRY(ensure_init());
    Pin pin(M);
    if (M->nparts > 1) {   // the GPU that owns the marker answers
        if (M->mt_orientation) return set_error(EG_ERR_ARG, "eg_store_extract_col: needs an M store");
        return run_all([&](int r) -> int {
            if (!(col >= M->off[r] && col < M->off[r + 1])) return EG_OK;
            return eg_store_extract_col(M->part[r], col - M->off[r], out);
        });
    }
    DevBuf d;
    EG_TRY(d.alloc((size_t)M->rows * 4, "column"));
    EG_TRY(eg_dev_extract_col(M->d, M->rows, M->pitch, col, d.as<int32_t>(), g_ctx.stream));
    EG_CUDA(cudaMemcpyAsync(out, d.p, (size_t)M->rows * 4, cudaMemcpyDeviceToHost, g_ctx.stream));
    EG_CUDA(cudaStreamSynchronize(g_ctx.stream));
    return EG_OK;
}

// ================================================================== device-level: scan pre-products (cuBLAS)
extern "C" int eg_dev_symmetry(const double* d_A, int64_t n, double* max_abs, double* max_asym, void* stream) {
    if (!d_A || n <= 0 || !max_abs || !max_asym) return set_error(EG_ERR_ARG, "eg_dev_symmetry: bad argument");
    EG_TRY(ensure_init());
    cudaStream_t st = (cudaStream_t)stream;
    static thread_local unsigned long long* d_out = nullptr;
    if (!d_out) EG_CUDA(cudaMalloc(&d_out, 2 * sizeof(unsigned long long)));
    EG_CUDA(cudaMemsetAsync(d_out, 0, 2 * sizeof(unsigned long long), st));
    const unsigned nb = (unsigned)((n + 63) / 64);
    symmetry_kernel<<<dim3(nb, nb), 256, 0, st>>>(d_A, n, d_out);
    EG_TRY(check_launch("symmetry_kernel"));
    unsigned long long h[2];
    EG_CUDA(cudaMemcpyAsync(h, d_out, sizeof(h), cudaMemcpyDeviceToHost, st));
    EG_CUDA(cudaStreamSynchronize(st));
    memcpy(max_abs, &h[0], 8);
    memcpy(max_asym, &h[1], 8);
    return EG_OK;
}

// Which path the n^3 pre-products of symmetric inputs take: the exact int8 digit-slice products (prep_i8.cu) from n = 512
// (below that the fixed cost of slicing and of the 7 level passes outweighs two tiny DGEMMs); EAGLE_PREP_MODE=i8 / f64
// forces one.  The digit-slice path is deterministic whatever the column split, so marker-sharded runs split the columns
// of W over the GPUs only when it is taken (a library DGEMM rounds differently for different splits).
extern "C" int eg_prep_uses_i8(int64_t n) {
    const char* env_pm = getenv("EAGLE_PREP_MODE");
    if (env_pm && env_pm[0] == 'i') return 1;
    if (env_pm && env_pm[0] == 'f') return 0;
    return n >= 512;
}

// Columns [col0, col1) of W = S * (V * S) into the packed Wp (ld = Kpad); d_tmp needs n * (col1-col0) doubles.
// upper_only != 0: only rows 0 .. col1-1 of those columns are computed (enough when W is symmetric).
extern "C" int eg_dev_scan_prepare_cols(const double* d_S, const double* d_V, int64_t n, int64_t col0, int64_t col1,
                                        int upper_only, double* d_tmp, double* d_Wp, void* stream) {
    if (!d_S || !d_V || !d_tmp || !d_Wp || n <= 0 || col0 < 0 || col1 > n || col0 > col1)
        return set_error(EG_ERR_ARG, "eg_dev_scan_prepare_cols: bad argument");
    if (col0 == col1) return EG_OK;
    EG_TRY(ensure_init());
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t Kpad = round_up(n, 32), nc = col1 - col0;
    // symmetric inputs: both products on the int8 tensor cores (prep_i8.cu) unless EAGLE_PREP_MODE=f64, the digit slices
    // do not fit in memory, or n is tiny (eg_prep_uses_i8)
    const bool want_i8 = eg_prep_uses_i8(n) != 0;
    if (upper_only && want_i8) {
        bool done = false;
        EG_TRY(launch_prepare_i8(d_S, d_V, n, col0, col1, d_tmp, d_Wp, Kpad, st, &done));
        if (done) return EG_OK;
    }
    const double one = 1.0, zero = 0.0;
    if (cublasSetStream(g_ctx.cublas, st) != CUBLAS_STATUS_SUCCESS) return set_error(EG_ERR_CUDA, "cublasSetStream");
    // calculate_a_and_vara_rcpp.cpp:97   tmp = dim_reduced_vara * inv_MMt_sqrt      (columns col0..col1)
    if (cublasDgemm(g_ctx.cublas, CUBLAS_OP_N, CUBLAS_OP_N, (int)n, (int)nc, (int)n, &one, d_V, (int)n, d_S + col0 * n,
                    (int)n, &zero, d_tmp, (int)n) != CUBLAS_STATUS_SUCCESS)
        return set_error(EG_ERR_CUDA, "cublasDgemm(V*S) failed");
    // :98   W = inv_MMt_sqrt * tmp, written straight into the packed layout (ld = Kpad)
    const int64_t step = upper_only ? 1024 : nc;
    for (int64_t b0 = 0; b0 < nc; b0 += step) {
        const int64_t nb = (b0 + step <= nc) ? step : nc - b0;
        const int64_t rows = upper_only ? (col0 + b0 + nb) : n;  // rows 0 .. last column of the block
        if (cublasDgemm(g_ctx.cublas, CUBLAS_OP_N, CUBLAS_OP_N, (int)rows, (int)nb, (int)n, &one, d_S, (int)n,
                        d_tmp + b0 * n, (int)n, &zero, d_Wp + (col0 + b0) * Kpad, (int)Kpad) != CUBLAS_STATUS_SUCCESS)
            return set_error(EG_ERR_CUDA, "cublasDgemm(S*tmp) failed");
    }
    return EG_OK;
}

// v = S * a into column n of Wp, then fold W into U = diag(W) + strict_upper(W + W^T) (needs ALL columns of W;
// w_is_upper != 0: W holds its upper triangle only and is symmetric, so U = diag + 2 * strict_upper)
extern "C" int eg_dev_scan_fold(const double* d_S, const double* d_a, int64_t n, int w_is_upper, double* d_Wp,
                                void* stream) {
    if (!d_S || !d_a || !d_Wp || n <= 0) return set_error(EG_ERR_ARG, "eg_dev_scan_fold: bad argument");
    EG_TRY(ensure_init());
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t Kpad = round_up(n, 32);
    const double one = 1.0, zero = 0.0;
    if (cublasSetStream(g_ctx.cublas, st) != CUBLAS_STATUS_SUCCESS) return set_error(EG_ERR_CUDA, "cublasSetStream");
    // :90   v = inv_MMt_sqrt * a  -> column n of Wp
    if (cublasDgemv(g_ctx.cublas, CUBLAS_OP_N, (int)n, (int)n, &one, d_S, (int)n, d_a, 1, &zero, d_Wp + n * Kpad, 1) !=
        CUBLAS_STATUS_SUCCESS)
        return set_error(EG_ERR_CUDA, "cublasDgemv(S*a) failed");
    // vara_j = m^T W m only sees the symmetric part of W: fold it into the upper triangle (scan_f64.cu)
    const unsigned nb = (unsigned)((n + 31) / 32);
    symmetrize_upper_kernel<<<dim3(nb, nb), 256, 0, st>>>(d_Wp, n, Kpad, w_is_upper);
    return check_launch("symmetrize_upper_kernel");
}

// S and V symmetric (to 1e-13 of their largest entry; always the case under AM(): chol2inv output and a
// variance matrix) => W = S V S is symmetric and only its upper triangle is computed (3 n^3 instead of 4 n^3 flops)
extern "C" int eg_dev_inputs_symmetric(const double* d_S, const double* d_V, int64_t n, int* yes, void* stream) {
    if (!yes) return set_error(EG_ERR_ARG, "null");
    double aS, dS, aV, dV;
    EG_TRY(eg_dev_symmetry(d_S, n, &aS, &dS, stream));
    EG_TRY(eg_dev_symmetry(d_V, n, &aV, &dV, stream));
    const char* env = getenv("EAGLE_SCAN_SYMMETRIC");
    *yes = !(env && env[0] == '0') && dS <= 1e-13 * aS && dV <= 1e-13 * aV;
    return EG_OK;
}

extern "C" int eg_dev_scan_prepare(const double* d_S, const double* d_V, const double* d_a, int64_t n, double* d_tmp,
                                   double* d_Wp, void* stream) {
    if (!d_S || !d_V || !d_a || !d_tmp || !d_Wp || n <= 0) return set_error(EG_ERR_ARG, "eg_dev_scan_prepare: bad argument");
    EG_TRY(ensure_init());
    int sym = 0;
    EG_TRY(eg_dev_inputs_symmetric(d_S, d_V, n, &sym, stream));
    EG_CUDA(cudaMemsetAsync(d_Wp, 0, (size_t)eg_scan_wp_elems(n) * 8, (cudaStream_t)stream));
    EG_TRY(eg_dev_scan_prepare_cols(d_S, d_V, n, 0, n, sym, d_tmp, d_Wp, stream));
    return eg_dev_scan_fold(d_S, d_a, n, sym, d_Wp, stream);
}

// ================================================================== reference-facing entry points
extern "C" int eg_ReadBlock(const char* asciifname, int64_t start_row, int64_t numcols, int64_t numrows_in_block,
                            double* out_colmajor) {
    if (!asciifname || !out_colmajor || start_row < 0 || numcols <= 0 || numrows_in_block <= 0)
        return set_error(EG_ERR_ARG, "ReadBlock: bad argument");
    EG_TRY(ensure_init());
    MappedFile f;
    EG_TRY(f.open_ro(asciifname));
    const void* nl = memchr(f.p, '\n', f.size);
    const int64_t line = nl ? (const uint8_t*)nl - f.p : (int64_t)f.size;  // characters per line
    if (numcols > line) return set_error(EG_ERR_FORMAT, "ReadBlock: lines of %s have %lld characters, %lld requested",
                                         asciifname, (long long)line, (long long)numcols);
    const int64_t nrows_file = ((int64_t)f.size + 1) / (line + 1);
    if (start_row + numrows_in_block > nrows_file)
        return set_error(EG_ERR_FORMAT, "ReadBlock: %s has %lld lines, rows [%lld,%lld) requested", asciifname,
                         (long long)nrows_file, (long long)start_row, (long long)(start_row + numrows_in_block));
    eg_store* s = nullptr;
    EG_TRY(store_from_image(f.p, line, start_row, start_row + numrows_in_block, 0, numcols, false, &s, f.fd));
    DevBuf d;
    int rc = d.alloc((size_t)numrows_in_block * numcols * 8, "ReadBlock output");
    if (rc == EG_OK) {
        dim3 grid((unsigned)((numcols + 31) / 32), (unsigned)((numrows_in_block + 31) / 32));
        if (grid.y > 65535) rc = set_error(EG_ERR_ARG, "ReadBlock: block of %lld rows is too tall", (long long)numrows_in_block);
        if (rc == EG_OK) {
            i8_to_f64_colmajor_kernel<<<grid, 256, 0, g_ctx.stream>>>(s->d, numrows_in_block, numcols, s->pitch, d.as<double>());
            rc = check_launch("i8_to_f64_colmajor_kernel");
        }
        if (rc == EG_OK)
            rc = check_cuda(cudaMemcpyAsync(out_colmajor, d.p, (size_t)numrows_in_block * numcols * 8,
                                            cudaMemcpyDeviceToHost, g_ctx.stream), "ReadBlock D2H");
        if (rc == EG_OK) rc = check_cuda(cudaStreamSynchronize(g_ctx.stream), "ReadBlock");
    }
    eg_store_free(s);
    return rc;
}

extern "C" int eg_calculateMMt_rcpp(const char* f_name_ascii, double max_memory_in_Gbytes, int num_cores,
                                    const double* selected_loci, int64_t n_selected_loci, const int64_t* dims,
                                    int quiet, eg_message_fn message, void* message_ctx, double* out_MMt) {
    (void)max_memory_in_Gbytes;
    (void)num_cores;
    if (!dims || !out_MMt) return set_error(EG_ERR_ARG, "calculateMMt_rcpp: null argument");
    eg_store* M = nullptr;
    EG_TRY(cached_store(f_name_ascii, dims[0], dims[1], true, &M));
    std::vector<int64_t> z;
    EG_TRY(parse_selected(selected_loci, n_selected_loci, dims[1], z, "calculateMMt_rcpp"));
    if (!quiet) say(message, message_ctx, " M %%*%% t(M) on GPU %d (int8 tensor cores, exact) ", g_ctx.device);
    return mmt_of_store(M, z, out_MMt, true);
}

extern "C" int eg_calculate_a_and_vara_rcpp(const char* f_name_ascii, const double* selected_loci,
                                            int64_t n_selected_loci, const double* inv_MMt_sqrt,
                                            const double* dim_reduced_vara, double max_memory_in_Gbytes,
                                            const int64_t* dims, const double* a, int quiet, eg_message_fn message,
                                            void* message_ctx, double* out_a, double* out_vara) {
    (void)max_memory_in_Gbytes;
    if (!dims || !inv_MMt_sqrt || !dim_reduced_vara || !a || !out_a || !out_vara)
        return set_error(EG_ERR_ARG, "calculate_a_and_vara_rcpp: null argument");
    eg_store* Mt = nullptr;
    EG_TRY(cached_store(f_name_ascii, dims[0], dims[1], false, &Mt));  // dims of Mt: (L, n)
    std::vector<int64_t> z;
    EG_TRY(parse_selected(selected_loci, n_selected_loci, dims[0], z, "calculate_a_and_vara_rcpp"));
    if (!quiet)
        say(message, message_ctx, "Inside internal function calculate_a_and_vara_rcpp: GPU %d, no blocking needed ",
            g_ctx.device);
    return scan_of_store(Mt, z, inv_MMt_sqrt, dim_reduced_vara, a, out_a, out_vara);
}

extern "C" int eg_calculate_reduced_a_rcpp(const char* f_name_ascii, double varG, const double* P, const double* y,
                                           double max_memory_in_Gbytes, const int64_t* dims,
                                           const double* selected_loci, int64_t n_selected_loci, int quiet,
                                           eg_message_fn message, void* message_ctx, double* out_ar) {
    (void)max_memory_in_Gbytes;
    if (!dims || !P || !y || !out_ar) return set_error(EG_ERR_ARG, "calculate_reduced_a_rcpp: null argument");
    const int64_t n = dims[0], L = dims[1];  // dims of M; the file is Mt.ascii (L lines of n characters)
    eg_store* Mt = nullptr;
    EG_TRY(cached_store(f_name_ascii, L, n, false, &Mt, false));   // a plain store on the first GPU
    Pin pin_mt(Mt);
    std::vector<int64_t> z;
    EG_TRY(parse_selected(selected_loci, n_selected_loci, L, z, "calculate_reduced_a_rcpp"));
    if (!quiet) say(message, message_ctx, "Inside internal function calculate_reduced_a_rcpp. GPU %d ", g_ctx.device);
    cudaStream_t st = g_ctx.stream;
    DevBuf dP, dy, dpy, dout;
    EG_TRY(dP.alloc((size_t)n * n * 8, "P"));
    EG_TRY(dy.alloc((size_t)n * 8, "y"));
    EG_TRY(dpy.alloc((size_t)n * 8, "P*y"));
    EG_TRY(dout.alloc((size_t)L * 8, "ar"));
    EG_CUDA(cudaMemcpyAsync(dP.p, P, (size_t)n * n * 8, cudaMemcpyHostToDevice, st));
    EG_CUDA(cudaMemcpyAsync(dy.p, y, (size_t)n * 8, cudaMemcpyHostToDevice, st));
    const double one = 1.0, zero = 0.0;
    if (cublasSetStream(g_ctx.cublas, st) != CUBLAS_STATUS_SUCCESS) return set_error(EG_ERR_CUDA, "cublasSetStream");
    if (cublasDgemv(g_ctx.cublas, CUBLAS_OP_N, (int)n, (int)n, &one, dP.as<double>(), (int)n, dy.as<double>(), 1, &zero,
                    dpy.as<double>(), 1) != CUBLAS_STATUS_SUCCESS)  // :82  ar = P * y
        return set_error(EG_ERR_CUDA, "cublasDgemv(P*y) failed");
    EG_TRY(eg_dev_gemv_i8(Mt->d, L, n, Mt->pitch, dpy.as<double>(), varG, dout.as<double>(), st));  // :83-84
    EG_CUDA(cudaMemcpyAsync(out_ar, dout.p, (size_t)L * 8, cudaMemcpyDeviceToHost, st));
    EG_CUDA(cudaStreamSynchronize(st));
    for (int64_t r : z) out_ar[r] = varG * 0.0;  // :74-78 zeroed rows of Mt
    return EG_OK;
}

extern "C" int eg_extract_geno_rcpp(const char* f_name_ascii, double max_memory_in_Gbytes, int64_t selected_locus,
                                    const int64_t* dims, int32_t* out) {
    (void)max_memory_in_Gbytes;
    if (!dims || !out) return set_error(EG_ERR_ARG, "extract_geno_rcpp: null argument");
    if (selected_locus < 0 || selected_locus >= dims[1])
        return set_error(EG_ERR_ARG, "extract_geno_rcpp: locus %lld outside [0, %lld)", (long long)selected_locus,
                         (long long)dims[1]);
    eg_store* M = nullptr;
    EG_TRY(cached_store(f_name_ascii, dims[0], dims[1], true, &M));  // shares the store with calculateMMt_rcpp
    return eg_store_extract_col(M, selected_locus, out);
}

// ================================================================== ingest: SURVEY.md section 8(f) rank 3 (csrc/ingest.cu)
namespace eg {
struct PinnedBuf {
    void* p = nullptr;
    size_t cap = 0;
    ~PinnedBuf() {
        if (p) cudaFreeHost(p);
    }
    int ensure(size_t n, const char* what) {
        if (n <= cap) return EG_OK;
        if (p) cudaFreeHost(p);
        p = nullptr;
        cap = 0;
        if (cudaMallocHost(&p, n) != cudaSuccess) {
            cudaGetLastError();
            p = nullptr;
            return set_error(EG_ERR_ALLOC, "out of page-locked host memory allocating %zu bytes for %s", n, what);
        }
        cap = n;
        return EG_OK;
    }
};
struct OutFile {
    FILE* f = nullptr;
    ~OutFile() {
        if (f) fclose(f);
    }
};
static bool host_ws(uint8_t b) { return b == ' ' || (b >= 9 && b <= 13); }
// read-only view of a whole file; an empty file is a valid (zero-row) input here
struct TextFile {
    int fd = -1;
    const uint8_t* p = nullptr;
    size_t size = 0;
    ~TextFile() {
        if (p) munmap(const_cast<uint8_t*>(p), size);
        if (fd >= 0) close(fd);
    }
    bool open_ro(const char* path) {
        fd = ::open(path, O_RDONLY);
        struct stat st;
        if (fd < 0 || fstat(fd, &st) != 0 || !S_ISREG(st.st_mode)) return false;
        size = (size_t)st.st_size;
        if (size == 0) return true;
        void* m = mmap(nullptr, size, PROT_READ, MAP_PRIVATE, fd, 0);
        if (m == MAP_FAILED) return false;
        p = static_cast<const uint8_t*>(m);
        madvise(m, size, MADV_SEQUENTIAL);
        return true;
    }
};

// bytes of text the tokeniser works on at a time (EAGLE_INGEST_PIECE_BYTES overrides the 256 MB; at least 64)
static int64_t ingest_piece_bytes() {
    const char* envp = getenv("EAGLE_INGEST_PIECE_BYTES");
    const int64_t piece_max = envp ? atoll(envp) : (256LL << 20);
    return piece_max < 64 ? 64 : piece_max;
}
// a piece = whole lines: the piece starting at `off` ends after the last '\n' inside the window, or extends to the end of
// a longer line
static size_t piece_end(const TextFile& in, size_t off, int64_t piece_max) {
    size_t end = off + (size_t)piece_max < in.size ? off + (size_t)piece_max : in.size;
    if (end < in.size) {
        const void* nlp = memrchr(in.p + off, '\n', end - off);
        if (nlp) end = (size_t)((const uint8_t*)nlp - in.p) + 1;
        else {
            const void* nx = memchr(in.p + end, '\n', in.size - end);
            end = nx ? (size_t)((const uint8_t*)nx - in.p) + 1 : in.size;
        }
    }
    return end;
}
// A piece of text on the device and the tokeniser's chunk prefix over it (tokens and '\n' before every chunk); the buffers
// grow to the largest piece seen.
struct TokenisedPiece {
    DevBuf text, counts, prefix;
    size_t text_cap = 0, chunk_cap = 0;
    // uploads piece[0, nb) and runs the tokeniser's scan; *newlines: the '\n' in the piece
    int scan(const uint8_t* piece, int64_t nb, const char* what, int64_t* newlines, cudaStream_t st) {
        const int64_t nch = eg_tokenise_chunks(nb);
        if ((size_t)nb + 64 > text_cap) {
            text_cap = (size_t)nb + 64;
            EG_TRY(text.alloc(text_cap, what));
        }
        if ((size_t)nch > chunk_cap) {
            chunk_cap = (size_t)nch;
            EG_TRY(counts.alloc(chunk_cap * 2 * sizeof(uint32_t), "tokeniser counts"));
            EG_TRY(prefix.alloc((chunk_cap + 1) * 2 * sizeof(int64_t), "tokeniser prefix"));
        }
        EG_CUDA(cudaMemcpyAsync(text.p, piece, (size_t)nb, cudaMemcpyHostToDevice, st));
        EG_TRY(eg_dev_tokenise_scan(text.as<uint8_t>(), nb, counts.as<uint32_t>(), prefix.as<int64_t>(), st));
        int64_t totals[2] = {0, 0};
        EG_CUDA(cudaMemcpyAsync(totals, prefix.as<int64_t>() + 2 * nch, sizeof(totals), cudaMemcpyDeviceToHost, st));
        EG_CUDA(cudaStreamSynchronize(st));
        *newlines = totals[1];
        return EG_OK;
    }
    // row and token count of the scanned piece before byte `pos` (an error event): the prefix of pos's chunk, then a walk
    int counts_before(const uint8_t* piece, int64_t nb, int64_t pos, int64_t* row, int64_t* toks, cudaStream_t st) {
        const int64_t cb = eg_tokenise_chunk_bytes();
        const int64_t ch = (pos >= nb ? nb - 1 : pos) / cb;
        int64_t pre[2];
        EG_CUDA(cudaMemcpyAsync(pre, prefix.as<int64_t>() + 2 * ch, sizeof(pre), cudaMemcpyDeviceToHost, st));
        EG_CUDA(cudaStreamSynchronize(st));
        *toks = pre[0];
        *row = pre[1];
        for (int64_t q = ch * cb; q < pos; q++) {
            if (piece[q] == '\n') (*row)++;
            else if (!host_ws(piece[q]) && (q == 0 || host_ws(piece[q - 1]))) (*toks)++;
        }
        return EG_OK;
    }
};

static void echo_first_lines(const TextFile& in, int nrowsp, int ncolsp, eg_message_fn message, void* mctx);

// CreateASCIInospace(fname, asciifname, dims, AA, AB, BB, quiet, message, missing)   src/CreateASCIInospace.cpp:17-164
// The text is tokenised on the device in pieces of whole lines; *ok mirrors the reference's bool.
static int create_ascii_nospace(const char* fname, const char* asciifname, const int64_t* dims, const char* AA, const char* AB,
                                const char* BB, int quiet, eg_message_fn message, void* mctx, const char* missing, int* ok) {
    *ok = 0;
    const int64_t L = dims[1];
    if (L <= 0) return set_error(EG_ERR_ARG, "CreateASCIInospace: dims[1] must be positive");
    EG_TRY(ensure_init());
    TextFile in;
    if (!in.open_ro(fname)) {
        say(message, mctx, "ERROR: Text file could not be opened with filename  %s\n", fname);  // :39-41
        return EG_OK;
    }
    OutFile outf;
    outf.f = fopen(asciifname, "wb");
    if (!outf.f) return set_error(EG_ERR_OPEN, "ERROR: Could not open  %s for writing", asciifname);
    if (!quiet) {  // :45-50
        say(message, mctx, "%s", "");
        say(message, mctx, " Reading text File  ");
        say(message, mctx, "%s", "");
        say(message, mctx, " Loading file ");
    }
    const int64_t piece_max = ingest_piece_bytes();
    cudaStream_t st = g_ctx.stream;
    TokenisedPiece tok;
    DevBuf dout, derr;
    PinnedBuf hout;
    EG_TRY(derr.alloc(sizeof(uint64_t), "tokeniser status"));
    size_t out_cap = 0;
    int64_t rows_done = 0;
    size_t off = 0;
    while (off < in.size) {
        const size_t end = piece_end(in, off, piece_max);
        const int64_t nb = (int64_t)(end - off);
        const uint8_t* piece = in.p + off;
        int64_t newlines = 0;
        EG_TRY(tok.scan(piece, nb, "text piece", &newlines, st));
        const int64_t lines = newlines + (piece[nb - 1] != '\n' ? 1 : 0);
        const size_t out_bytes = (size_t)lines * (size_t)(L + 1);
        if (out_bytes + 16 > out_cap) {
            out_cap = out_bytes + 16;
            EG_TRY(dout.alloc(out_cap, "no-space ASCII rows"));
        }
        EG_TRY(hout.ensure(out_bytes + 16, "no-space ASCII rows"));
        uint64_t h_err = UINT64_MAX;
        EG_CUDA(cudaMemcpyAsync(derr.p, &h_err, sizeof(h_err), cudaMemcpyHostToDevice, st));
        EG_TRY(eg_dev_tokenise_emit(tok.text.as<uint8_t>(), nb, tok.prefix.as<int64_t>(), L, AA, AB, BB, missing, dout.as<uint8_t>(),
                                    lines, derr.as<uint64_t>(), st));
        EG_CUDA(cudaMemcpyAsync(&h_err, derr.p, sizeof(h_err), cudaMemcpyDeviceToHost, st));
        EG_CUDA(cudaStreamSynchronize(st));
        int64_t good_rows = lines;
        if (h_err != UINT64_MAX) {
            // first error event of the piece: recover its row and what the reference would have printed
            const int64_t pos = (int64_t)h_err;
            int64_t row = 0, toks = 0;
            EG_TRY(tok.counts_before(piece, nb, pos, &row, &toks, st));
            good_rows = row;
            const long long row1 = (long long)(rows_done + row + 1);
            if (pos >= nb || piece[pos] == '\n') {  // :108-116
                say(message, mctx, "\n");
                say(message, mctx, "Error:  Marker text file contains an unequal number of columns per row.  ");
                say(message, mctx, "        The error has occurred at row %lld which contains %lld but ", row1, (long long)(toks - row * L));
                say(message, mctx, "        it should contain %lld columns of data. ", (long long)L);
                say(message, mctx, "\n");
                say(message, mctx, " ReadMarkerData has terminated with errors");
            } else {  // :94-104
                int64_t e = pos;
                while (e < nb && !host_ws(piece[e])) e++;
                std::string token((const char*)piece + pos, (size_t)(e - pos));
                if (AB && strcmp(AB, "NA") == 0)
                    say(message, mctx, "\n Marker file contains marker genotypes that are different to AA=%s BB=%s", AA, BB);
                else
                    say(message, mctx, "\n Marker file contains marker genotypes that are different to AA=%s AB=%s BB=%s", AA, AB, BB);
                say(message, mctx, " For example , %s in row %lld", token.c_str(), row1);
                say(message, mctx, "\n ReadMarker has terminated with errors\n");
            }
        }
        // rows before the first error are complete (the reference has written them by then, too)
        const size_t wbytes = (size_t)good_rows * (size_t)(L + 1);
        if (wbytes) {
            EG_CUDA(cudaMemcpyAsync(hout.p, dout.p, wbytes, cudaMemcpyDeviceToHost, st));
            EG_CUDA(cudaStreamSynchronize(st));
            if (fwrite(hout.p, 1, wbytes, outf.f) != wbytes) return set_error(EG_ERR_OPEN, "short write to %s", asciifname);
        }
        if (h_err != UINT64_MAX) return EG_OK;  // *ok stays 0
        rows_done += lines;
        off = end;
    }
    if (fflush(outf.f) != 0) return set_error(EG_ERR_OPEN, "short write to %s", asciifname);
    {   // :129-157  echo of the first lines (printed whatever `quiet` says)
        const int nrowsp = dims[0] < 5 ? (int)dims[0] : 5, ncolsp = L < 12 ? (int)L : 12;
        say(message, mctx, " First %d lines and %d columns of the marker text  file. ", nrowsp, ncolsp);
        echo_first_lines(in, nrowsp, ncolsp, message, mctx);
    }
    *ok = 1;
    return EG_OK;
}

// echo of the first lines of the input (CreateASCIInospace.cpp:129-157, CreateASCIInospace_PLINK.cpp:203-236)
static void echo_first_lines(const TextFile& in, int nrowsp, int ncolsp, eg_message_fn message, void* mctx) {
    size_t q = 0;
    std::string tmp;
    for (int r = 0; r < nrowsp && q < in.size; r++) {
        const void* nlp = memchr(in.p + q, '\n', in.size - q);
        const size_t e = nlp ? (size_t)((const uint8_t*)nlp - in.p) : in.size;
        std::string rowline;
        size_t c = q;
        for (int i = 0; i < ncolsp; i++) {
            while (c < e && host_ws(in.p[c])) c++;
            size_t t0 = c;
            while (c < e && !host_ws(in.p[c])) c++;
            if (c > t0) tmp.assign((const char*)in.p + t0, c - t0);  // a failed extraction leaves tmp as it was
            rowline += tmp;
            rowline += " ";
        }
        say(message, mctx, "%s", rowline.c_str());
        q = e + 1;
    }
}

// CreateASCIInospace_PLINK(fname, asciifname, dims, quiet, message)            src/CreateASCIInospace_PLINK.cpp:16-248
// dims = (rows, 6 + 2 * nsnp) of the ped file.  Allele tokens must be single characters (the reference reads the alleles
// character by character, :88-93, and silently misreads anything else; here that is EG_ERR_FORMAT).
static int create_ascii_nospace_plink(const char* fname, const char* asciifname, const int64_t* dims, int quiet,
                                      eg_message_fn message, void* mctx, int* ok) {
    (void)quiet;
    *ok = 0;
    const int64_t ncols = dims[1], nsnp = (ncols - 6) / 2;
    if (ncols < 8 || ((ncols - 6) & 1)) return set_error(EG_ERR_ARG, "CreateASCIInospace_PLINK: dims[1] must be 6 + 2 * (number of SNPs)");
    EG_TRY(ensure_init());
    TextFile in;
    if (!in.open_ro(fname)) {  // :38-42
        say(message, mctx, "ERROR: PLINK ped file could not be opened with filename  %s", fname);
        say(message, mctx, "ERROR: ReadMarkerData has terminated with errors.  ");
        return EG_OK;
    }
    OutFile outf;
    outf.f = fopen(asciifname, "wb");
    if (!outf.f) return set_error(EG_ERR_OPEN, "ERROR: Could not open  %s for writing", asciifname);
    const int64_t piece_max = ingest_piece_bytes();
    cudaStream_t st = g_ctx.stream;
    TokenisedPiece tok;
    DevBuf dall, dout, dstat, dstate;
    PinnedBuf hout;
    EG_TRY(dstat.alloc(3 * sizeof(uint64_t), "ped status"));
    EG_TRY(dstate.alloc((size_t)nsnp * 2, "allele state"));
    size_t rows_cap = 0;
    int64_t rows_done = 0;
    bool warned = false;
    size_t off = 0;
    while (off < in.size) {
        const size_t end = piece_end(in, off, piece_max);
        const int64_t nb = (int64_t)(end - off);
        const uint8_t* piece = in.p + off;
        int64_t newlines = 0;
        EG_TRY(tok.scan(piece, nb, "ped piece", &newlines, st));
        const int64_t lines = newlines + (piece[nb - 1] != '\n' ? 1 : 0);
        if ((size_t)lines > rows_cap) {
            rows_cap = (size_t)lines;
            EG_TRY(dall.alloc(rows_cap * (size_t)nsnp * 2 + 16, "allele characters"));
            EG_TRY(dout.alloc(rows_cap * (size_t)(nsnp + 1) + 16, "no-space ASCII rows"));
        }
        EG_TRY(hout.ensure((size_t)lines * (size_t)(nsnp + 1) + 16, "no-space ASCII rows"));
        uint64_t h_stat[3] = {UINT64_MAX, UINT64_MAX, UINT64_MAX};  // stage-1 error position, third-allele key, missing key
        EG_CUDA(cudaMemcpyAsync(dstat.p, h_stat, sizeof(h_stat), cudaMemcpyHostToDevice, st));
        EG_TRY(eg_dev_ped_alleles(tok.text.as<uint8_t>(), nb, tok.prefix.as<int64_t>(), ncols, dall.as<uint8_t>(), lines,
                                  dstat.as<uint64_t>(), st));
        EG_CUDA(cudaMemcpyAsync(h_stat, dstat.p, sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        EG_CUDA(cudaStreamSynchronize(st));
        int64_t good_rows = lines, bad_cols = -1;
        if (h_stat[0] != UINT64_MAX) {  // rows before the offending line are still processed, as in the reference
            const int64_t pos = (int64_t)h_stat[0];
            int64_t row = 0, toks = 0;
            EG_TRY(tok.counts_before(piece, nb, pos, &row, &toks, st));
            if (!(pos >= nb || piece[pos] == '\n')) {
                int64_t e = pos;
                while (e < nb && !host_ws(piece[e])) e++;
                return set_error(EG_ERR_FORMAT, "PLINK ped file: allele \"%.*s\" in row %lld is not a single character", (int)(e - pos),
                                 (const char*)piece + pos, (long long)(rows_done + row + 1));
            }
            good_rows = row;
            bad_cols = toks - row * ncols;
        }
        EG_TRY(eg_dev_ped_genotypes(dall.as<uint8_t>(), good_rows, nsnp, rows_done == 0 ? 1 : 0, rows_done, dstate.as<uint8_t>(),
                                    dout.as<uint8_t>(), dstat.as<uint64_t>() + 1, st));
        EG_CUDA(cudaMemcpyAsync(h_stat + 1, dstat.as<uint64_t>() + 1, 2 * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        EG_CUDA(cudaStreamSynchronize(st));
        const bool third = h_stat[1] != UINT64_MAX;
        if (!warned && h_stat[2] != UINT64_MAX && (!third || h_stat[2] < h_stat[1])) {  // :119-129, printed once
            warned = true;
            say(message, mctx, "\n");
            say(message, mctx, " Warning:  PLINK file contains missing alleles (i.e. 0 or - ) ");
            say(message, mctx, "           These missing genotypes should be imputed before running Eagle.");
            say(message, mctx, "           As an approximation, AMpus has set these missing genotypes to heterozygotes. ");
            say(message, mctx, "           Since Eagle assumes an additive model, heterozygote genotypes do not contribute to the estimation of ");
            say(message, mctx, "           the additive effects.  ");
            say(message, mctx, "\n");
        }
        if (third) good_rows = (int64_t)(h_stat[1] / (uint64_t)nsnp) - rows_done;
        const size_t wbytes = (size_t)good_rows * (size_t)(nsnp + 1);
        if (wbytes) {
            EG_CUDA(cudaMemcpyAsync(hout.p, dout.p, wbytes, cudaMemcpyDeviceToHost, st));
            EG_CUDA(cudaStreamSynchronize(st));
            if (fwrite(hout.p, 1, wbytes, outf.f) != wbytes) return set_error(EG_ERR_OPEN, "short write to %s", asciifname);
        }
        if (third) {  // :161-167
            say(message, mctx, "\n");
            say(message, mctx, "Error:  PLINK file cannot contain more than two alleles at a locus.");
            say(message, mctx, "        The error has occurred at snp locus %lld for individual %lld", (long long)(h_stat[1] % (uint64_t)nsnp) + 1,
                (long long)(h_stat[1] / (uint64_t)nsnp) + 1);
            say(message, mctx, "\n");
            say(message, mctx, " ReadMarkerData has terminated with errors");
            return EG_OK;
        }
        if (bad_cols >= 0) {  // :69-76
            say(message, mctx, "\n");
            say(message, mctx, "Error:  PLINK file contains an unequal number of columns per row.  ");
            say(message, mctx, "        The error has occurred at row %lld which contains %lld but ", (long long)(rows_done + good_rows + 1), (long long)bad_cols);
            say(message, mctx, "        it should contain %lld columns of data. ", (long long)ncols);
            say(message, mctx, "\n");
            say(message, mctx, " ReadMarkerData has terminated with errors");
            return EG_OK;
        }
        rows_done += lines;
        off = end;
    }
    if (fflush(outf.f) != 0) return set_error(EG_ERR_OPEN, "short write to %s", asciifname);
    const int nrowsp = dims[0] < 5 ? (int)dims[0] : 5, ncolsp = ncols < 25 ? (int)ncols : 24;  // :209-214
    say(message, mctx, " First %d lines and %d columns of the PLINK ped file. ", nrowsp, ncolsp);
    echo_first_lines(in, nrowsp, ncolsp, message, mctx);
    *ok = 1;
    return EG_OK;
}
// A row-major store as a no-space ASCII file: encode in row blocks of ~256 MB, two page-locked buffers, the D2H of block k
// running while block k-1 is written.
static int write_store_ascii(const eg_store* T, const char* path) {
    if (!T->pitch) return set_error(EG_ERR_ARG, "write_store_ascii: needs a row-major store");
    const int64_t rows = T->rows, cols = T->cols, line = cols + 1;
    OutFile outf;
    outf.f = fopen(path, "wb");
    int rc = outf.f ? EG_OK : set_error(EG_ERR_OPEN, "ERROR: Could not open  %s for writing", path);
    int64_t block_rows = (256LL << 20) / line;
    if (block_rows < 1) block_rows = 1;
    if (block_rows > rows) block_rows = rows;
    DevBuf denc[2];
    PinnedBuf henc[2];
    cudaEvent_t done[2] = {nullptr, nullptr};
    for (int i = 0; i < 2 && rc == EG_OK; i++) {
        rc = denc[i].alloc((size_t)block_rows * line + 16, "ASCII rows");
        if (rc == EG_OK) rc = henc[i].ensure((size_t)block_rows * line + 16, "ASCII rows");
        if (rc == EG_OK) rc = check_cuda(cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming), "cudaEventCreate");
    }
    int64_t pending_rows[2] = {0, 0};
    int k = 0;
    for (int64_t r = 0; rc == EG_OK && r < rows; r += block_rows, k++) {
        const int b = k & 1;
        const int64_t nr = r + block_rows <= rows ? block_rows : rows - r;
        rc = eg_dev_encode_ascii(T->d, T->pitch, cols, r, nr, denc[b].as<uint8_t>(), g_ctx.stream);
        if (rc == EG_OK)
            rc = check_cuda(cudaMemcpyAsync(henc[b].p, denc[b].p, (size_t)nr * line, cudaMemcpyDeviceToHost, g_ctx.stream), "D2H of ASCII rows");
        if (rc == EG_OK) rc = check_cuda(cudaEventRecord(done[b], g_ctx.stream), "cudaEventRecord");
        pending_rows[b] = nr;
        if (rc == EG_OK && k >= 1) {  // write the previous block while this one is in flight
            const int pb = b ^ 1;
            rc = check_cuda(cudaEventSynchronize(done[pb]), "ASCII rows");
            const size_t wb = (size_t)pending_rows[pb] * line;
            if (rc == EG_OK && fwrite(henc[pb].p, 1, wb, outf.f) != wb) rc = set_error(EG_ERR_OPEN, "short write to %s", path);
            pending_rows[pb] = 0;
        }
    }
    if (rc == EG_OK && k >= 1) {
        const int pb = (k - 1) & 1;
        rc = check_cuda(cudaEventSynchronize(done[pb]), "ASCII rows");
        const size_t wb = (size_t)pending_rows[pb] * line;
        if (rc == EG_OK && fwrite(henc[pb].p, 1, wb, outf.f) != wb) rc = set_error(EG_ERR_OPEN, "short write to %s", path);
    }
    cudaStreamSynchronize(g_ctx.stream);
    for (int i = 0; i < 2; i++)
        if (done[i]) cudaEventDestroy(done[i]);
    if (outf.f) {
        if (fclose(outf.f) != 0 && rc == EG_OK) rc = set_error(EG_ERR_OPEN, "short write to %s", path);
        outf.f = nullptr;
    }
    return rc;
}
}  // namespace eg

extern "C" int eg_createM_ASCII_rcpp(const char* f_name, const char* f_name_ascii, const char* type, const char* AA, const char* AB,
                                     const char* BB, double max_memory_in_Gbytes, const int64_t* dims, int quiet,
                                     eg_message_fn message, void* message_ctx, const char* missing, int* ok) {
    (void)max_memory_in_Gbytes;  // both branches of the reference call the same line-by-line routine (createM_ASCII_rcpp.cpp:88-96)
    if (!f_name || !f_name_ascii || !type || !AA || !AB || !BB || !missing || !dims || !ok)
        return set_error(EG_ERR_ARG, "createM_ASCII_rcpp: null argument");
    if (strcmp(type, "PLINK") == 0)  // :71-78
        return create_ascii_nospace_plink(f_name, f_name_ascii, dims, quiet, message, message_ctx, ok);
    if (!quiet) say(message, message_ctx, " A text file is being assumed as the input data file type. ");  // :85-86
    return create_ascii_nospace(f_name, f_name_ascii, dims, AA, AB, BB, quiet, message, message_ctx, missing, ok);
}

// createMt_ASCII_rcpp(f_name, f_name_ascii, type, max_memory_in_Gbytes, dims, quiet, message)   src/createMt_ASCII_rcpp.cpp:15-245
// f_name = M.ascii (dims = (n, L)), f_name_ascii = Mt.ascii to be written.  Decode -> transpose -> encode on the device; both
// resident stores stay in the path cache, so the calculateMMt_rcpp / calculate_a_and_vara_rcpp calls that follow do not
// upload anything.
extern "C" int eg_createMt_ASCII_rcpp(const char* f_name, const char* f_name_ascii, const char* type, double max_memory_in_Gbytes,
                                      const int64_t* dims, int quiet, eg_message_fn message, void* message_ctx) {
    (void)quiet;
    if (!f_name || !f_name_ascii || !type || !dims) return set_error(EG_ERR_ARG, "createMt_ASCII_rcpp: null argument");
    const int64_t n = dims[0], L = dims[1];
    EG_TRY(ensure_init());
    {   // the reference's Rcpp::stop text (:72-75)
        struct stat stt;
        if (stat(f_name, &stt) != 0) return set_error(EG_ERR_OPEN, "\n\nERROR: Could not open  %s\n\n\n", f_name);
    }
    eg_store* M = nullptr;
    EG_TRY(cached_store(f_name, n, L, true, &M, false));
    Pin pin_m(M);   // held while the transpose is allocated (eviction under memory pressure must skip it)
    eg_store* Mt = nullptr;
    EG_TRY(eg_store_transpose(M, &Mt));
    int rc = write_store_ascii(Mt, f_name_ascii);
    if (rc != EG_OK) {
        eg_store_free(Mt);
        return rc;
    }
    {   // the Mt store now corresponds to the file just written: keep it for calculate_a_and_vara_rcpp
        std::string key;
        if (cache_key(f_name_ascii, L, n, false, key) == EG_OK) cache_insert(key, Mt);
        else eg_store_free(Mt);
    }
    // :224-243  summary (printed whatever `quiet` says); bits_in_int/8 == 3 in the reference's integer arithmetic
    const double mem_bytes = 3.5 * (double)n * (double)L * 3.0;
    say(message, message_ctx, "\n\n                    Summary of Marker File  ");
    say(message, message_ctx, "                   ~~~~~~~~~~~~~~~~~~~~~~~~   ");
    say(message, message_ctx, " File type:                   %s", type);
    say(message, message_ctx, " Reformatted ASCII file name:  %s", f_name);
    say(message, message_ctx, " Number of individuals:        %lld", (long long)n);
    say(message, message_ctx, " Number of loci:               %lld", (long long)L);
    say(message, message_ctx, " File size (gigabytes):       %.15g", mem_bytes / 1000000000);
    say(message, message_ctx, " Available memory (gigabytes): %.15g", max_memory_in_Gbytes);
    say(message, message_ctx, "\n\n");
    say(message, message_ctx, " The marker file has been Uploaded");
    return EG_OK;
}

// ReshapeM_rcpp(fnameM, fnameMt, indxNA, dims)                                      src/ReshapeM_rcpp.cpp:16-117
// Writes <fnameM>tmp (M.ascii without the rows listed in indxNA, 0-based) and <fnameMt>tmp (Mt.ascii with those
// characters erased from every line, one after the other in the order given -- R passes them in decreasing order,
// R/check_for_NA_in_trait.R:5), returns newdims = (rows kept, line length of M.ascii).  On the device this is a row
// gather of the resident M store and a column gather of Mt (= its transpose when the two index maps agree); both
// results are encoded back to ASCII for the files AM() switches to (R/AM.R:353-370) and stay resident under those names.
extern "C" int eg_ReshapeM_rcpp(const char* fnameM, const char* fnameMt, const int64_t* indxNA, int64_t n_indx, const int64_t* dims,
                                int64_t* newdims) {
    if (!fnameM || !fnameMt || !dims || !newdims || n_indx < 0 || (n_indx > 0 && !indxNA))
        return set_error(EG_ERR_ARG, "ReshapeM_rcpp: null argument");
    const int64_t n = dims[0], L = dims[1];
    EG_TRY(ensure_init());
    struct stat stt;
    if (stat(fnameM, &stt) != 0) return set_error(EG_ERR_OPEN, "\n\nERROR: Could not open  %s\n\n\n", fnameM);    // :44-47
    if (stat(fnameMt, &stt) != 0) return set_error(EG_ERR_OPEN, "\n\nERROR: Could not open  %s\n\n\n", fnameMt);  // :86-89
    // rows of M: a line is dropped when its number equals any entry (:60-64)
    std::vector<char> drop((size_t)n, 0);
    for (int64_t i = 0; i < n_indx; i++)
        if (indxNA[i] >= 0 && indxNA[i] < n) drop[(size_t)indxNA[i]] = 1;
    std::vector<int64_t> rows_keep;
    for (int64_t r = 0; r < n; r++)
        if (!drop[(size_t)r]) rows_keep.push_back(r);
    // columns of Mt: line.erase(indxNA[ii], 1) one after the other (:104-106); std::string::erase throws beyond the end
    std::vector<int64_t> cols_keep((size_t)n);
    for (int64_t c = 0; c < n; c++) cols_keep[(size_t)c] = c;
    for (int64_t i = 0; i < n_indx; i++) {
        if (indxNA[i] < 0 || indxNA[i] > (int64_t)cols_keep.size())
            return set_error(EG_ERR_ARG, "ReshapeM_rcpp: basic_string::erase: position %lld is beyond a line of %zu characters",
                             (long long)indxNA[i], cols_keep.size());
        if (indxNA[i] < (int64_t)cols_keep.size()) cols_keep.erase(cols_keep.begin() + indxNA[i]);
    }
    if (rows_keep.empty() || cols_keep.empty()) return set_error(EG_ERR_ARG, "ReshapeM_rcpp: no individual left");
    eg_store* M = nullptr;
    EG_TRY(cached_store(fnameM, n, L, true, &M, false));
    Pin pin_m(M);
    const int64_t n1 = (int64_t)rows_keep.size(), n2 = (int64_t)cols_keep.size();
    DevBuf dmap;
    EG_TRY(dmap.alloc((size_t)(n1 > n2 ? n1 : n2) * sizeof(int64_t), "ReshapeM index map"));
    EG_CUDA(cudaMemcpyAsync(dmap.p, rows_keep.data(), (size_t)n1 * sizeof(int64_t), cudaMemcpyHostToDevice, g_ctx.stream));
    eg_store *M1 = nullptr, *T1 = nullptr, *Mrm = nullptr, *Mt1 = nullptr;
    auto cleanup = [&](int rc) {
        cudaStreamSynchronize(g_ctx.stream);
        eg_store_free(M1);
        if (Mt1 != T1) eg_store_free(Mt1);
        eg_store_free(T1);
        eg_store_free(Mrm);
        return rc;
    };
    EG_TRY(store_alloc(n1, L, true, &M1));
    int rc = eg_dev_gather_rows(M->d, n, L, 0, dmap.as<int64_t>(), n1, M1->d, 0, g_ctx.stream);
    if (rc == EG_OK) rc = check_cuda(cudaStreamSynchronize(g_ctx.stream), "ReshapeM row gather");
    if (rc == EG_OK) rc = eg_store_transpose(M1, &T1);                       // L x n1, row-major
    if (rc == EG_OK) rc = eg_store_transpose(T1, &Mrm);                      // n1 x L, row-major: the lines of M.asciitmp
    if (rc != EG_OK) return cleanup(rc);
    std::string outM = std::string(fnameM) + "tmp", outMt = std::string(fnameMt) + "tmp";  // :51, :93
    rc = write_store_ascii(Mrm, outM.c_str());
    eg_store_free(Mrm);
    Mrm = nullptr;
    if (rc != EG_OK) return cleanup(rc);
    if (rows_keep == cols_keep) {
        Mt1 = T1;
    } else {  // an index list that is not decreasing: the erased characters are not the dropped rows
        eg_store* Mt = nullptr;
        rc = cached_store(fnameMt, L, n, false, &Mt, false);
        Pin pin_mt(rc == EG_OK ? Mt : nullptr);
        if (rc == EG_OK) rc = store_alloc(L, n2, false, &Mt1);
        if (rc == EG_OK) rc = check_cuda(cudaMemcpyAsync(dmap.p, cols_keep.data(), (size_t)n2 * sizeof(int64_t), cudaMemcpyHostToDevice, g_ctx.stream), "H2D");
        if (rc == EG_OK) rc = eg_dev_gather_cols(Mt->d, L, Mt->pitch, dmap.as<int64_t>(), n2, Mt1->d, Mt1->pitch, g_ctx.stream);
        if (rc == EG_OK) rc = check_cuda(cudaStreamSynchronize(g_ctx.stream), "ReshapeM column gather");
        if (rc != EG_OK) return cleanup(rc);
    }
    rc = write_store_ascii(Mt1, outMt.c_str());
    if (rc != EG_OK) return cleanup(rc);
    newdims[0] = n1;  // :67
    newdims[1] = L;   // :71  length of the last line read
    {   // the reshaped stores are what the following calls on the two new files need
        std::string key;
        eg_store* keepT = Mt1;
        if (cache_key(outMt.c_str(), L, n2, false, key) == EG_OK) cache_insert(key, keepT);
        else eg_store_free(keepT);
        if (Mt1 != T1) eg_store_free(T1);
        if (cache_key(outM.c_str(), n1, L, true, key) == EG_OK) cache_insert(key, M1);
        else eg_store_free(M1);
    }
    return EG_OK;
}

// getRowColumn(fname)                                                                src/getRowColumn.cpp:19-72
// dimen[0] = number of lines (an unterminated last line counts), dimen[1] = whitespace-separated tokens of the first
// line.  The line count is the tokeniser's newline scan over the file in pieces.
extern "C" int eg_getRowColumn(const char* fname, int64_t* dimen) {
    if (!fname || !dimen) return set_error(EG_ERR_ARG, "getRowColumn: null argument");
    EG_TRY(ensure_init());
    TextFile in;
    if (!in.open_ro(fname)) return set_error(EG_ERR_OPEN, "\n\n ERROR: Could not open  %s\n\n\n", fname);  // :36-39
    dimen[0] = dimen[1] = 0;
    if (in.size == 0) return EG_OK;
    const int64_t piece_max = ingest_piece_bytes();
    const int64_t cap = (int64_t)in.size < piece_max ? (int64_t)in.size : piece_max;
    TokenisedPiece tok;   // sized by the first (largest) piece
    for (size_t off = 0; off < in.size; off += (size_t)cap) {   // fixed-size cuts: only '\n' are counted
        const int64_t nb = (int64_t)(in.size - off < (size_t)cap ? in.size - off : (size_t)cap);
        int64_t newlines = 0;
        EG_TRY(tok.scan(in.p + off, nb, "text piece", &newlines, g_ctx.stream));
        dimen[0] += newlines;
    }
    if (in.p[in.size - 1] != '\n') dimen[0]++;
    const void* nlp = memchr(in.p, '\n', in.size);
    const size_t e = nlp ? (size_t)((const uint8_t*)nlp - in.p) : in.size;
    for (size_t c = 0; c < e;) {  // :58-65  tokens of the first line
        while (c < e && host_ws(in.p[c])) c++;
        if (c >= e) break;
        while (c < e && !host_ws(in.p[c])) c++;
        dimen[1]++;
    }
    return EG_OK;
}
