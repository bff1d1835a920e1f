// api.cu — the C ABI of include/jvector_b200.h, batched GPU group: handle management, host<->HBM staging, launches.
// No CPU fallback lives here: without an sm_100 device every entry point returns JV_ERR_NO_DEVICE.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "../../include/jvector_b200.h"
#include "kernels.h"

using namespace jv;

namespace {

thread_local std::string t_err;
std::mutex g_mu;
constexpr int MAX_DEVICES = 16;
// One process may drive several GPUs (the reference host is one JVM, all parallelism is threads: base:vector/
// VectorizationProvider.java:79-177, base:graph/GraphIndexBuilder.java:440-444): every handle remembers the device it lives on,
// every caller thread owns one context (stream + staging buffers) per device.
unsigned g_mask = 0;                 // devices bound by jv_gpu_init / jv_gpu_init_mask
int g_default_device = -1;           // first device bound
int g_sm_counts[MAX_DEVICES] = {0};
thread_local int t_device = -1;      // device new data sets / graphs of this thread are created on (jv_gpu_set_device); -1 = default
thread_local int t_active = 0;       // device of the call in progress

int fail(int code, const std::string &msg)
{
    t_err = msg;
    return code;
}
int cuda_fail(cudaError_t e, const char *what)
{
    t_err = std::string(what) + ": " + cudaGetErrorString(e);
    return e == cudaErrorMemoryAllocation ? JV_ERR_OOM : JV_ERR_CUDA;
}
#define CK(x, what)                                      \
    do {                                                 \
        cudaError_t e_ = (x);                            \
        if (e_ != cudaSuccess) return cuda_fail(e_, what); \
    } while (0)
// enter a call that creates something: the thread's target device
#define NEED_INIT()                                                                            \
    do {                                                                                       \
        const int d0_ = t_device >= 0 ? t_device : g_default_device;                           \
        if (d0_ < 0) return fail(JV_ERR_NO_DEVICE, "jv_gpu_init() has not succeeded");         \
        t_active = d0_;                                                                        \
        cudaError_t e0_ = cudaSetDevice(d0_);                                                  \
        if (e0_ != cudaSuccess) return cuda_fail(e0_, "cudaSetDevice");                        \
    } while (0)
// enter a call on an existing handle: the handle's device
#define ON_DEVICE_OF(h)                                                                        \
    do {                                                                                       \
        if (g_default_device < 0) return fail(JV_ERR_NO_DEVICE, "jv_gpu_init() has not succeeded"); \
        if (!(h)) return fail(JV_ERR_INVALID, "null handle");                                  \
        t_active = (h)->device;                                                                \
        cudaError_t e0_ = cudaSetDevice(t_active);                                             \
        if (e0_ != cudaSuccess) return cuda_fail(e0_, "cudaSetDevice");                        \
    } while (0)
#define g_sm_count (g_sm_counts[t_active])

// per-thread, per-device stream + growable staging buffers (callers are ForkJoinPool workers: no global locks on the score
// path); released when the thread exits
struct ThreadCtx {
    static constexpr int SLOTS = 8;
    int device = -1;
    cudaStream_t stream = nullptr;
    void *dbuf[SLOTS] = {};
    size_t dcap[SLOTS] = {};
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // host-pointer searches: a second stream carries the query chunks while the search kernel already runs (arrival watermark)
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_copy = nullptr;
    int *marks_pinned = nullptr;  // pinned: the watermark values the copy stream writes behind each chunk
    static constexpr int MARKS = 16;
    int init_copy()
    {
        if (copy_stream) return JV_OK;
        CK(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking), "cudaStreamCreate(copy)");
        CK(cudaEventCreateWithFlags(&ev_copy, cudaEventDisableTiming), "cudaEventCreate(copy)");
        CK(cudaHostAlloc((void **)&marks_pinned, MARKS * sizeof(int), cudaHostAllocDefault), "cudaHostAlloc(marks)");
        return JV_OK;
    }
    int init()
    {
        if (stream) return JV_OK;
        device = t_active;
        CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking), "cudaStreamCreate");
        CK(cudaEventCreate(&ev0), "cudaEventCreate");
        CK(cudaEventCreate(&ev1), "cudaEventCreate");
        return JV_OK;
    }
    int ensure(int slot, size_t bytes)
    {
        if (bytes <= dcap[slot]) return JV_OK;
        if (dbuf[slot]) cudaFree(dbuf[slot]);
        dbuf[slot] = nullptr;
        dcap[slot] = 0;
        size_t want = bytes + bytes / 4 + 256;
        CK(cudaMalloc(&dbuf[slot], want), "cudaMalloc(staging)");
        dcap[slot] = want;
        return JV_OK;
    }
    ~ThreadCtx()
    {
        if (!stream) return;
        int cur = -1;
        if (cudaGetDevice(&cur) != cudaSuccess) return;  // runtime already torn down at process exit: nothing left to free
        if (cudaSetDevice(device) != cudaSuccess) return;
        cudaStreamSynchronize(stream);
        for (int i = 0; i < SLOTS; i++)
            if (dbuf[i]) cudaFree(dbuf[i]);
        cudaEventDestroy(ev0);
        cudaEventDestroy(ev1);
        cudaStreamDestroy(stream);
        if (copy_stream) {
            cudaStreamSynchronize(copy_stream);
            cudaStreamDestroy(copy_stream);
            cudaEventDestroy(ev_copy);
            cudaFreeHost(marks_pinned);
            copy_stream = nullptr;
        }
        stream = nullptr;
        if (cur >= 0) cudaSetDevice(cur);
    }
};
thread_local ThreadCtx t_ctxs[MAX_DEVICES];
thread_local ThreadCtx *t_ctx_override = nullptr;  // worker threads of the multi-device entry points run on the shard's own context
#define t_ctx (*(t_ctx_override ? t_ctx_override : &t_ctxs[t_active]))
thread_local BuildStats t_build_stats = {0, 0, 0, 0, 0};

int round4(int v) { return (v + 3) & ~3; }

void pq_layout(int dim, int M, std::vector<int> &sizes, std::vector<int> &offsets)
{
    // base:quantization/ProductQuantization.java:535-550
    sizes.resize(M);
    offsets.resize(M);
    int base = dim / M, rem = dim % M, off = 0;
    for (int m = 0; m < M; m++) {
        sizes[m] = base + (m < rem ? 1 : 0);
        offsets[m] = off;
        off += sizes[m];
    }
}

}  // namespace

struct jv_dataset_s {
    int device = 0;
    bool borrowed_rows = false;  // jv_dataset_adopt_f32_device: rows belong to the caller
    DataDesc d;
    std::vector<void *> allocs;
    size_t bytes = 0;
    // fp32 DOT_PRODUCT walks: the projection sketch (kernels.h F32Sketch), built by the first search that can use it. Handles are
    // shared across threads: sketch_mu guards the build and jv_dataset_invalidate_sketch.
    std::mutex sketch_mu;
    int sketch_state = 0;  // 0 not built, 1 built, -1 skipped: the basis captured too little of the rows' energy to drop anything
    double sketch_captured = 0.0;
    void *sketch_mem = nullptr;
    F32Sketch sketch = {};
    int alloc(void **p, size_t n)
    {
        CK(cudaMalloc(p, n ? n : 16), "cudaMalloc(dataset)");
        allocs.push_back(*p);
        bytes += n;
        return JV_OK;
    }
    ~jv_dataset_s()
    {
        for (void *p : allocs) cudaFree(p);
        if (sketch_mem) cudaFree(sketch_mem);
    }
};

struct jv_query_s {
    int device = 0;
    jv_dataset ds;
    int metric;
    float *blob = nullptr;
    int pooled = 0;  // blob belongs to a jv_query_batch
};

struct jv_graph_s {
    int device = 0;
    GraphDesc g;
    uint8_t *fused = nullptr;  // FusedPQ records
    int32_t *adj0 = nullptr;
    int32_t *upper_row = nullptr;
    int32_t *upper_adj = nullptr;
    long long *upper_off = nullptr;
    std::vector<std::vector<int32_t>> level_ids;  // host copies, level >= 1
    std::vector<std::vector<int32_t>> level_adj;
    ~jv_graph_s()
    {
        cudaFree(adj0); cudaFree(upper_row); cudaFree(upper_adj); cudaFree(upper_off); cudaFree(fused);
    }
};

struct jv_multi_s {
    int kind = 0, dim = 0;
    int64_t n = 0;
    std::vector<int> devices;
    std::vector<int64_t> lo;        // shard i holds rows [lo[i], lo[i + 1])
    std::vector<jv_dataset> shards;
    std::vector<ThreadCtx *> ctx;   // one persistent context per shard (worker threads come and go)
};

static void shard_ranges(int64_t n, int parts, std::vector<int64_t> &lo)
{
    lo.resize(parts + 1);
    const int64_t base = n / parts, rem = n % parts;
    for (int i = 0; i <= parts; i++) lo[i] = i * base + std::min<int64_t>(i, rem);
}

static int multi_devices(std::vector<int> &devs)
{
    devs.clear();
    for (int d = 0; d < MAX_DEVICES; d++)
        if (g_mask & (1u << d)) devs.push_back(d);
    if (devs.empty()) return fail(JV_ERR_NO_DEVICE, "jv_gpu_init_mask() has not succeeded");
    return JV_OK;
}

template <typename F>
static int multi_register(jv_multi m, F reg)
{
    int rc = multi_devices(m->devices);
    if (rc) return rc;
    const int parts = (int)std::min<int64_t>((int64_t)m->devices.size(), m->n);
    m->devices.resize(parts);
    shard_ranges(m->n, parts, m->lo);
    const int saved = t_device;
    for (int i = 0; i < parts; i++) {
        t_device = m->devices[i];
        jv_dataset ds = nullptr;
        rc = reg(i, m->lo[i], m->lo[i + 1] - m->lo[i], &ds);
        if (rc) break;
        m->shards.push_back(ds);
        m->ctx.push_back(new ThreadCtx());
    }
    t_device = saved;
    return rc;
}

extern "C" {

int jv_gpu_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

static int bind_device(int device)
{
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) return fail(JV_ERR_NO_DEVICE, std::string("no CUDA device: ") + cudaGetErrorString(e));
    if (device < 0 || device >= n || device >= MAX_DEVICES) return fail(JV_ERR_INVALID, "device index out of range");
    cudaDeviceProp p;
    CK(cudaGetDeviceProperties(&p, device), "cudaGetDeviceProperties");
    if (p.major != 10) return fail(JV_ERR_NO_DEVICE, "device is not sm_100 (this library carries sm_100a code only)");
    CK(cudaSetDevice(device), "cudaSetDevice");
    g_sm_counts[device] = p.multiProcessorCount;
    g_mask |= 1u << device;
    if (g_default_device < 0) g_default_device = device;
    return JV_OK;
}

int jv_gpu_init(int device)
{
    std::lock_guard<std::mutex> lk(g_mu);
    int rc = bind_device(device);
    if (rc) return rc;
    t_device = device;  // the calling thread creates its data sets here; handles remember their device, so a later
    return JV_OK;       // jv_gpu_init(other) never invalidates them
}

int jv_gpu_init_mask(uint32_t device_mask)
{
    std::lock_guard<std::mutex> lk(g_mu);
    if (device_mask == 0) return fail(JV_ERR_INVALID, "gpu_init_mask: empty mask");
    for (int d = 0; d < MAX_DEVICES; d++)
        if (device_mask & (1u << d)) {
            int rc = bind_device(d);
            if (rc) return rc;
        }
    // peer access between every pair (NVLink / NVSwitch): the multi-device entry points copy shard results device to device
    for (int a = 0; a < MAX_DEVICES; a++)
        for (int b = 0; b < MAX_DEVICES; b++)
            if (a != b && (g_mask & (1u << a)) && (g_mask & (1u << b))) {
                int can = 0;
                if (cudaDeviceCanAccessPeer(&can, a, b) == cudaSuccess && can) {
                    cudaSetDevice(a);
                    cudaError_t e = cudaDeviceEnablePeerAccess(b, 0);
                    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return cuda_fail(e, "cudaDeviceEnablePeerAccess");
                    cudaGetLastError();
                }
            }
    cudaSetDevice(g_default_device);
    return JV_OK;
}

int jv_gpu_set_device(int device)
{
    if (device < 0 || device >= MAX_DEVICES || !(g_mask & (1u << device))) return fail(JV_ERR_INVALID, "gpu_set_device: device was not bound by jv_gpu_init / jv_gpu_init_mask");
    t_device = device;
    return JV_OK;
}

uint32_t jv_gpu_bound_mask(void) { return g_mask; }

const char *jv_last_error(void) { return t_err.c_str(); }
const char *jv_version(void) { return "jvector-b200 0.1 (sm_100a)"; }
int jv_gpu_sm_count(void) { return g_default_device >= 0 ? g_sm_counts[t_device >= 0 ? t_device : g_default_device] : 0; }
int64_t jv_kernel_launch_count(void) { return (int64_t)g_launches.load(); }
static std::atomic<long long> g_rows_read{0};
int64_t jv_search_rows_read(void) { return (int64_t)g_rows_read.load(); }

// ------------------------------------------------------------------------------------------------ data sets
int jv_dataset_register_f32(const float *rows, int64_t n, int dim, jv_dataset *out)
{
    NEED_INIT();
    if (!rows || !out || n <= 0 || dim <= 0 || n > 0x7fffffffLL) return fail(JV_ERR_INVALID, "register_f32: bad arguments");
    jv_dataset ds = new jv_dataset_s();
    ds->device = t_active;
    memset(&ds->d, 0, sizeof(DataDesc));
    ds->d.kind = KIND_F32;
    ds->d.dim = dim;
    ds->d.n = n;
    ds->d.stride = round4(dim);
    float *dev = nullptr;
    int rc = ds->alloc((void **)&dev, (size_t)n * ds->d.stride * sizeof(float));
    if (rc) { delete ds; return rc; }
    cudaError_t e;
    if (ds->d.stride == dim) e = cudaMemcpy(dev, rows, (size_t)n * dim * sizeof(float), cudaMemcpyHostToDevice);
    else {
        e = cudaMemset(dev, 0, (size_t)n * ds->d.stride * sizeof(float));
        if (e == cudaSuccess)
            e = cudaMemcpy2D(dev, (size_t)ds->d.stride * 4, rows, (size_t)dim * 4, (size_t)dim * 4, (size_t)n, cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) { delete ds; return cuda_fail(e, "upload rows"); }
    ds->d.rows = dev;
    *out = ds;
    return JV_OK;
}

int jv_dataset_register_pq(const uint8_t *codes, int64_t n, int dim, int M, int k, const float *codebooks, const float *centroid, jv_dataset *out)
{
    NEED_INIT();
    if (!codes || !codebooks || !out || n <= 0 || dim <= 0 || M <= 0 || M > dim || k <= 0 || k > 256 || n > 0x7fffffffLL)
        return fail(JV_ERR_INVALID, "register_pq: bad arguments");
    jv_dataset ds = new jv_dataset_s();
    ds->device = t_active;
    memset(&ds->d, 0, sizeof(DataDesc));
    DataDesc &d = ds->d;
    d.kind = KIND_PQ; d.dim = dim; d.n = n; d.M = M; d.k = k; d.code_stride = round4(M);
    std::vector<int> sizes, offsets;
    pq_layout(dim, M, sizes, offsets);
    uint8_t *dcodes = nullptr;
    float *dcb = nullptr, *dcen = nullptr, *dmag = nullptr;
    int *dsz = nullptr, *doff = nullptr;
    int rc;
    if ((rc = ds->alloc((void **)&dcodes, (size_t)n * d.code_stride)) || (rc = ds->alloc((void **)&dcb, (size_t)k * dim * 4)) ||
        (rc = ds->alloc((void **)&dsz, (size_t)M * 4)) || (rc = ds->alloc((void **)&doff, (size_t)M * 4)) ||
        (rc = ds->alloc((void **)&dmag, (size_t)M * k * 4)) || (centroid && (rc = ds->alloc((void **)&dcen, (size_t)dim * 4)))) {
        delete ds;
        return rc;
    }
    cudaError_t e;
    if (d.code_stride == M) e = cudaMemcpy(dcodes, codes, (size_t)n * M, cudaMemcpyHostToDevice);
    else {
        e = cudaMemset(dcodes, 0, (size_t)n * d.code_stride);
        if (e == cudaSuccess) e = cudaMemcpy2D(dcodes, d.code_stride, codes, M, M, (size_t)n, cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) e = cudaMemcpy(dcb, codebooks, (size_t)k * dim * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dsz, sizes.data(), (size_t)M * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(doff, offsets.data(), (size_t)M * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess && centroid) e = cudaMemcpy(dcen, centroid, (size_t)dim * 4, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { delete ds; return cuda_fail(e, "upload pq"); }
    d.codes = dcodes; d.codebooks = dcb; d.sub_sizes = dsz; d.sub_offsets = doff; d.centroid = dcen; d.mag = dmag;
    e = launch_pq_self_magnitudes(d, dmag, 0);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { delete ds; return cuda_fail(e, "pq self magnitudes"); }
    *out = ds;
    return JV_OK;
}

int jv_dataset_register_bq(const uint64_t *words, int64_t n, int dim, jv_dataset *out)
{
    NEED_INIT();
    if (!words || !out || n <= 0 || dim <= 0 || n > 0x7fffffffLL) return fail(JV_ERR_INVALID, "register_bq: bad arguments");
    jv_dataset ds = new jv_dataset_s();
    ds->device = t_active;
    memset(&ds->d, 0, sizeof(DataDesc));
    ds->d.kind = KIND_BQ; ds->d.dim = dim; ds->d.n = n; ds->d.W = (dim + 63) / 64;
    unsigned long long *dw = nullptr;
    int rc = ds->alloc((void **)&dw, (size_t)n * ds->d.W * 8);
    if (rc) { delete ds; return rc; }
    cudaError_t e = cudaMemcpy(dw, words, (size_t)n * ds->d.W * 8, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { delete ds; return cuda_fail(e, "upload bq"); }
    ds->d.words = dw;
    *out = ds;
    return JV_OK;
}

int jv_dataset_register_nvq(const uint8_t *bytes, const float *params, int64_t n, int dim, int nsub, const float *mean, jv_dataset *out)
{
    NEED_INIT();
    if (!bytes || !params || !mean || !out || n <= 0 || dim <= 0 || nsub <= 0 || nsub > dim || n > 0x7fffffffLL)
        return fail(JV_ERR_INVALID, "register_nvq: bad arguments");
    jv_dataset ds = new jv_dataset_s();
    ds->device = t_active;
    memset(&ds->d, 0, sizeof(DataDesc));
    DataDesc &d = ds->d;
    d.kind = KIND_NVQ; d.dim = dim; d.n = n; d.nsub = nsub; d.stride = round4(dim); d.byte_stride = round4(dim);
    std::vector<int> sizes, offsets;
    pq_layout(dim, nsub, sizes, offsets);  // base:quantization/NVQuantization.java:236-251 uses the same split
    uint8_t *db = nullptr;
    float *dp = nullptr, *dm = nullptr;
    int *dsz = nullptr, *doff = nullptr;
    int rc;
    if ((rc = ds->alloc((void **)&db, (size_t)n * d.byte_stride)) || (rc = ds->alloc((void **)&dp, (size_t)n * nsub * 16)) ||
        (rc = ds->alloc((void **)&dm, (size_t)d.stride * 4)) || (rc = ds->alloc((void **)&dsz, (size_t)nsub * 4)) ||
        (rc = ds->alloc((void **)&doff, (size_t)nsub * 4))) {
        delete ds;
        return rc;
    }
    cudaError_t e;
    if (d.byte_stride == dim) e = cudaMemcpy(db, bytes, (size_t)n * dim, cudaMemcpyHostToDevice);
    else {
        e = cudaMemset(db, 0, (size_t)n * d.byte_stride);
        if (e == cudaSuccess) e = cudaMemcpy2D(db, d.byte_stride, bytes, dim, dim, (size_t)n, cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) e = cudaMemcpy(dp, params, (size_t)n * nsub * 16, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemset(dm, 0, (size_t)d.stride * 4);
    if (e == cudaSuccess) e = cudaMemcpy(dm, mean, (size_t)dim * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(dsz, sizes.data(), (size_t)nsub * 4, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(doff, offsets.data(), (size_t)nsub * 4, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { delete ds; return cuda_fail(e, "upload nvq"); }
    d.bytes = db; d.params = dp; d.mean = dm; d.sub_sizes = dsz; d.sub_offsets = doff;
    *out = ds;
    return JV_OK;
}

static int check_metric(const DataDesc &d, int metric);

int jv_dataset_pq_pair_table(jv_dataset pq, int metric)
{
    ON_DEVICE_OF(pq);
    if (pq->d.kind != KIND_PQ) return fail(JV_ERR_INVALID, "pq_pair_table: not a PQ data set");
    int rc = check_metric(pq->d, metric);
    if (rc) return rc;
    const int which = metric == JV_METRIC_EUCLIDEAN ? 0 : 1;  // cosine sums the dot-product table (ImmutablePQVectors.java:78-92)
    if (pq->d.pair_table[which]) return JV_OK;
    if ((rc = t_ctx.init())) return rc;
    float *t = nullptr;
    const size_t entries = (size_t)pq->d.M * ((size_t)pq->d.k * (pq->d.k + 1) / 2);
    if ((rc = pq->alloc((void **)&t, entries * 4))) return rc;
    CK(launch_pq_pair_table(pq->d, which == 0, t, t_ctx.stream), "pq_pair_table");
    CK(cudaStreamSynchronize(t_ctx.stream), "pq_pair_table");
    pq->d.pair_table[which] = t;
    return JV_OK;
}

int jv_dataset_pq_pair_table_download(jv_dataset pq, int metric, float *table_out)
{
    ON_DEVICE_OF(pq);
    const int which = metric == JV_METRIC_EUCLIDEAN ? 0 : 1;
    if (pq->d.kind != KIND_PQ || !pq->d.pair_table[which] || !table_out) return fail(JV_ERR_INVALID, "pq_pair_table_download: no table for this metric");
    const size_t entries = (size_t)pq->d.M * ((size_t)pq->d.k * (pq->d.k + 1) / 2);
    CK(cudaMemcpy(table_out, pq->d.pair_table[which], entries * 4, cudaMemcpyDeviceToHost), "D2H pair table");
    return JV_OK;
}

int jv_kmeans_assign_batch(const float *points, int64_t n, int dim, const float *centroids, int k, int32_t *assignments_out)
{
    NEED_INIT();
    if (!points || !centroids || !assignments_out || n <= 0 || dim <= 0 || k <= 0) return fail(JV_ERR_INVALID, "kmeans_assign: bad arguments");
    int rc;
    if ((rc = t_ctx.init()) || (rc = t_ctx.ensure(0, (size_t)n * dim * 4)) || (rc = t_ctx.ensure(1, (size_t)n * 4)) || (rc = t_ctx.ensure(2, (size_t)k * dim * 4))) return rc;
    cudaStream_t s = t_ctx.stream;
    CK(cudaMemcpyAsync(t_ctx.dbuf[0], points, (size_t)n * dim * 4, cudaMemcpyHostToDevice, s), "H2D points");
    CK(cudaMemcpyAsync(t_ctx.dbuf[2], centroids, (size_t)k * dim * 4, cudaMemcpyHostToDevice, s), "H2D centroids");
    CK(launch_kmeans_assign((const float *)t_ctx.dbuf[0], n, dim, dim, (const float *)t_ctx.dbuf[2], k, (int32_t *)t_ctx.dbuf[1], s), "kmeans_assign");
    CK(cudaMemcpyAsync(assignments_out, t_ctx.dbuf[1], (size_t)n * 4, cudaMemcpyDeviceToHost, s), "D2H assignments");
    CK(cudaStreamSynchronize(s), "sync");
    return JV_OK;
}

int jv_dataset_adopt_f32_device(const float *rows_device, int64_t n, int dim, int row_stride, jv_dataset *out)
{
    NEED_INIT();
    if (!rows_device || !out || n <= 0 || dim <= 0 || n > 0x7fffffffLL || row_stride < dim || (row_stride & 3) || ((uintptr_t)rows_device & 15))
        return fail(JV_ERR_INVALID, "adopt_f32_device: need 16-byte aligned rows and a row stride that is a multiple of 4 floats >= dim");
    if (row_stride != round4(dim)) return fail(JV_ERR_INVALID, "adopt_f32_device: row_stride must equal dim rounded up to 4 (padding floats must be zero)");
    jv_dataset ds = new jv_dataset_s();
    ds->device = t_active;
    ds->borrowed_rows = true;
    memset(&ds->d, 0, sizeof(DataDesc));
    ds->d.kind = KIND_F32;
    ds->d.dim = dim;
    ds->d.n = n;
    ds->d.stride = row_stride;
    ds->d.rows = rows_device;
    *out = ds;
    return JV_OK;
}

int jv_dataset_device(jv_dataset ds) { return ds ? ds->device : -1; }

int jv_dataset_free(jv_dataset ds)
{
    if (!ds) return JV_OK;
    cudaSetDevice(ds->device);
    cudaDeviceSynchronize();
    delete ds;
    return JV_OK;
}
int jv_dataset_invalidate_sketch(jv_dataset ds)
{
    ON_DEVICE_OF(ds);
    std::lock_guard<std::mutex> lk(ds->sketch_mu);
    CK(cudaDeviceSynchronize(), "invalidate_sketch: synchronize");
    if (ds->sketch_mem) cudaFree(ds->sketch_mem);
    ds->sketch_mem = nullptr;
    ds->sketch = {};
    ds->sketch_state = 0;
    return JV_OK;
}

int jv_dataset_f32_sketch(jv_dataset ds, int *state, double *captured, float *basis_out, float *proj_out, float *norms_out)
{
    ON_DEVICE_OF(ds);
    std::lock_guard<std::mutex> lk(ds->sketch_mu);
    if (state) *state = ds->sketch_state;
    if (captured) *captured = ds->sketch_captured;
    if (!basis_out && !proj_out && !norms_out) return JV_OK;
    if (ds->sketch_state != 1) return fail(JV_ERR_INVALID, "f32_sketch: the data set has no sketch");
    if (basis_out) CK(cudaMemcpy(basis_out, ds->sketch.basis, (size_t)SKETCH_K * ds->d.stride * 4, cudaMemcpyDeviceToHost), "D2H sketch basis");
    if (proj_out) CK(cudaMemcpy(proj_out, ds->sketch.proj, (size_t)ds->d.n * SKETCH_K * 4, cudaMemcpyDeviceToHost), "D2H sketch projections");
    if (norms_out) CK(cudaMemcpy(norms_out, ds->sketch.norms, (size_t)ds->d.n * 8, cudaMemcpyDeviceToHost), "D2H sketch norms");
    return JV_OK;
}

int64_t jv_dataset_size(jv_dataset ds) { return ds ? ds->d.n : 0; }
int jv_dataset_dim(jv_dataset ds) { return ds ? ds->d.dim : 0; }
int64_t jv_dataset_device_bytes(jv_dataset ds) { return ds ? (int64_t)ds->bytes : 0; }

// ------------------------------------------------------------------------------------------------ one query
static int check_metric(const DataDesc &d, int metric)
{
    if (metric < 0 || metric > 2) return fail(JV_ERR_INVALID, "unknown similarity function");
    (void)d;
    return JV_OK;
}

int jv_query_begin(jv_dataset ds, const float *q, int metric, jv_query *out)
{
    ON_DEVICE_OF(ds);
    if (!ds || !q || !out) return fail(JV_ERR_INVALID, "query_begin: null argument");
    int rc = check_metric(ds->d, metric);
    if (rc) return rc;
    if ((rc = t_ctx.init())) return rc;
    jv_query h = new jv_query_s();
    h->ds = ds;
    h->device = ds->device;
    h->metric = metric;
    cudaError_t e = cudaMalloc((void **)&h->blob, (size_t)blob_floats(ds->d) * 4);
    if (e != cudaSuccess) { delete h; return cuda_fail(e, "cudaMalloc(query)"); }
    if ((rc = t_ctx.ensure(0, (size_t)ds->d.dim * 4))) { cudaFree(h->blob); delete h; return rc; }
    cudaStream_t s = t_ctx.stream;
    e = cudaMemcpyAsync(t_ctx.dbuf[0], q, (size_t)ds->d.dim * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = launch_prepare(ds->d, metric, (const float *)t_ctx.dbuf[0], 1, h->blob, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) { cudaFree(h->blob); delete h; return cuda_fail(e, "prepare query"); }
    *out = h;
    return JV_OK;
}

int jv_score_batch(jv_query q, const int32_t *ids, int n, float *scores_out)
{
    ON_DEVICE_OF(q);
    if (!q || (n > 0 && (!ids || !scores_out)) || n < 0) return fail(JV_ERR_INVALID, "score_batch: bad arguments");
    if (n == 0) return JV_OK;
    int rc;
    if ((rc = t_ctx.init()) || (rc = t_ctx.ensure(1, (size_t)n * 4)) || (rc = t_ctx.ensure(2, (size_t)n * 4))) return rc;
    cudaStream_t s = t_ctx.stream;
    CK(cudaMemcpyAsync(t_ctx.dbuf[1], ids, (size_t)n * 4, cudaMemcpyHostToDevice, s), "H2D ids");
    CK(launch_score_ragged(q->ds->d, q->metric, q->blob, 1, (const int32_t *)t_ctx.dbuf[1], nullptr, n, n, (float *)t_ctx.dbuf[2], s), "score_ragged");
    CK(cudaMemcpyAsync(scores_out, t_ctx.dbuf[2], (size_t)n * 4, cudaMemcpyDeviceToHost, s), "D2H scores");
    CK(cudaStreamSynchronize(s), "sync");
    return JV_OK;
}

int jv_query_get_lut(jv_query q, float *lut_out)
{
    ON_DEVICE_OF(q);
    if (!q || !lut_out || q->ds->d.kind != KIND_PQ) return fail(JV_ERR_INVALID, "get_lut: not a PQ query");
    CK(cudaMemcpy(lut_out, q->blob, (size_t)q->ds->d.M * q->ds->d.k * 4, cudaMemcpyDeviceToHost), "D2H lut");
    return JV_OK;
}

int jv_query_end(jv_query q)
{
    if (!q) return JV_OK;
    cudaSetDevice(q->device);
    if (!q->pooled) cudaFree(q->blob);
    delete q;
    return JV_OK;
}

int jv_score_multi(jv_dataset ds, int metric, const float *queries, int nq, const int32_t *ids, const int32_t *offsets, float *scores_out)
{
    ON_DEVICE_OF(ds);
    if (!ds || !queries || !ids || !offsets || !scores_out || nq <= 0) return fail(JV_ERR_INVALID, "score_multi: bad arguments");
    if (nq > 65535) return fail(JV_ERR_INVALID, "score_multi: at most 65535 queries per call");
    int rc = check_metric(ds->d, metric);
    if (rc) return rc;
    const int total = offsets[nq];
    int maxc = 0;
    for (int i = 0; i < nq; i++) {
        if (offsets[i + 1] < offsets[i]) return fail(JV_ERR_INVALID, "score_multi: offsets not monotone");
        maxc = std::max(maxc, offsets[i + 1] - offsets[i]);
    }
    if (total == 0) return JV_OK;
    const size_t bf = (size_t)blob_floats(ds->d);
    if ((rc = t_ctx.init()) || (rc = t_ctx.ensure(0, (size_t)nq * ds->d.dim * 4)) || (rc = t_ctx.ensure(1, (size_t)total * 4)) ||
        (rc = t_ctx.ensure(2, (size_t)total * 4)) || (rc = t_ctx.ensure(3, (size_t)(nq + 1) * 4)) || (rc = t_ctx.ensure(4, (size_t)nq * bf * 4)))
        return rc;
    cudaStream_t s = t_ctx.stream;
    CK(cudaMemcpyAsync(t_ctx.dbuf[0], queries, (size_t)nq * ds->d.dim * 4, cudaMemcpyHostToDevice, s), "H2D queries");
    CK(cudaMemcpyAsync(t_ctx.dbuf[1], ids, (size_t)total * 4, cudaMemcpyHostToDevice, s), "H2D ids");
    CK(cudaMemcpyAsync(t_ctx.dbuf[3], offsets, (size_t)(nq + 1) * 4, cudaMemcpyHostToDevice, s), "H2D offsets");
    CK(launch_prepare(ds->d, metric, (const float *)t_ctx.dbuf[0], nq, (float *)t_ctx.dbuf[4], s), "prepare");
    CK(launch_score_ragged(ds->d, metric, (const float *)t_ctx.dbuf[4], nq, (const int32_t *)t_ctx.dbuf[1], (const int32_t *)t_ctx.dbuf[3], 0, maxc,
                           (float *)t_ctx.dbuf[2], s),
       "score_ragged");
    CK(cudaMemcpyAsync(scores_out, t_ctx.dbuf[2], (size_t)total * 4, cudaMemcpyDeviceToHost, s), "D2H scores");
    CK(cudaStreamSynchronize(s), "sync");
    return JV_OK;
}

int jv_score_pairs(jv_dataset ds, int metric, const int32_t *a, const int32_t *b, int n, float *scores_out)
{
    ON_DEVICE_OF(ds);
    if (!ds || n < 0 || (n > 0 && (!a || !b || !scores_out))) return fail(JV_ERR_INVALID, "score_pairs: bad arguments");
    if (ds->d.kind == KIND_NVQ) return fail(JV_ERR_UNSUPPORTED, "score_pairs: NVQ has no node-vs-node scorer in the reference");
    if (n == 0) return JV_OK;
    for (int i = 0; i < n; i++)
        if (a[i] < 0 || a[i] >= ds->d.n || b[i] < 0 || b[i] >= ds->d.n) return fail(JV_ERR_INVALID, "score_pairs: node id out of range");
    int rc = check_metric(ds->d, metric);
    if (rc) return rc;
    if ((rc = t_ctx.init()) || (rc = t_ctx.ensure(1, (size_t)n * 8)) || (rc = t_ctx.ensure(2, (size_t)n * 4))) return rc;
    cudaStream_t s = t_ctx.stream;
    int32_t *da = (int32_t *)t_ctx.dbuf[1], *db = da + n;
    CK(cudaMemcpyAsync(da, a, (size_t)n * 4, cudaMemcpyHostToDevice, s), "H2D a");
    CK(cudaMemcpyAsync(db, b, (size_t)n * 4, cudaMemcpyHostToDevice, s), "H2D b");
    CK(launch_score_pairs(ds->d, metric, da, db, n, (float *)t_ctx.dbuf[2], s), "score_pairs");
    CK(cudaMemcpyAsync(scores_out, t_ctx.dbuf[2], (size_t)n * 4, cudaMemcpyDeviceToHost, s), "D2H scores");
    CK(cudaStreamSynchronize(s), "sync");
    return JV_OK;
}

// generic exhaustive top-k (any storage kind): sample -> key threshold -> filtered pass -> per-query selection, with a host
// decision between passes (kernels_batch.cu). Queries and keys in HBM; id_base is added to every node id.
static int topk_device_generic(jv_dataset ds, int metric, const float *queries_dev, int nq, int k, int64_t id_base, long long *keys_dev)
{
    cudaStream_t s = t_ctx.stream;
    int rc;
    const size_t bf = (size_t)blob_floats(ds->d);
    const int chunk_max = (int)std::max<size_t>(1, std::min<size_t>(4096, ((size_t)512 << 20) / (bf * 4)));
    TopkScratch ts;
    ts.S = (int)std::min<long long>(ds->d.n, 16384);
    {
        // expected survivors of the aggressive threshold (see launch_topk_bruteforce): j n / S with j - 6 sqrt(j) >= k S / n
        const double f = (double)ts.S / (double)ds->d.n, kf = k * f;
        int ja = k;
        for (int j = 1; j < k; j++)
            if ((double)j - 6.0 * sqrt((double)j) >= kf) { ja = j; break; }
        const double expect = ds->d.n <= ts.S ? (double)ds->d.n : ja / f;
        ts.cap = expect * 2 > 8192 ? 16384 : (expect * 2 > 4096 ? 8192 : 4096);
        if (ts.cap < ts.S && ds->d.n <= ts.S) ts.cap = 16384;
    }
    for (int q0 = 0; q0 < nq; q0 += chunk_max) {
        const int cq = std::min(chunk_max, nq - q0);
        if ((rc = t_ctx.ensure(4, (size_t)cq * bf * 4)) || (rc = t_ctx.ensure(1, (size_t)ts.S * 4 + (size_t)cq * ts.S * 4 + 64)) ||
            (rc = t_ctx.ensure(2, (size_t)cq * 16 + (size_t)cq * 12 + 64 + (size_t)cq * ts.cap * 8)) || (rc = t_ctx.ensure(3, 64)))
            return rc;
        ts.sample_ids = (int32_t *)t_ctx.dbuf[1];
        ts.sample_scores = (float *)((char *)t_ctx.dbuf[1] + (((size_t)ts.S * 4 + 15) & ~(size_t)15));
        ts.buf = (long long *)t_ctx.dbuf[2];
        ts.thr = ts.buf + (size_t)cq * ts.cap;
        ts.thr_safe = ts.thr + cq;
        ts.cnt = (int *)(ts.thr_safe + cq);
        ts.qlist_a = ts.cnt + cq;
        ts.qlist_b = ts.qlist_a + cq;
        int *dflag = (int *)t_ctx.dbuf[3];
        CK(cudaMemsetAsync(dflag, 0, sizeof(int), s), "memset flag");
        CK(launch_prepare(ds->d, metric, queries_dev + (size_t)q0 * ds->d.dim, cq, (float *)t_ctx.dbuf[4], s), "prepare");
        CK(launch_topk_bruteforce(ds->d, metric, (const float *)t_ctx.dbuf[4], cq, k, ts, keys_dev + (size_t)q0 * k, dflag, s), "topk");
        if (id_base) CK(launch_key_rebase(keys_dev + (size_t)q0 * k, (long long)cq * k, (long long)id_base, s), "rebase");
        int flag = 0;
        CK(cudaMemcpyAsync(&flag, dflag, sizeof(int), cudaMemcpyDeviceToHost, s), "D2H flag");
        CK(cudaStreamSynchronize(s), "sync");
        if (flag) return fail(JV_ERR_OVERFLOW, "topk_bruteforce: candidate buffer overflow (adversarial score distribution)");
    }
    return JV_OK;
}

constexpr int IMMA_QUERY_CHUNK = 4096;  // queries per bq_imma launch sequence (bounds the capture buffers: 64 KB per query)

// BQ: the tensor-core contraction (bq_imma.cu), enqueued on `s` without any host synchronisation. status_dev receives the number of
// queries the integer-threshold path left unresolved (0 in the normal case).
static int topk_bq_imma_enqueue(jv_dataset ds, const float *queries_dev, int nq, int k, int64_t id_base, long long *keys_dev, int *status_dev, cudaStream_t s)
{
    int rc;
    const int chunk = std::min(nq, IMMA_QUERY_CHUNK);
    if ((rc = t_ctx.ensure(7, bq_imma_scratch_bytes(ds->d.n, chunk, ds->d.W) + 64))) return rc;
    int *tmp = (int *)((char *)t_ctx.dbuf[7] + bq_imma_scratch_bytes(ds->d.n, chunk, ds->d.W));
    for (int q0 = 0; q0 < nq; q0 += chunk) {
        const int cq = std::min(chunk, nq - q0);
        // one status word per call: chunks after the first accumulate through a scratch word
        int *st = q0 == 0 ? status_dev : tmp;
        CK(launch_bq_topk_imma(ds->d, queries_dev + (size_t)q0 * ds->d.dim, cq, k, (long long)id_base, t_ctx.dbuf[7], keys_dev + (size_t)q0 * k, st, g_sm_count, s), "bq_topk_imma");
        if (q0 > 0) CK(launch_add_int(status_dev, tmp, s), "status");
    }
    return JV_OK;
}

static int topk_device(jv_dataset ds, int metric, const float *queries_dev, int nq, int k, int64_t id_base, long long *keys_dev)
{
    const char *force = getenv("JV_BQ_BRUTEFORCE");  // "popc": keep the round-1 popcount kernels (A/B timing, fallback tests)
    if (bq_imma_supported(ds->d, k) && !(force && force[0] == 'p')) {
        int rc;
        if ((rc = t_ctx.ensure(3, 64))) return rc;
        int *dflag = (int *)t_ctx.dbuf[3];
        if ((rc = topk_bq_imma_enqueue(ds, queries_dev, nq, k, id_base, keys_dev, dflag, t_ctx.stream))) return rc;
        int unresolved = 0;
        CK(cudaMemcpyAsync(&unresolved, dflag, sizeof(int), cudaMemcpyDeviceToHost, t_ctx.stream), "D2H status");
        CK(cudaStreamSynchronize(t_ctx.stream), "sync");
        if (unresolved == 0) return JV_OK;
        // a Hamming bin wider than the capture buffer (very low dimension, or adversarial duplicates): the key-threshold path decides
    }
    return topk_device_generic(ds, metric, queries_dev, nq, k, id_base, keys_dev);
}

int jv_topk_bruteforce(jv_dataset ds, int metric, const float *queries, int nq, int k, int64_t *keys_out)
{
    ON_DEVICE_OF(ds);
    if (!ds || !queries || !keys_out || nq <= 0 || k <= 0) return fail(JV_ERR_INVALID, "topk_bruteforce: bad arguments");
    if (k > 2048) return fail(JV_ERR_INVALID, "topk_bruteforce: k <= 2048");
    int rc = check_metric(ds->d, metric);
    if (rc) return rc;
    if ((rc = t_ctx.init()) || (rc = t_ctx.ensure(0, (size_t)nq * ds->d.dim * 4)) || (rc = t_ctx.ensure(5, (size_t)nq * k * 8))) return rc;
    cudaStream_t s = t_ctx.stream;
    CK(cudaMemcpyAsync(t_ctx.dbuf[0], queries, (size_t)nq * ds->d.dim * 4, cudaMemcpyHostToDevice, s), "H2D queries");
    if ((rc = topk_device(ds, metric, (const float *)t_ctx.dbuf[0], nq, k, 0, (long long *)t_ctx.dbuf[5]))) return rc;
    CK(cudaMemcpyAsync(keys_out, t_ctx.dbuf[5], (size_t)nq * k * 8, cudaMemcpyDeviceToHost, s), "D2H keys");
    CK(cudaStreamSynchronize(s), "sync");
    return JV_OK;
}

int jv_topk_bruteforce_device(jv_dataset ds, int metric, const float *queries_device, int nq, int k, int64_t id_base, int64_t *keys_out_device)
{
    ON_DEVICE_OF(ds);
    if (!ds || !queries_device || !keys_out_device || nq <= 0 || k <= 0 || k > 2048 || id_base < 0) return fail(JV_ERR_INVALID, "topk_bruteforce_device: bad arguments");
    int rc = check_metric(ds->d, metric);
    if (rc) return rc;
    if ((rc = t_ctx.init())) return rc;
    return topk_device(ds, metric, queries_device, nq, k, id_base, (long long *)keys_out_device);
}

int jv_topk_merge_device(const int64_t *keys_in_device, int nq, int parts, int k, int64_t *keys_out_device)
{
    NEED_INIT();
    if (!keys_in_device || !keys_out_device || nq <= 0 || parts <= 0 || k <= 0 || (long long)parts * k > 16384) return fail(JV_ERR_INVALID, "topk_merge: bad arguments");
    int rc;
    if ((rc = t_ctx.init())) return rc;
    CK(launch_topk_merge((const long long *)keys_in_device, nq, parts, k, (long long *)keys_out_device, t_ctx.stream), "topk_merge");
    CK(cudaStreamSynchronize(t_ctx.stream), "sync");
    return JV_OK;
}

int jv_topk_bruteforce_device_async(jv_dataset ds, int metric, const float *queries_device, int nq, int k, int64_t id_base, int64_t *keys_out_device,
                                    int32_t *status_device, void *cuda_stream)
{
    ON_DEVICE_OF(ds);
    if (!queries_device || !keys_out_device || !status_device || nq <= 0 || k <= 0 || id_base < 0) return fail(JV_ERR_INVALID, "topk_bruteforce_device_async: bad arguments");
    (void)metric;
    if (!bq_imma_supported(ds->d, k)) return fail(JV_ERR_UNSUPPORTED, "topk_bruteforce_device_async: BQ data sets (even word count, n >= 4096) only; use jv_topk_bruteforce_device");
    int rc;
    if ((rc = t_ctx.init())) return rc;
    return topk_bq_imma_enqueue(ds, queries_device, nq, k, id_base, (long long *)keys_out_device, status_device, (cudaStream_t)cuda_stream);
}

int jv_topk_merge_device_async(const int64_t *keys_in_device, int nq, int parts, int k, int64_t *keys_out_device, void *cuda_stream)
{
    NEED_INIT();
    if (!keys_in_device || !keys_out_device || nq <= 0 || parts <= 0 || k <= 0 || (long long)parts * k > 16384) return fail(JV_ERR_INVALID, "topk_merge: bad arguments");
    CK(launch_topk_merge_strided((const long long *)keys_in_device, nq, parts, k, (long long *)keys_out_device, (cudaStream_t)cuda_stream), "topk_merge");
    return JV_OK;
}

// ------------------------------------------------------------------------------------------------ encoders
static int bq_encode_impl(const float *rows_host, const float *rows_dev, int row_stride, int64_t n, int dim, uint64_t *words_out)
{
    int rc;
    const int W = (dim + 63) / 64;
    if ((rc = t_ctx.init()) || (rows_host && (rc = t_ctx.ensure(0, (size_t)n * dim * 4))) || (rc = t_ctx.ensure(1, (size_t)n * W * 8))) return rc;
    cudaStream_t s = t_ctx.stream;
    if (rows_host) {
        CK(cudaMemcpyAsync(t_ctx.dbuf[0], rows_host, (size_t)n * dim * 4, cudaMemcpyHostToDevice, s), "H2D rows");
        rows_dev = (const float *)t_ctx.dbuf[0];
        row_stride = dim;
    }
    CK(launch_bq_encode(rows_dev, n, dim, row_stride, (unsigned long long *)t_ctx.dbuf[1], s), "bq_encode");
    CK(cudaMemcpyAsync(words_out, t_ctx.dbuf[1], (size_t)n * W * 8, cudaMemcpyDeviceToHost, s), "D2H words");
    CK(cudaStreamSynchronize(s), "sync");
    return JV_OK;
}

int jv_bq_encode_batch(const float *rows, int64_t n, int dim, uint64_t *words_out)
{
    NEED_INIT();
    if (!rows || !words_out || n <= 0 || dim <= 0) return fail(JV_ERR_INVALID, "bq_encode: bad arguments");
    return bq_encode_impl(rows, nullptr, 0, n, dim, words_out);
}

int jv_bq_encode_dataset(jv_dataset f32, uint64_t *words_out)
{
    ON_DEVICE_OF(f32);
    if (!f32 || f32->d.kind != KIND_F32 || !words_out) return fail(JV_ERR_INVALID, "bq_encode_dataset: needs an fp32 data set");
    return bq_encode_impl(nullptr, f32->d.rows, f32->d.stride, f32->d.n, f32->d.dim, words_out);
}

static int pq_encode_impl(const float *rows, const float *rows_dev, int row_stride, int64_t n, int dim, int M, int k, const float *codebooks,
                          const float *centroid, uint8_t *codes_out)
{
    int rc;
    std::vector<int> sizes, offsets;
    pq_layout(dim, M, sizes, offsets);
    const size_t cb_bytes = (size_t)k * dim * 4;
    const size_t aux = cb_bytes + (size_t)dim * 4 + (size_t)M * 8 + 64;
    if ((rc = t_ctx.init()) || (rows && (rc = t_ctx.ensure(0, (size_t)n * dim * 4))) || (rc = t_ctx.ensure(1, (size_t)n * M)) || (rc = t_ctx.ensure(2, aux))) return rc;
    cudaStream_t s = t_ctx.stream;
    char *a = (char *)t_ctx.dbuf[2];
    float *dcb = (float *)a, *dcen = (float *)(a + cb_bytes);
    int *dsz = (int *)(a + cb_bytes + (size_t)dim * 4), *doff = dsz + M;
    if (rows) {
        CK(cudaMemcpyAsync(t_ctx.dbuf[0], rows, (size_t)n * dim * 4, cudaMemcpyHostToDevice, s), "H2D rows");
        rows_dev = (const float *)t_ctx.dbuf[0];
        row_stride = dim;
    }
    CK(cudaMemcpyAsync(dcb, codebooks, cb_bytes, cudaMemcpyHostToDevice, s), "H2D codebooks");
    if (centroid) CK(cudaMemcpyAsync(dcen, centroid, (size_t)dim * 4, cudaMemcpyHostToDevice, s), "H2D centroid");
    CK(cudaMemcpyAsync(dsz, sizes.data(), (size_t)M * 4, cudaMemcpyHostToDevice, s), "H2D sizes");
    CK(cudaMemcpyAsync(doff, offsets.data(), (size_t)M * 4, cudaMemcpyHostToDevice, s), "H2D offsets");
    DataDesc d;
    memset(&d, 0, sizeof(d));
    d.kind = KIND_PQ; d.dim = dim; d.n = n; d.M = M; d.k = k; d.codebooks = dcb; d.sub_sizes = dsz; d.sub_offsets = doff; d.centroid = centroid ? dcen : nullptr;
    CK(launch_pq_encode(d, rows_dev, n, row_stride, (uint8_t *)t_ctx.dbuf[1], s), "pq_encode");
    CK(cudaMemcpyAsync(codes_out, t_ctx.dbuf[1], (size_t)n * M, cudaMemcpyDeviceToHost, s), "D2H codes");
    CK(cudaStreamSynchronize(s), "sync");
    return JV_OK;
}

int jv_pq_encode_batch(const float *rows, int64_t n, int dim, int M, int k, const float *codebooks, const float *centroid, uint8_t *codes_out)
{
    NEED_INIT();
    if (!rows || !codebooks || !codes_out || n <= 0 || dim <= 0 || M <= 0 || M > dim || k <= 0 || k > 256) return fail(JV_ERR_INVALID, "pq_encode: bad arguments");
    return pq_encode_impl(rows, nullptr, 0, n, dim, M, k, codebooks, centroid, codes_out);
}

int jv_pq_encode_dataset(jv_dataset f32, int M, int k, const float *codebooks, const float *centroid, uint8_t *codes_out)
{
    ON_DEVICE_OF(f32);
    if (!f32 || f32->d.kind != KIND_F32 || !codebooks || !codes_out || M <= 0 || M > f32->d.dim || k <= 0 || k > 256)
        return fail(JV_ERR_INVALID, "pq_encode_dataset: bad arguments");
    return pq_encode_impl(nullptr, f32->d.rows, f32->d.stride, f32->d.n, f32->d.dim, M, k, codebooks, centroid, codes_out);
}

static int nvq_encode_impl(const float *rows, const float *rows_dev, int row_stride, int64_t n, int dim, int nsub, const float *mean, int learn,
                           float *params_out, uint8_t *bytes_out)
{
    int rc;
    std::vector<int> sizes, offsets;
    pq_layout(dim, nsub, sizes, offsets);
    const size_t aux = (size_t)dim * 4 + (size_t)nsub * 8 + 64;
    if ((rc = t_ctx.init()) || (rows && (rc = t_ctx.ensure(0, (size_t)n * dim * 4))) || (rc = t_ctx.ensure(1, (size_t)n * dim)) ||
        (rc = t_ctx.ensure(2, aux)) || (rc = t_ctx.ensure(3, (size_t)n * nsub * 16)))
        return rc;
    cudaStream_t s = t_ctx.stream;
    char *a = (char *)t_ctx.dbuf[2];
    float *dmean = (float *)a;
    int *dsz = (int *)(a + (size_t)dim * 4), *doff = dsz + nsub;
    if (rows) {
        CK(cudaMemcpyAsync(t_ctx.dbuf[0], rows, (size_t)n * dim * 4, cudaMemcpyHostToDevice, s), "H2D rows");
        rows_dev = (const float *)t_ctx.dbuf[0];
        row_stride = dim;
    }
    CK(cudaMemcpyAsync(dmean, mean, (size_t)dim * 4, cudaMemcpyHostToDevice, s), "H2D mean");
    CK(cudaMemcpyAsync(dsz, sizes.data(), (size_t)nsub * 4, cudaMemcpyHostToDevice, s), "H2D sizes");
    CK(cudaMemcpyAsync(doff, offsets.data(), (size_t)nsub * 4, cudaMemcpyHostToDevice, s), "H2D offsets");
    CK(launch_nvq_encode(rows_dev, n, row_stride, nsub, dsz, doff, dmean, learn, (float *)t_ctx.dbuf[3], (uint8_t *)t_ctx.dbuf[1], dim, s), "nvq_encode");
    CK(cudaMemcpyAsync(params_out, t_ctx.dbuf[3], (size_t)n * nsub * 16, cudaMemcpyDeviceToHost, s), "D2H params");
    CK(cudaMemcpyAsync(bytes_out, t_ctx.dbuf[1], (size_t)n * dim, cudaMemcpyDeviceToHost, s), "D2H bytes");
    CK(cudaStreamSynchronize(s), "sync");
    return JV_OK;
}

int jv_nvq_encode_batch(const float *rows, int64_t n, int dim, int nsub, const float *mean, int learn, float *params_out, uint8_t *bytes_out)
{
    NEED_INIT();
    if (!rows || !mean || !params_out || !bytes_out || n <= 0 || dim <= 0 || nsub <= 0 || nsub > dim) return fail(JV_ERR_INVALID, "nvq_encode: bad arguments");
    return nvq_encode_impl(rows, nullptr, 0, n, dim, nsub, mean, learn, params_out, bytes_out);
}

int jv_nvq_encode_dataset(jv_dataset f32, int nsub, const float *mean, int learn, float *params_out, uint8_t *bytes_out)
{
    ON_DEVICE_OF(f32);
    if (!f32 || f32->d.kind != KIND_F32 || !mean || !params_out || !bytes_out || nsub <= 0 || nsub > f32->d.dim)
        return fail(JV_ERR_INVALID, "nvq_encode_dataset: bad arguments");
    return nvq_encode_impl(nullptr, f32->d.rows, f32->d.stride, f32->d.n, f32->d.dim, nsub, mean, learn, params_out, bytes_out);
}

// NVQ "inline vectors" without a host round trip: encode the resident fp32 rows into a new resident NVQ data set
int jv_nvq_encode_dataset_resident(jv_dataset f32, int nsub, const float *mean, int learn, jv_dataset *out)
{
    ON_DEVICE_OF(f32);
    if (f32->d.kind != KIND_F32 || !mean || !out || nsub <= 0 || nsub > f32->d.dim) return fail(JV_ERR_INVALID, "nvq_encode_dataset_resident: bad arguments");
    int rc;
    if ((rc = t_ctx.init())) return rc;
    const int dim = f32->d.dim;
    const int64_t n = f32->d.n;
    jv_dataset ds = new jv_dataset_s();
    ds->device = f32->device;
    memset(&ds->d, 0, sizeof(DataDesc));
    DataDesc &d = ds->d;
    d.kind = KIND_NVQ; d.dim = dim; d.n = n; d.nsub = nsub; d.stride = round4(dim); d.byte_stride = round4(dim);
    std::vector<int> sizes, offsets;
    pq_layout(dim, nsub, sizes, offsets);
    uint8_t *db = nullptr;
    float *dp = nullptr, *dm = nullptr;
    int *dsz = nullptr, *doff = nullptr;
    if ((rc = ds->alloc((void **)&db, (size_t)n * d.byte_stride)) || (rc = ds->alloc((void **)&dp, (size_t)n * nsub * 16)) ||
        (rc = ds->alloc((void **)&dm, (size_t)d.stride * 4)) || (rc = ds->alloc((void **)&dsz, (size_t)nsub * 4)) ||
        (rc = ds->alloc((void **)&doff, (size_t)nsub * 4))) {
        delete ds;
        return rc;
    }
    cudaStream_t s = t_ctx.stream;
    cudaError_t e = cudaMemsetAsync(dm, 0, (size_t)d.stride * 4, s);
    if (e == cudaSuccess && d.byte_stride != dim) e = cudaMemsetAsync(db, 0, (size_t)n * d.byte_stride, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dm, mean, (size_t)dim * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(dsz, sizes.data(), (size_t)nsub * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(doff, offsets.data(), (size_t)nsub * 4, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = launch_nvq_encode(f32->d.rows, n, f32->d.stride, nsub, dsz, doff, dm, learn, dp, db, d.byte_stride, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);
    if (e != cudaSuccess) { delete ds; return cuda_fail(e, "nvq_encode_dataset_resident"); }
    d.bytes = db; d.params = dp; d.mean = dm; d.sub_sizes = dsz; d.sub_offsets = doff;
    *out = ds;
    return JV_OK;
}

// ------------------------------------------------------------------------------------------------ graph
int jv_graph_create(int32_t n, int degree, const int32_t *adj0, int32_t entry_node, jv_graph *out)
{
    NEED_INIT();
    if (!adj0 || !out || n <= 0 || degree <= 0 || degree > MAX_DEGREE || entry_node < 0 || entry_node >= n)
        return fail(JV_ERR_INVALID, "graph_create: bad arguments");
    // one pass over data that is copied anyway: a neighbour id outside [-1, n) would be an illegal address inside the search kernel
    for (size_t i = 0, tot = (size_t)n * degree; i < tot; i++)
        if (adj0[i] < -1 || adj0[i] >= n) return fail(JV_ERR_INVALID, "graph_create: neighbour id out of range");
    jv_graph g = new jv_graph_s();
    g->device = t_active;
    memset(&g->g, 0, sizeof(GraphDesc));
    cudaError_t e = cudaMalloc((void **)&g->adj0, (size_t)n * degree * 4);
    if (e == cudaSuccess) e = cudaMemcpy(g->adj0, adj0, (size_t)n * degree * 4, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { delete g; return cuda_fail(e, "upload adjacency"); }
    g->g.n = n; g->g.degree = degree; g->g.levels = 1; g->g.entry_node = entry_node; g->g.entry_level = 0; g->g.adj0 = g->adj0;
    *out = g;
    return JV_OK;
}

static int graph_rebuild_upper(jv_graph g)
{
    const int L = (int)g->level_ids.size();
    cudaFree(g->upper_row); cudaFree(g->upper_adj); cudaFree(g->upper_off);
    g->upper_row = nullptr; g->upper_adj = nullptr; g->upper_off = nullptr;
    if (L == 0) return JV_OK;
    const int n = g->g.n, degree = g->g.degree;
    std::vector<int32_t> rows((size_t)L * n, -1);
    std::vector<long long> offs(L);
    std::vector<int32_t> adj;
    long long o = 0;
    for (int l = 0; l < L; l++) {
        offs[l] = o;
        for (size_t i = 0; i < g->level_ids[l].size(); i++) rows[(size_t)l * n + g->level_ids[l][i]] = (int32_t)i;
        adj.insert(adj.end(), g->level_adj[l].begin(), g->level_adj[l].end());
        o += (long long)g->level_ids[l].size();
    }
    CK(cudaMalloc((void **)&g->upper_row, rows.size() * 4), "cudaMalloc(upper_row)");
    CK(cudaMalloc((void **)&g->upper_adj, std::max<size_t>(adj.size(), 1) * 4), "cudaMalloc(upper_adj)");
    CK(cudaMalloc((void **)&g->upper_off, (size_t)L * 8), "cudaMalloc(upper_off)");
    CK(cudaMemcpy(g->upper_row, rows.data(), rows.size() * 4, cudaMemcpyHostToDevice), "H2D upper_row");
    CK(cudaMemcpy(g->upper_adj, adj.data(), adj.size() * 4, cudaMemcpyHostToDevice), "H2D upper_adj");
    CK(cudaMemcpy(g->upper_off, offs.data(), (size_t)L * 8, cudaMemcpyHostToDevice), "H2D upper_off");
    g->g.upper_row = g->upper_row; g->g.upper_adj = g->upper_adj; g->g.upper_off = g->upper_off;
    g->g.levels = L + 1;
    g->g.entry_level = L;
    (void)degree;
    return JV_OK;
}

int jv_graph_add_level(jv_graph g, int32_t count, const int32_t *node_ids, const int32_t *adj)
{
    ON_DEVICE_OF(g);
    if (!g || count <= 0 || !node_ids || !adj) return fail(JV_ERR_INVALID, "graph_add_level: bad arguments");
    for (size_t i = 0, tot = (size_t)count * g->g.degree; i < tot; i++)
        if (adj[i] < -1 || adj[i] >= g->g.n) return fail(JV_ERR_INVALID, "graph_add_level: neighbour id out of range");
    bool has_entry = false;
    for (int i = 0; i < count; i++) {
        if (node_ids[i] < 0 || node_ids[i] >= g->g.n) return fail(JV_ERR_INVALID, "graph_add_level: node id out of range");
        if (node_ids[i] == g->g.entry_node) has_entry = true;
    }
    if (!has_entry) return fail(JV_ERR_INVALID, "graph_add_level: the entry node must belong to every level");
    g->level_ids.emplace_back(node_ids, node_ids + count);
    g->level_adj.emplace_back(adj, adj + (size_t)count * g->g.degree);
    return graph_rebuild_upper(g);
}

int jv_graph_fuse_pq(jv_graph g, jv_dataset pq)
{
    ON_DEVICE_OF(g);
    if (!pq || pq->d.kind != KIND_PQ) return fail(JV_ERR_INVALID, "graph_fuse_pq: needs a PQ data set");
    if (pq->device != g->device || pq->d.n != g->g.n) return fail(JV_ERR_INVALID, "graph_fuse_pq: data set and graph differ in device or size");
    int rc;
    if ((rc = t_ctx.init())) return rc;
    const int rec = (g->g.degree * (4 + pq->d.code_stride) + 15) & ~15;
    cudaFree(g->fused);
    g->fused = nullptr;
    g->g.fused = nullptr;
    CK(cudaMalloc((void **)&g->fused, (size_t)g->g.n * rec), "cudaMalloc(fused records)");
    CK(launch_fuse_pq(g->g, pq->d, g->fused, rec, t_ctx.stream), "fuse_pq");
    CK(cudaStreamSynchronize(t_ctx.stream), "fuse_pq");
    g->g.fused = g->fused;
    g->g.fused_codes_of = pq->d.codes;
    g->g.fused_rec = rec;
    g->g.fused_code_stride = pq->d.code_stride;
    return JV_OK;
}

int jv_graph_fused_download(jv_graph g, uint8_t *records_out, int *record_bytes)
{
    ON_DEVICE_OF(g);
    if (!g->fused) return fail(JV_ERR_INVALID, "graph_fused_download: jv_graph_fuse_pq has not been called");
    if (record_bytes) *record_bytes = g->g.fused_rec;
    if (records_out) CK(cudaMemcpy(records_out, g->fused, (size_t)g->g.n * g->g.fused_rec, cudaMemcpyDeviceToHost), "D2H fused records");
    return JV_OK;
}

int jv_graph_free(jv_graph g)
{
    if (!g) return JV_OK;
    cudaSetDevice(g->device);
    cudaDeviceSynchronize();
    delete g;
    return JV_OK;
}

int jv_graph_info(jv_graph g, int32_t *n, int *degree, int *levels, int32_t *entry_node)
{
    if (!g) return fail(JV_ERR_INVALID, "graph_info: null graph");
    if (n) *n = g->g.n;
    if (degree) *degree = g->g.degree;
    if (levels) *levels = g->g.levels;
    if (entry_node) *entry_node = g->g.entry_node;
    return JV_OK;
}

int jv_graph_download(jv_graph g, int level, int32_t *node_ids_out, int32_t *adj_out, int32_t *count_out)
{
    ON_DEVICE_OF(g);
    if (!g || level < 0 || level >= g->g.levels) return fail(JV_ERR_INVALID, "graph_download: bad level");
    if (level == 0) {
        if (count_out) *count_out = g->g.n;
        if (node_ids_out)
            for (int i = 0; i < g->g.n; i++) node_ids_out[i] = i;
        if (adj_out) CK(cudaMemcpy(adj_out, g->adj0, (size_t)g->g.n * g->g.degree * 4, cudaMemcpyDeviceToHost), "D2H adjacency");
        return JV_OK;
    }
    const auto &ids = g->level_ids[level - 1];
    if (count_out) *count_out = (int32_t)ids.size();
    if (node_ids_out) memcpy(node_ids_out, ids.data(), ids.size() * 4);
    if (adj_out) memcpy(adj_out, g->level_adj[level - 1].data(), g->level_adj[level - 1].size() * 4);
    return JV_OK;
}

// The sketch pays where a walk's rows come from HBM: rows of at least 1 KB (a sketch line + norms cost 160 bytes of reads) and a data
// set of at least twice the 126 MB L2. JV_F32_SKETCH=0 turns it off.
static bool sketch_wanted(const jv_dataset approx, int metric)
{
    if (approx->d.kind != KIND_F32 || metric != JV_METRIC_DOT || approx->d.dim < 256) return false;
    if ((double)approx->d.n * approx->d.stride * 4 < 2.0 * 126e6) return false;
    const char *e = getenv("JV_F32_SKETCH");
    return !(e && e[0] == '0');
}

static int sketch_ensure(jv_dataset ds, cudaStream_t s)
{
    std::lock_guard<std::mutex> lk(ds->sketch_mu);
    if (ds->sketch_state != 0) return JV_OK;
    const size_t bytes = f32_sketch_bytes(ds->d);
    CK(cudaMalloc(&ds->sketch_mem, bytes), "cudaMalloc(sketch)");
    cudaError_t e = build_f32_sketch(ds->d, ds->sketch_mem, &ds->sketch, &ds->sketch_captured, s);
    if (e != cudaSuccess) {
        cudaFree(ds->sketch_mem);
        ds->sketch_mem = nullptr;
        return cuda_fail(e, "build_f32_sketch");
    }
    // 32 of 768 directions of i.i.d. rows hold ~4 % of their energy: the bound would drop nothing and cost 160 bytes a candidate
    if (ds->sketch_captured < 0.5) {
        cudaFree(ds->sketch_mem);
        ds->sketch_mem = nullptr;
        ds->sketch = {};
        ds->sketch_state = -1;
    } else ds->sketch_state = 1;
    return JV_OK;
}

static int search_device(jv_graph g, jv_dataset approx, jv_dataset reranker, int metric, const float *queries_dev, int nq, int topK, int rerankK,
                         const SearchFilter *filter, int32_t *nodes_dev, float *scores_dev, jv_search_stats *stats)
{
    if (!g || !approx || !queries_dev || !nodes_dev || !scores_dev || nq <= 0) return fail(JV_ERR_INVALID, "graph_search: bad arguments");
    if (topK < 1 || rerankK < topK) return fail(JV_ERR_INVALID, "graph_search: need 1 <= topK <= rerankK");
    if (rerankK > 4096) return fail(JV_ERR_INVALID, "graph_search: rerankK <= 4096");
    if (approx->d.n != g->g.n) return fail(JV_ERR_INVALID, "graph_search: data set and graph sizes differ");
    if (approx->device != g->device || (reranker && reranker->device != g->device)) return fail(JV_ERR_INVALID, "graph_search: graph and data sets live on different devices");
    if (reranker && (reranker->d.n != g->g.n || reranker->d.dim != approx->d.dim)) return fail(JV_ERR_INVALID, "graph_search: reranker shape mismatch");
    if (reranker && reranker->d.kind != KIND_F32 && reranker->d.kind != KIND_NVQ)
        return fail(JV_ERR_UNSUPPORTED, "graph_search: the reranker must be fp32 or NVQ (OnDiskGraphIndex.java:705-713)");
    int rc = check_metric(approx->d, metric);
    if (rc) return rc;
    if ((rc = t_ctx.init())) return rc;
    cudaStream_t s = t_ctx.stream;
    const DataDesc *rr = reranker ? &reranker->d : nullptr;
    const F32Sketch *sketch = nullptr;
    if (sketch_wanted(approx, metric)) {
        if ((rc = sketch_ensure(approx, s))) return rc;
        if (approx->sketch_state == 1) sketch = &approx->sketch;
    }
    SearchPlan plan;
    // JV_VISITED_CAP / JV_LIST_CAP: first visited-table / candidate-list sizes (testing and tuning knobs; queries that outgrow
    // either are re-run below with 4x)
    const char *cap_env = getenv("JV_VISITED_CAP");
    const char *lcap_env = getenv("JV_LIST_CAP");
    const int cap_hint = cap_env ? atoi(cap_env) : 0, lcap_hint = lcap_env ? atoi(lcap_env) : 0;
    CK(plan_search(approx->d, rr, g->g, topK, rerankK, nq, cap_hint > 0 ? cap_hint : 0, lcap_hint > 0 ? lcap_hint : 0, g_sm_count, &plan), "plan_search");
    const size_t aux = sizeof(SearchCounters) + 64 + (size_t)nq + (size_t)nq * 4 + 64;
    if ((rc = t_ctx.ensure(5, search_scratch_bytes(plan))) || (rc = t_ctx.ensure(3, aux))) return rc;
    char *a = (char *)t_ctx.dbuf[3];
    SearchCounters *dcnt = (SearchCounters *)a;
    int *dwork = (int *)(a + sizeof(SearchCounters));
    uint8_t *dover = (uint8_t *)(a + sizeof(SearchCounters) + 64);
    int32_t *dindex = (int32_t *)(a + sizeof(SearchCounters) + 64 + (((size_t)nq + 63) & ~(size_t)63));
    CK(cudaMemsetAsync(dcnt, 0, sizeof(SearchCounters), s), "memset counters");
    CK(cudaEventRecord(t_ctx.ev0, s), "event");
    CK(launch_search(g->g, approx->d, rr, metric, queries_dev, nq, topK, rerankK, plan, t_ctx.dbuf[5], dwork, nodes_dev, scores_dev, dcnt, dover, nullptr, 0, filter, s,
                     sketch),
       "launch_search");
    CK(cudaEventRecord(t_ctx.ev1, s), "event");
    SearchCounters hc;
    CK(cudaMemcpyAsync(&hc, dcnt, sizeof(hc), cudaMemcpyDeviceToHost, s), "D2H counters");
    CK(cudaStreamSynchronize(s), "search kernel");
    float ms = 0.f;
    cudaEventElapsedTime(&ms, t_ctx.ev0, t_ctx.ev1);
    long long retried = 0;
    int cap = plan.visited_cap, lcap = plan.list_cap;
    // queries whose visited table filled up (code 1) or whose candidate list could not hold a tie tail (code 2) are re-run with a
    // 4x larger table / list: the result does not depend on either size, only whether the run completes does
    for (int attempt = 0; hc.overflowed > 0 && attempt < 6; attempt++) {
        std::vector<uint8_t> hover(nq);
        CK(cudaMemcpy(hover.data(), dover, (size_t)nq, cudaMemcpyDeviceToHost), "D2H overflow flags");
        std::vector<int32_t> idx;
        bool need_table = false, need_list = false;
        for (int i = 0; i < nq; i++)
            if (hover[i]) {
                idx.push_back(i);
                if (hover[i] == 1) need_table = true;
                else need_list = true;
            }
        if (idx.empty()) break;
        retried += (long long)idx.size();
        if (need_table) cap *= 4;
        if (need_list) {
            if (lcap >= MAX_LIST_CAP) return fail(JV_ERR_OVERFLOW, "graph_search: more equal-score (or filtered-out) candidates than the longest candidate list holds");
            lcap = std::min(MAX_LIST_CAP, lcap * 4);
        }
        SearchPlan p2;
        CK(plan_search(approx->d, rr, g->g, topK, rerankK, (int)idx.size(), cap, lcap, g_sm_count, &p2), "plan_search(retry)");
        if ((rc = t_ctx.ensure(5, search_scratch_bytes(p2)))) return rc;
        CK(cudaMemcpyAsync(dindex, idx.data(), idx.size() * 4, cudaMemcpyHostToDevice, s), "H2D retry index");
        unsigned long long zero = 0;
        CK(cudaMemcpyAsync(&dcnt->overflowed, &zero, sizeof(zero), cudaMemcpyHostToDevice, s), "reset overflow");
        CK(cudaEventRecord(t_ctx.ev0, s), "event");
        CK(launch_search(g->g, approx->d, rr, metric, queries_dev, (int)idx.size(), topK, rerankK, p2, t_ctx.dbuf[5], dwork, nodes_dev, scores_dev, dcnt, dover,
                         dindex, 0, filter, s, sketch),
           "launch_search(retry)");
        CK(cudaEventRecord(t_ctx.ev1, s), "event");
        CK(cudaMemcpyAsync(&hc, dcnt, sizeof(hc), cudaMemcpyDeviceToHost, s), "D2H counters");
        CK(cudaStreamSynchronize(s), "search kernel (retry)");
        float ms2 = 0.f;
        cudaEventElapsedTime(&ms2, t_ctx.ev0, t_ctx.ev1);
        ms += ms2;
    }
    if (hc.overflowed > 0) return fail(JV_ERR_OVERFLOW, "graph_search: visited table / candidate list overflow after retries");
    g_rows_read += (long long)hc.rows_read;  // the counters add up over the re-runs (only `overflowed` is reset)
    if (stats) {
        stats->visited = (int64_t)hc.visited;
        stats->expanded = (int64_t)hc.expanded;
        stats->expanded_base = (int64_t)hc.expanded_base;
        stats->reranked = (int64_t)hc.reranked;
        stats->retried = retried;
        stats->device_ms = ms;
    }
    return JV_OK;
}

// jv_search_options -> device-side SearchFilter (the bitset is uploaded when it is a host pointer)
static int make_filter(const jv_search_options *opts, jv_graph g, int nq, bool bits_on_device, SearchFilter *f, bool *use)
{
    *use = false;
    memset(f, 0, sizeof(*f));
    if (!opts) return JV_OK;
    if (opts->threshold < 0.f || opts->rerank_floor < 0.f || opts->accept_stride_words < 0) return fail(JV_ERR_INVALID, "graph_search: negative threshold / rerankFloor / stride");
    f->threshold = opts->threshold;
    f->rerank_floor = opts->rerank_floor;
    f->lenient = 0;
    f->accept_stride_words = opts->accept_stride_words;
    if (opts->accept_bits) {
        const size_t words = ((size_t)g->g.n + 31) / 32;
        if (opts->accept_stride_words != 0 && (size_t)opts->accept_stride_words < words) return fail(JV_ERR_INVALID, "graph_search: accept_stride_words shorter than one bitset");
        if (bits_on_device) f->accept_bits = opts->accept_bits;
        else {
            const size_t total = opts->accept_stride_words ? (size_t)opts->accept_stride_words * (size_t)(nq - 1) + words : words;
            int rc = t_ctx.ensure(6, total * 4);
            if (rc) return rc;
            CK(cudaMemcpyAsync(t_ctx.dbuf[6], opts->accept_bits, total * 4, cudaMemcpyHostToDevice, t_ctx.stream), "H2D accept bits");
            f->accept_bits = (const uint32_t *)t_ctx.dbuf[6];
        }
    }
    *use = f->accept_bits != nullptr || f->threshold > 0.f || f->rerank_floor > 0.f;
    return JV_OK;
}

int jv_graph_search_batch_device_ex(jv_graph g, jv_dataset approx, jv_dataset reranker, int metric, const float *queries_device, int nq, int topK,
                                    int rerankK, const jv_search_options *opts_device_bits, int32_t *nodes_out_device, float *scores_out_device,
                                    jv_search_stats *stats)
{
    ON_DEVICE_OF(g);
    if (!g || nq <= 0) return fail(JV_ERR_INVALID, "graph_search: bad arguments");
    int rc;
    if ((rc = t_ctx.init())) return rc;
    SearchFilter f;
    bool use;
    if ((rc = make_filter(opts_device_bits, g, nq, true, &f, &use))) return rc;
    return search_device(g, approx, reranker, metric, queries_device, nq, topK, rerankK, use ? &f : nullptr, nodes_out_device, scores_out_device, stats);
}

int jv_graph_search_batch_device(jv_graph g, jv_dataset approx, jv_dataset reranker, int metric, const float *queries_device, int nq, int topK,
                                 int rerankK, int32_t *nodes_out_device, float *scores_out_device, jv_search_stats *stats)
{
    return jv_graph_search_batch_device_ex(g, approx, reranker, metric, queries_device, nq, topK, rerankK, nullptr, nodes_out_device, scores_out_device, stats);
}

int jv_graph_search_batch_ex(jv_graph g, jv_dataset approx, jv_dataset reranker, int metric, const float *queries, int nq, int topK, int rerankK,
                             const jv_search_options *opts, int32_t *nodes_out, float *scores_out, jv_search_stats *stats)
{
    ON_DEVICE_OF(g);
    if (!g || !approx || !queries || !nodes_out || !scores_out || nq <= 0 || topK < 1) return fail(JV_ERR_INVALID, "graph_search: bad arguments");
    int rc;
    const size_t qb = (size_t)nq * approx->d.dim * 4, ob = (size_t)nq * topK * 4;
    if ((rc = t_ctx.init()) || (rc = t_ctx.ensure(0, qb)) || (rc = t_ctx.ensure(1, ob)) || (rc = t_ctx.ensure(2, ob))) return rc;
    cudaStream_t s = t_ctx.stream;
    SearchFilter f;
    bool use;
    if ((rc = make_filter(opts, g, nq, false, &f, &use))) return rc;
    // Large batches: the queries travel in chunks on a second stream, each followed by a 4-byte watermark ("queries [0, w) have
    // arrived"), and the search kernel — launched at once — takes query i only when the watermark has passed it. The H2D copy
    // (30 MB at c2) hides behind the first wave of queries instead of preceding the kernel. JV_SEARCH_OVERLAP=0 disables.
    const char *ov = getenv("JV_SEARCH_OVERLAP");
    const bool overlap = qb >= ((size_t)1 << 20) && nq >= 64 && !(ov && ov[0] == '0');
    if (overlap) {
        if ((rc = t_ctx.init_copy()) || (rc = t_ctx.ensure(7, 256))) return rc;
        int *arrived = (int *)t_ctx.dbuf[7];
        CK(cudaMemsetAsync(arrived, 0, sizeof(int), s), "memset watermark");
        CK(cudaEventRecord(t_ctx.ev_copy, s), "event");
        cudaStream_t s2 = t_ctx.copy_stream;
        CK(cudaStreamSynchronize(s2), "copy stream");  // the pinned watermark values of the previous call are free again
        CK(cudaStreamWaitEvent(s2, t_ctx.ev_copy, 0), "wait");
        const int chunks = ThreadCtx::MARKS;
        const size_t row = (size_t)approx->d.dim * 4;
        for (int c = 0; c < chunks; c++) {
            // first chunk small (one kernel wave starts as early as possible), the rest equal. Boundaries are multiples of 32 queries:
            // 32 rows of 4 * dim bytes end on a 128-byte line, so no cache line holds queries of two chunks (a kernel that has read
            // the last query of a chunk can never hold a stale L1 copy of the first bytes of the next one)
            auto bound = [&](int c_) -> long long {
                if (c_ <= 0) return 0;
                if (c_ >= chunks) return nq;
                const long long rest = nq > 2048 ? nq - 2048 : 0;
                const long long b = 2048 + rest * (c_ - 1) / (chunks - 1);
                return std::min<long long>(nq, b & ~31ll);
            };
            const long long lo = bound(c), hi = bound(c + 1);
            if (hi <= lo) continue;
            CK(cudaMemcpyAsync((char *)t_ctx.dbuf[0] + (size_t)lo * row, (const char *)queries + (size_t)lo * row, (size_t)(hi - lo) * row, cudaMemcpyHostToDevice, s2), "H2D queries");
            t_ctx.marks_pinned[c] = (int)hi;
            CK(cudaMemcpyAsync(arrived, &t_ctx.marks_pinned[c], sizeof(int), cudaMemcpyHostToDevice, s2), "H2D watermark");
        }
        f.arrived = arrived;
        rc = search_device(g, approx, reranker, metric, (const float *)t_ctx.dbuf[0], nq, topK, rerankK, &f, (int32_t *)t_ctx.dbuf[1], (float *)t_ctx.dbuf[2], stats);
    } else {
        CK(cudaMemcpyAsync(t_ctx.dbuf[0], queries, qb, cudaMemcpyHostToDevice, s), "H2D queries");
        rc = search_device(g, approx, reranker, metric, (const float *)t_ctx.dbuf[0], nq, topK, rerankK, use ? &f : nullptr, (int32_t *)t_ctx.dbuf[1], (float *)t_ctx.dbuf[2], stats);
    }
    if (rc) return rc;
    CK(cudaMemcpyAsync(nodes_out, t_ctx.dbuf[1], ob, cudaMemcpyDeviceToHost, s), "D2H nodes");
    CK(cudaMemcpyAsync(scores_out, t_ctx.dbuf[2], ob, cudaMemcpyDeviceToHost, s), "D2H scores");
    CK(cudaStreamSynchronize(s), "sync");
    return JV_OK;
}

int jv_graph_search_batch(jv_graph g, jv_dataset approx, jv_dataset reranker, int metric, const float *queries, int nq, int topK, int rerankK,
                          int32_t *nodes_out, float *scores_out, jv_search_stats *stats)
{
    return jv_graph_search_batch_ex(g, approx, reranker, metric, queries, nq, topK, rerankK, nullptr, nodes_out, scores_out, stats);
}

static int build_params_check(const jv_build_params *params, BuildParams *bp)
{
    if (params->degree < 1 || params->degree > 64 || params->beam_width < 1 || params->beam_width > 256 || params->overflow < 1.0f || params->alpha < 1.0f)
        return fail(JV_ERR_INVALID, "graph_build: need 1 <= degree <= 64, 1 <= beam <= 256, overflow >= 1, alpha >= 1");
    bp->degree = params->degree; bp->beam = params->beam_width; bp->overflow = params->overflow; bp->alpha = params->alpha;
    bp->max_batch = params->max_batch; bp->window = params->concurrent_window;
    return JV_OK;
}

// HNSW-style levels (GraphIndexBuilder.java:562-575): level(node) = floor(-ln(U) / ln(M)); returns the members of every level >= 1
// (ascending ids) and the entry node (the first node of the top level)
static void assign_levels(int n, int degree, uint64_t seed, std::vector<std::vector<int32_t>> &members, int *entry)
{
    uint64_t st = seed ? seed : 0x9E3779B97F4A7C15ull;
    auto next_u = [&st]() {
        st ^= st << 13; st ^= st >> 7; st ^= st << 17;
        return ((st >> 11) + 1) * (1.0 / 9007199254740993.0);
    };
    const double ml = degree == 1 ? 1.0 : 1.0 / log((double)degree);
    std::vector<int> level(n);
    int maxl = 0;
    for (int i = 0; i < n; i++) {
        level[i] = (int)(-log(next_u()) * ml);
        maxl = std::max(maxl, level[i]);
    }
    *entry = 0;
    for (int i = 0; i < n; i++)
        if (level[i] == maxl) { *entry = i; break; }
    members.assign(maxl, {});
    for (int i = 0; i < n; i++)
        for (int l = 1; l <= level[i]; l++) members[l - 1].push_back(i);
}

// every upper level is a Vamana graph over its members, built by the same device builder on the members' rows (one gather kernel)
static int build_upper_levels(jv_graph g, jv_dataset f32, int metric, const BuildParams &bp, uint64_t seed, cudaStream_t s)
{
    const int n = (int)f32->d.n, degree = bp.degree;
    std::vector<std::vector<int32_t>> members;
    int entry = 0;
    assign_levels(n, degree, seed, members, &entry);
    g->g.entry_node = entry;
    int rc;
    for (size_t l = 0; l < members.size(); l++) {
        const std::vector<int32_t> &ids = members[l];
        const int cnt = (int)ids.size();
        std::vector<int32_t> ladj((size_t)cnt * degree, -1);
        if (cnt > 1) {
            jv_dataset_s sub;
            sub.device = f32->device;
            memset(&sub.d, 0, sizeof(DataDesc));
            sub.d.kind = KIND_F32; sub.d.dim = f32->d.dim; sub.d.stride = f32->d.stride; sub.d.n = cnt;
            float *drows = nullptr;
            int32_t *dadj = nullptr, *dids = nullptr;
            if ((rc = sub.alloc((void **)&drows, (size_t)cnt * sub.d.stride * 4)) || (rc = sub.alloc((void **)&dadj, (size_t)cnt * degree * 4)) ||
                (rc = sub.alloc((void **)&dids, (size_t)cnt * 4)))
                return rc;
            cudaError_t e = cudaMemcpyAsync(dids, ids.data(), (size_t)cnt * 4, cudaMemcpyHostToDevice, s);
            if (e == cudaSuccess) e = launch_gather_rows(f32->d, dids, cnt, drows, s);
            sub.d.rows = drows;
            BuildStats bs2;
            if (e == cudaSuccess) e = build_graph_flat(sub.d, metric, bp, dadj, g_sm_count, &bs2, s);
            if (e == cudaSuccess) e = cudaMemcpyAsync(ladj.data(), dadj, ladj.size() * 4, cudaMemcpyDeviceToHost, s);
            if (e == cudaSuccess) e = cudaStreamSynchronize(s);
            if (e != cudaSuccess) return cuda_fail(e, "build upper level");
            for (auto &x : ladj)
                if (x >= 0) x = ids[x];
        }
        g->level_ids.push_back(ids);
        g->level_adj.push_back(ladj);
    }
    return graph_rebuild_upper(g);
}

int jv_graph_build(jv_dataset f32, int metric, const jv_build_params *params, jv_graph *out, double *device_ms)
{
    ON_DEVICE_OF(f32);
    if (!f32 || !params || !out || f32->d.kind != KIND_F32) return fail(JV_ERR_INVALID, "graph_build: needs an fp32 data set");
    int rc = check_metric(f32->d, metric);
    if (rc) return rc;
    if ((rc = t_ctx.init())) return rc;
    cudaStream_t s = t_ctx.stream;
    BuildParams bp;
    if ((rc = build_params_check(params, &bp))) return rc;
    const int n = (int)f32->d.n, degree = params->degree;
    jv_graph g = new jv_graph_s();
    g->device = f32->device;
    memset(&g->g, 0, sizeof(GraphDesc));
    cudaError_t e = cudaMalloc((void **)&g->adj0, (size_t)n * degree * 4);
    if (e != cudaSuccess) { delete g; return cuda_fail(e, "cudaMalloc(adjacency)"); }
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    cudaEventCreate(&e0);
    cudaEventCreate(&e1);
    cudaEventRecord(e0, s);
    BuildStats bs;
    e = build_graph_flat(f32->d, metric, bp, g->adj0, g_sm_count, &bs, s);
    t_build_stats = bs;
    g->g.n = n; g->g.degree = degree; g->g.levels = 1; g->g.entry_node = 0; g->g.entry_level = 0; g->g.adj0 = g->adj0;
    rc = e == cudaSuccess ? JV_OK : cuda_fail(e, "build_graph_flat");
    if (!rc && params->add_hierarchy && n > 1) rc = build_upper_levels(g, f32, metric, bp, params->seed, s);
    cudaEventRecord(e1, s);  // the upper levels are part of the build and of its time
    cudaStreamSynchronize(s);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (rc) { delete g; return rc; }
    if (device_ms) *device_ms = ms;
    *out = g;
    return JV_OK;
}

// ---- the same build advanced batch by batch, for a build SHARDED over several GPUs (BASELINE config 5) ----------------------
// Every rank holds a replica of the rows and of the adjacency. Per batch: each rank searches + prunes ITS slice of the batch
// (jv_builder_insert_slice -> rows in a caller buffer), the slices are all-gathered by the caller (NCCL; jvector_b200/parallel.py),
// every rank applies the whole batch deterministically (jv_builder_apply_new), then the rows that passed overflow * M are
// re-pruned slice-wise and exchanged the same way. The device pointers are the caller's (e.g. torch tensors = the NCCL buffers).
struct jv_builder_s {
    int device = 0;
    jv_dataset f32 = nullptr;
    int metric = 0;
    jv_build_params params;
    BuildParams bp;
    GraphBuilder *B = nullptr;
    cudaStream_t stream = nullptr;
    cudaEvent_t e0 = nullptr;
};

int jv_builder_create(jv_dataset f32, int metric, const jv_build_params *params, void *cuda_stream, jv_builder *out)
{
    ON_DEVICE_OF(f32);
    if (!params || !out || f32->d.kind != KIND_F32) return fail(JV_ERR_INVALID, "builder_create: needs an fp32 data set");
    int rc = check_metric(f32->d, metric);
    if (rc) return rc;
    jv_builder b = new jv_builder_s();
    b->device = f32->device; b->f32 = f32; b->metric = metric; b->params = *params; b->stream = (cudaStream_t)cuda_stream;
    if ((rc = build_params_check(params, &b->bp))) { delete b; return rc; }
    cudaEventCreate(&b->e0);
    cudaEventRecord(b->e0, b->stream);
    cudaError_t e = builder_create(f32->d, metric, b->bp, g_sm_count, &b->B, b->stream);
    if (e != cudaSuccess) { cudaEventDestroy(b->e0); delete b; return cuda_fail(e, "builder_create"); }
    *out = b;
    return JV_OK;
}

int jv_builder_info(jv_builder b, int *degree, int *row_cap, int *max_batch)
{
    if (!b) return fail(JV_ERR_INVALID, "builder_info: null");
    if (degree) *degree = builder_degree(b->B);
    if (row_cap) *row_cap = builder_row_cap(b->B);
    if (max_batch) *max_batch = builder_max_batch(b->B);
    return JV_OK;
}

int jv_builder_next_batch(jv_builder b, int32_t *first, int32_t *count)
{
    if (!b || !first || !count) return fail(JV_ERR_INVALID, "builder_next_batch: null");
    int f = 0, c = 0;
    const bool more = builder_next_batch(b->B, &f, &c);
    *first = f;
    *count = more ? c : 0;
    return JV_OK;
}

int jv_builder_insert_slice(jv_builder b, int32_t first, int32_t count, int32_t lo, int32_t hi, int32_t *rows_out_device, int32_t *deg_out_device)
{
    ON_DEVICE_OF(b);
    if (lo < 0 || hi > count || !rows_out_device || !deg_out_device) return fail(JV_ERR_INVALID, "builder_insert_slice: bad arguments");
    CK(builder_insert_slice(b->B, first, count, lo, hi, rows_out_device, deg_out_device, b->stream), "builder_insert_slice");
    return JV_OK;
}

int jv_builder_apply_new(jv_builder b, int32_t first, int32_t count, const int32_t *rows_device, const int32_t *deg_device, int32_t *overflow_rows)
{
    ON_DEVICE_OF(b);
    if (!rows_device || !deg_device) return fail(JV_ERR_INVALID, "builder_apply_new: bad arguments");
    CK(builder_apply_new(b->B, first, count, rows_device, deg_device, b->stream), "builder_apply_new");
    if (overflow_rows) {
        int c = 0;
        CK(builder_list_count(b->B, &c, b->stream), "builder_list_count");
        *overflow_rows = c;
    }
    return JV_OK;
}

int jv_builder_reprune_slice(jv_builder b, int32_t lo, int32_t hi, int32_t *rows_out_device, int32_t *deg_out_device)
{
    ON_DEVICE_OF(b);
    if (!rows_out_device || !deg_out_device || lo < 0) return fail(JV_ERR_INVALID, "builder_reprune_slice: bad arguments");
    CK(builder_reprune_slice(b->B, lo, hi, rows_out_device, deg_out_device, b->stream), "builder_reprune_slice");
    return JV_OK;
}

int jv_builder_apply_repruned(jv_builder b, int32_t count, const int32_t *rows_device, const int32_t *deg_device)
{
    ON_DEVICE_OF(b);
    CK(builder_apply_repruned(b->B, count, rows_device, deg_device, b->stream), "builder_apply_repruned");
    return JV_OK;
}

int jv_builder_collect_over_degree(jv_builder b, int32_t *rows)
{
    ON_DEVICE_OF(b);
    CK(builder_collect_over_degree(b->B, b->stream), "builder_collect_over_degree");
    int c = 0;
    CK(builder_list_count(b->B, &c, b->stream), "builder_list_count");
    if (rows) *rows = c;
    return JV_OK;
}

// compacts the level-0 adjacency into a graph; the upper levels (3 % of the nodes at M = 32) are built by every replica itself
int jv_builder_finish(jv_builder b, jv_graph *out, double *device_ms)
{
    ON_DEVICE_OF(b);
    if (!out) return fail(JV_ERR_INVALID, "builder_finish: null");
    int rc;
    if ((rc = t_ctx.init())) return rc;
    const int n = (int)b->f32->d.n, degree = b->bp.degree;
    jv_graph g = new jv_graph_s();
    g->device = b->device;
    memset(&g->g, 0, sizeof(GraphDesc));
    cudaError_t e = cudaMalloc((void **)&g->adj0, (size_t)n * degree * 4);
    if (e != cudaSuccess) { delete g; return cuda_fail(e, "cudaMalloc(adjacency)"); }
    BuildStats bs;
    e = builder_finish(b->B, g->adj0, &bs, b->stream);
    t_build_stats = bs;
    if (e != cudaSuccess) { delete g; return cuda_fail(e, "builder_finish"); }
    g->g.n = n; g->g.degree = degree; g->g.levels = 1; g->g.entry_node = 0; g->g.entry_level = 0; g->g.adj0 = g->adj0;
    if (b->params.add_hierarchy && n > 1 && (rc = build_upper_levels(g, b->f32, b->metric, b->bp, b->params.seed, b->stream))) { delete g; return rc; }
    cudaEvent_t e1;
    cudaEventCreate(&e1);
    cudaEventRecord(e1, b->stream);
    cudaStreamSynchronize(b->stream);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, b->e0, e1);
    cudaEventDestroy(e1);
    if (device_ms) *device_ms = ms;
    *out = g;
    return JV_OK;
}

int jv_builder_free(jv_builder b)
{
    if (!b) return JV_OK;
    cudaSetDevice(b->device);
    if (b->stream) cudaStreamSynchronize(b->stream);
    else cudaDeviceSynchronize();
    builder_destroy(b->B);
    if (b->e0) cudaEventDestroy(b->e0);
    delete b;
    return JV_OK;
}

int jv_graph_build_stats(int64_t *scored_vectors, int64_t *batches, int64_t *dropped_backlinks)
{
    if (scored_vectors) *scored_vectors = t_build_stats.searched;
    if (batches) *batches = t_build_stats.batches;
    if (dropped_backlinks) *dropped_backlinks = t_build_stats.dropped_backlinks;
    return JV_OK;
}

// ------------------------------------------------------------------------------------------------ query batches (host-driven seam)
// north_star's literal form of the path: the host expands the frontier and sends each hop's candidate set as one launch. What
// makes that seam fast is what persists between calls: the prepared queries (LUTs / bit packs / shifted copies) stay in HBM for
// the life of the batch, and ids / offsets / scores travel through pinned, device-mapped staging that belongs to the batch.
struct jv_query_batch_s {
    int device = 0;
    jv_dataset ds = nullptr;
    int metric = 0, nq = 0;
    float *blobs = nullptr;        // [nq][blob_floats]
    size_t blob_floats = 0;
    // pinned + mapped staging (grown on demand)
    int32_t *h_ids = nullptr, *h_off = nullptr;
    float *h_scores = nullptr;
    size_t cap_ids = 0, cap_off = 0;
    int32_t *d_ids = nullptr, *d_off = nullptr;
    float *d_scores = nullptr;
    size_t dcap = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    // single-hop path: mapped pinned ids / scores / completion flag the kernel reads and writes directly, a device-side CTA counter
    int32_t *hop_ids = nullptr, *hop_ids_dev = nullptr;
    float *hop_scores = nullptr, *hop_scores_dev = nullptr;
    int *hop_flag = nullptr, *hop_flag_dev = nullptr, *hop_done = nullptr;
    size_t hop_cap = 0;
    int hop_seq = 0;
};

static void query_batch_release(jv_query_batch_s *b)
{
    if (!b) return;
    cudaSetDevice(b->device);
    if (b->stream) cudaStreamSynchronize(b->stream);
    cudaFree(b->blobs); cudaFree(b->d_ids); cudaFree(b->d_off); cudaFree(b->d_scores);
    cudaFreeHost(b->h_ids); cudaFreeHost(b->h_off); cudaFreeHost(b->h_scores);
    cudaFreeHost(b->hop_ids); cudaFreeHost(b->hop_scores); cudaFreeHost(b->hop_flag); cudaFree(b->hop_done);
    if (b->ev0) cudaEventDestroy(b->ev0);
    if (b->ev1) cudaEventDestroy(b->ev1);
    if (b->stream) cudaStreamDestroy(b->stream);
    delete b;
}

int jv_query_batch_begin(jv_dataset ds, int metric, const float *queries, int nq, jv_query_batch *out)
{
    ON_DEVICE_OF(ds);
    if (!queries || !out || nq <= 0 || nq > 65535) return fail(JV_ERR_INVALID, "query_batch_begin: 1 <= nq <= 65535");
    int rc = check_metric(ds->d, metric);
    if (rc) return rc;
    if ((rc = t_ctx.init()) || (rc = t_ctx.ensure(0, (size_t)nq * ds->d.dim * 4))) return rc;
    jv_query_batch_s *b = new jv_query_batch_s();
    b->device = ds->device; b->ds = ds; b->metric = metric; b->nq = nq; b->blob_floats = (size_t)blob_floats(ds->d);
    cudaError_t e = cudaMalloc((void **)&b->blobs, (size_t)nq * b->blob_floats * 4);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&b->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&b->ev1);
    if (e == cudaSuccess) e = cudaMemcpyAsync(t_ctx.dbuf[0], queries, (size_t)nq * ds->d.dim * 4, cudaMemcpyHostToDevice, t_ctx.stream);
    if (e == cudaSuccess) e = launch_prepare(ds->d, metric, (const float *)t_ctx.dbuf[0], nq, b->blobs, t_ctx.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(t_ctx.stream);
    if (e != cudaSuccess) { query_batch_release(b); return cuda_fail(e, "query_batch_begin"); }
    *out = b;
    return JV_OK;
}

static int query_batch_staging(jv_query_batch_s *b, size_t total, size_t noff)
{
    if (total > b->cap_ids) {
        cudaFreeHost(b->h_ids); cudaFreeHost(b->h_scores);
        b->h_ids = nullptr; b->h_scores = nullptr; b->cap_ids = 0;
        const size_t want = total + total / 2 + 256;
        CK(cudaHostAlloc((void **)&b->h_ids, want * 4, cudaHostAllocMapped), "cudaHostAlloc(ids)");
        CK(cudaHostAlloc((void **)&b->h_scores, want * 4, cudaHostAllocMapped), "cudaHostAlloc(scores)");
        b->cap_ids = want;
    }
    if (noff > b->cap_off) {
        cudaFreeHost(b->h_off);
        b->h_off = nullptr; b->cap_off = 0;
        CK(cudaHostAlloc((void **)&b->h_off, (noff + 64) * 4, cudaHostAllocMapped), "cudaHostAlloc(offsets)");
        b->cap_off = noff + 64;
    }
    if (total > b->dcap) {
        cudaFree(b->d_ids); cudaFree(b->d_scores); cudaFree(b->d_off);
        b->d_ids = nullptr; b->d_scores = nullptr; b->d_off = nullptr; b->dcap = 0;
        const size_t want = total + total / 2 + 256;
        CK(cudaMalloc((void **)&b->d_ids, want * 4), "cudaMalloc(ids)");
        CK(cudaMalloc((void **)&b->d_scores, want * 4), "cudaMalloc(scores)");
        CK(cudaMalloc((void **)&b->d_off, ((size_t)b->nq + 64) * 4), "cudaMalloc(offsets)");
        b->dcap = want;
    }
    return JV_OK;
}

// one step of all the batch's searches: query i scores ids[offsets[i] .. offsets[i+1]); only ids + offsets go up, scores come down
int jv_query_batch_score(jv_query_batch b, const int32_t *ids, const int32_t *offsets, float *scores_out, double *device_ms)
{
    ON_DEVICE_OF(b);
    if (!ids || !offsets || !scores_out) return fail(JV_ERR_INVALID, "query_batch_score: null argument");
    const int nq = b->nq;
    const int total = offsets[nq];
    int maxc = 0;
    for (int i = 0; i < nq; i++) {
        if (offsets[i + 1] < offsets[i]) return fail(JV_ERR_INVALID, "query_batch_score: offsets not monotone");
        maxc = std::max(maxc, offsets[i + 1] - offsets[i]);
    }
    if (device_ms) *device_ms = 0.0;
    if (total <= 0) return JV_OK;
    int rc = query_batch_staging(b, (size_t)total, (size_t)nq + 1);
    if (rc) return rc;
    // caller buffers that are already pinned (jv_host_register / cudaHostAlloc) are copied from / to directly; pageable ones go
    // through the batch's own pinned staging so that the copies stay asynchronous and full speed
    auto pinned = [](const void *p) {
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
        return a.type == cudaMemoryTypeHost;
    };
    const bool ids_pinned = pinned(ids), out_pinned = pinned(scores_out);
    if (!ids_pinned) memcpy(b->h_ids, ids, (size_t)total * 4);
    memcpy(b->h_off, offsets, ((size_t)nq + 1) * 4);
    cudaStream_t s = b->stream;
    CK(cudaMemcpyAsync(b->d_ids, ids_pinned ? ids : b->h_ids, (size_t)total * 4, cudaMemcpyHostToDevice, s), "H2D ids");
    CK(cudaMemcpyAsync(b->d_off, b->h_off, ((size_t)nq + 1) * 4, cudaMemcpyHostToDevice, s), "H2D offsets");
    CK(cudaEventRecord(b->ev0, s), "event");
    CK(launch_score_ragged(b->ds->d, b->metric, b->blobs, nq, b->d_ids, b->d_off, 0, maxc, b->d_scores, s), "score_ragged");
    CK(cudaEventRecord(b->ev1, s), "event");
    CK(cudaMemcpyAsync(out_pinned ? scores_out : b->h_scores, b->d_scores, (size_t)total * 4, cudaMemcpyDeviceToHost, s), "D2H scores");
    CK(cudaStreamSynchronize(s), "sync");
    if (!out_pinned) memcpy(scores_out, b->h_scores, (size_t)total * 4);
    if (device_ms) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, b->ev0, b->ev1);
        *device_ms = ms;
    }
    return JV_OK;
}

// one hop of ONE search of the batch. Latency path: the kernel reads the ids from, and writes the scores and a completion
// sequence number to, mapped pinned memory; the host spins on that word instead of synchronising the stream (a blocking
// cudaStreamSynchronize costs more than the launch and the kernel together), and polls the stream only to notice a failed launch.
int jv_query_batch_score_one(jv_query_batch b, int query_index, const int32_t *ids, int n, float *scores_out)
{
    ON_DEVICE_OF(b);
    if (query_index < 0 || query_index >= b->nq || n < 0 || (n > 0 && (!ids || !scores_out))) return fail(JV_ERR_INVALID, "query_batch_score_one: bad arguments");
    if (n == 0) return JV_OK;
    if ((size_t)n > b->hop_cap) {
        CK(cudaStreamSynchronize(b->stream), "sync");
        cudaFreeHost(b->hop_ids); cudaFreeHost(b->hop_scores);
        b->hop_ids = nullptr; b->hop_scores = nullptr; b->hop_cap = 0;
        const size_t want = (size_t)n + 1024;
        CK(cudaHostAlloc((void **)&b->hop_ids, want * 4, cudaHostAllocMapped), "cudaHostAlloc(hop ids)");
        CK(cudaHostAlloc((void **)&b->hop_scores, want * 4, cudaHostAllocMapped), "cudaHostAlloc(hop scores)");
        CK(cudaHostGetDevicePointer((void **)&b->hop_ids_dev, b->hop_ids, 0), "cudaHostGetDevicePointer");
        CK(cudaHostGetDevicePointer((void **)&b->hop_scores_dev, b->hop_scores, 0), "cudaHostGetDevicePointer");
        if (!b->hop_flag) {
            CK(cudaHostAlloc((void **)&b->hop_flag, 64, cudaHostAllocMapped), "cudaHostAlloc(hop flag)");
            CK(cudaHostGetDevicePointer((void **)&b->hop_flag_dev, b->hop_flag, 0), "cudaHostGetDevicePointer");
            *b->hop_flag = 0;
            CK(cudaMalloc((void **)&b->hop_done, 64), "cudaMalloc(hop counter)");
            CK(cudaMemset(b->hop_done, 0, 64), "memset");
        }
        b->hop_cap = want;
    }
    const float *blob = b->blobs + (size_t)query_index * b->blob_floats;
    if (n <= HOP_MAX_IDS) {
        // ids in the kernel parameters, every score word pre-set to a pattern no score can have and polled until it is overwritten
        volatile uint32_t *sc = reinterpret_cast<volatile uint32_t *>(b->hop_scores);
        for (int i = 0; i < n; i++) sc[i] = 0xffffffffu;
        __atomic_thread_fence(__ATOMIC_SEQ_CST);
        CK(launch_score_hop(b->ds->d, b->metric, blob, ids, n, b->hop_scores_dev, b->stream), "score_hop");
        unsigned spins = 0;
        for (int i = 0; i < n; i++) {
            while (sc[i] == 0xffffffffu) {
                if ((++spins & 0x3fffu) == 0) {
                    const cudaError_t e = cudaStreamQuery(b->stream);
                    if (e == cudaSuccess) {
                        if (sc[i] != 0xffffffffu) break;
                        return fail(JV_ERR_CUDA, "query_batch_score_one: the kernel finished without writing its scores");
                    }
                    if (e != cudaErrorNotReady) return cuda_fail(e, "query_batch_score_one");
                }
#if defined(__x86_64__)
                __builtin_ia32_pause();
#endif
            }
        }
        __atomic_thread_fence(__ATOMIC_ACQUIRE);
        memcpy(scores_out, b->hop_scores, (size_t)n * 4);
        return JV_OK;
    }
    memcpy(b->hop_ids, ids, (size_t)n * 4);
    const int seq = ++b->hop_seq == 0 ? ++b->hop_seq : b->hop_seq;
    // one lane group per id and 4 ids per CTA: the hop's rows are fetched in one wave instead of one CTA walking them in turn
    CK(launch_score_ragged(b->ds->d, b->metric, blob, 1, b->hop_ids_dev, nullptr, n, n, b->hop_scores_dev, b->stream, 4, b->hop_done, b->hop_flag_dev, seq),
       "score_ragged");
    volatile int *flag = b->hop_flag;
    for (unsigned spins = 1; *flag != seq; spins++) {
        if ((spins & 0x3fffu) == 0) {
            const cudaError_t e = cudaStreamQuery(b->stream);
            if (e == cudaSuccess) {
                if (*flag == seq) break;
                return fail(JV_ERR_CUDA, "query_batch_score_one: the kernel finished without its completion signal");
            }
            if (e != cudaErrorNotReady) return cuda_fail(e, "query_batch_score_one");
        }
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
    }
    __atomic_thread_fence(__ATOMIC_ACQUIRE);
    memcpy(scores_out, b->hop_scores, (size_t)n * 4);
    return JV_OK;
}

int jv_query_batch_end(jv_query_batch b)
{
    query_batch_release(b);
    return JV_OK;
}

// ------------------------------------------------------------------------------------------------ several GPUs, one process
// The reference host is ONE JVM whose parallelism is threads (base:vector/VectorizationProvider.java:79-177,
// base:graph/GraphIndexBuilder.java:440-444), so the sharding of SURVEY §8e has to be reachable from one process: the base
// range-sharded by contiguous node id over the bound devices, every shard scoring all queries on its own stream, the per-shard
// top-k keys (global ids) copied to the first device over NVLink (peer copies) and merged there.
int jv_multi_free(jv_multi m)
{
    if (!m) return JV_OK;
    for (jv_dataset ds : m->shards) jv_dataset_free(ds);
    for (size_t i = 0; i < m->ctx.size(); i++) {
        t_active = m->devices[i];
        cudaSetDevice(m->devices[i]);
        delete m->ctx[i];
    }
    delete m;
    return JV_OK;
}

int jv_multi_register_bq(const uint64_t *words, int64_t n, int dim, jv_multi *out)
{
    if (!words || !out || n <= 0 || dim <= 0 || n > 0x7fffffffLL) return fail(JV_ERR_INVALID, "multi_register_bq: bad arguments");
    jv_multi m = new jv_multi_s();
    m->kind = KIND_BQ; m->dim = dim; m->n = n;
    const int W = (dim + 63) / 64;
    int rc = multi_register(m, [&](int, int64_t lo, int64_t cnt, jv_dataset *ds) { return jv_dataset_register_bq(words + (size_t)lo * W, cnt, dim, ds); });
    if (rc) { jv_multi_free(m); return rc; }
    *out = m;
    return JV_OK;
}

int jv_multi_register_f32(const float *rows, int64_t n, int dim, jv_multi *out)
{
    if (!rows || !out || n <= 0 || dim <= 0 || n > 0x7fffffffLL) return fail(JV_ERR_INVALID, "multi_register_f32: bad arguments");
    jv_multi m = new jv_multi_s();
    m->kind = KIND_F32; m->dim = dim; m->n = n;
    int rc = multi_register(m, [&](int, int64_t lo, int64_t cnt, jv_dataset *ds) { return jv_dataset_register_f32(rows + (size_t)lo * dim, cnt, dim, ds); });
    if (rc) { jv_multi_free(m); return rc; }
    *out = m;
    return JV_OK;
}

int jv_multi_shard_count(jv_multi m) { return m ? (int)m->shards.size() : 0; }

int jv_multi_shard_info(jv_multi m, int shard, int *device, int64_t *first_row, int64_t *rows)
{
    if (!m || shard < 0 || shard >= (int)m->shards.size()) return fail(JV_ERR_INVALID, "multi_shard_info: bad shard");
    if (device) *device = m->devices[shard];
    if (first_row) *first_row = m->lo[shard];
    if (rows) *rows = m->lo[shard + 1] - m->lo[shard];
    return JV_OK;
}

int jv_multi_topk_bruteforce(jv_multi m, int metric, const float *queries, int nq, int k, int64_t *keys_out)
{
    if (!m || !queries || !keys_out || nq <= 0 || k <= 0 || k > 2048) return fail(JV_ERR_INVALID, "multi_topk_bruteforce: bad arguments");
    const int parts = (int)m->shards.size();
    if ((long long)parts * k > 16384) return fail(JV_ERR_INVALID, "multi_topk_bruteforce: shards * k <= 16384");
    const size_t qb = (size_t)nq * m->dim * 4, kb = (size_t)nq * k * 8;
    std::vector<int> rcs(parts, JV_OK);
    std::vector<std::string> errs(parts);
    // the gathered keys live on the first shard's device: [parts][nq][k]
    ThreadCtx *c0 = m->ctx[0];
    {
        t_active = m->devices[0];
        t_ctx_override = c0;
        cudaSetDevice(m->devices[0]);
        int rc = c0->init();
        if (!rc) rc = c0->ensure(6, kb * parts + kb);
        t_ctx_override = nullptr;
        if (rc) return rc;
    }
    long long *gathered = (long long *)c0->dbuf[6];
    auto work = [&](int i) {
        t_active = m->devices[i];
        t_ctx_override = m->ctx[i];
        ThreadCtx &c = *m->ctx[i];
        int rc = JV_OK;
        do {
            if (cudaSetDevice(m->devices[i]) != cudaSuccess) { rc = fail(JV_ERR_CUDA, "cudaSetDevice"); break; }
            if ((rc = c.init()) || (rc = c.ensure(0, qb)) || (rc = c.ensure(5, kb))) break;
            if (cudaMemcpyAsync(c.dbuf[0], queries, qb, cudaMemcpyHostToDevice, c.stream) != cudaSuccess) { rc = fail(JV_ERR_CUDA, "H2D queries"); break; }
            if ((rc = topk_device(m->shards[i], metric, (const float *)c.dbuf[0], nq, k, m->lo[i], (long long *)c.dbuf[5]))) break;
            // shard keys -> the first device (NVLink peer copy; a plain device copy for shard 0)
            cudaError_t e = cudaMemcpyPeerAsync(gathered + (size_t)i * nq * k, m->devices[0], c.dbuf[5], m->devices[i], kb, c.stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(c.stream);
            if (e != cudaSuccess) rc = cuda_fail(e, "peer copy of shard keys");
        } while (0);
        rcs[i] = rc;
        if (rc) errs[i] = t_err;
        t_ctx_override = nullptr;
    };
    std::vector<std::thread> th;
    for (int i = 1; i < parts; i++) th.emplace_back(work, i);
    work(0);
    for (auto &t : th) t.join();
    for (int i = 0; i < parts; i++)
        if (rcs[i]) return fail(rcs[i], "shard " + std::to_string(i) + ": " + errs[i]);
    // merge on the first device: [parts][nq][k] -> per query the k best of parts * k
    t_active = m->devices[0];
    t_ctx_override = c0;
    int rc = JV_OK;
    do {
        if (cudaSetDevice(m->devices[0]) != cudaSuccess) { rc = fail(JV_ERR_CUDA, "cudaSetDevice"); break; }
        long long *merged = gathered + (size_t)parts * nq * k;
        cudaError_t e = parts == 1 ? cudaMemcpyAsync(merged, gathered, kb, cudaMemcpyDeviceToDevice, c0->stream)
                                   : launch_topk_merge_strided(gathered, nq, parts, k, merged, c0->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(keys_out, merged, kb, cudaMemcpyDeviceToHost, c0->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c0->stream);
        if (e != cudaSuccess) rc = cuda_fail(e, "merge");
    } while (0);
    t_ctx_override = nullptr;
    return rc;
}

// replicas: graph + data sets registered once per device (jv_gpu_set_device + the ordinary register calls); the query batch is
// split into contiguous slices, one per replica, searched concurrently (no data-path exchange: SURVEY §8e "shard queries")
int jv_multi_graph_search_batch(int replicas, const jv_graph *graphs, const jv_dataset *approx, const jv_dataset *rerankers, int metric,
                                const float *queries, int nq, int topK, int rerankK, const jv_search_options *opts, int32_t *nodes_out,
                                float *scores_out, jv_search_stats *stats)
{
    if (replicas <= 0 || !graphs || !approx || !queries || !nodes_out || !scores_out || nq <= 0) return fail(JV_ERR_INVALID, "multi_graph_search: bad arguments");
    if (opts && opts->accept_bits && opts->accept_stride_words == 0 && replicas > 1) { /* a shared bitset is simply reused by every slice */ }
    const int parts = std::min(replicas, nq);
    const int dim = approx[0]->d.dim;
    // worker threads come and go; their contexts (streams, visited-table scratch) must not: one persistent context per device,
    // calls of this entry point are serialised
    static ThreadCtx *worker_ctx[MAX_DEVICES] = {nullptr};
    static std::mutex worker_mu;
    std::lock_guard<std::mutex> lk(worker_mu);
    for (int i = 0; i < parts; i++) {
        if (!graphs[i] || !approx[i]) return fail(JV_ERR_INVALID, "multi_graph_search: null replica handle");
        if (!worker_ctx[graphs[i]->device]) worker_ctx[graphs[i]->device] = new ThreadCtx();
        for (int j = 0; j < i; j++)
            if (graphs[j]->device == graphs[i]->device) return fail(JV_ERR_INVALID, "multi_graph_search: two replicas on one device");
    }
    std::vector<int> rcs(parts, JV_OK);
    std::vector<std::string> errs(parts);
    std::vector<jv_search_stats> st(parts);
    std::vector<int64_t> lo;
    shard_ranges(nq, parts, lo);
    auto work = [&](int i) {
        const int q0 = (int)lo[i], cq = (int)(lo[i + 1] - lo[i]);
        jv_search_options o2;
        const jv_search_options *op = opts;
        if (opts && opts->accept_bits && opts->accept_stride_words) {
            o2 = *opts;
            o2.accept_bits = opts->accept_bits + (size_t)q0 * opts->accept_stride_words;
            op = &o2;
        }
        t_ctx_override = worker_ctx[graphs[i]->device];
        rcs[i] = jv_graph_search_batch_ex(graphs[i], approx[i], rerankers ? rerankers[i] : nullptr, metric, queries + (size_t)q0 * dim, cq, topK, rerankK, op,
                                          nodes_out + (size_t)q0 * topK, scores_out + (size_t)q0 * topK, &st[i]);
        if (rcs[i]) errs[i] = t_err;
        t_ctx_override = nullptr;
    };
    std::vector<std::thread> th;
    for (int i = 1; i < parts; i++) th.emplace_back(work, i);
    work(0);
    for (auto &t : th) t.join();
    for (int i = 0; i < parts; i++)
        if (rcs[i]) return fail(rcs[i], "replica " + std::to_string(i) + ": " + errs[i]);
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        for (int i = 0; i < parts; i++) {
            stats->visited += st[i].visited; stats->expanded += st[i].expanded; stats->expanded_base += st[i].expanded_base;
            stats->reranked += st[i].reranked; stats->retried += st[i].retried;
            stats->device_ms = std::max(stats->device_ms, st[i].device_ms);  // the replicas run concurrently: the step takes the slowest one
        }
    }
    return JV_OK;
}

// ------------------------------------------------------------------------------------------------ memory helpers
int jv_device_malloc(void **out, size_t bytes)
{
    NEED_INIT();
    if (!out) return fail(JV_ERR_INVALID, "device_malloc: null");
    CK(cudaMalloc(out, bytes ? bytes : 16), "cudaMalloc");
    return JV_OK;
}
int jv_device_free(void *p)
{
    NEED_INIT();
    CK(cudaFree(p), "cudaFree");
    return JV_OK;
}
int jv_memcpy_h2d(void *dst, const void *src, size_t bytes)
{
    NEED_INIT();
    CK(cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice), "cudaMemcpy H2D");
    return JV_OK;
}
int jv_memcpy_d2h(void *dst, const void *src, size_t bytes)
{
    NEED_INIT();
    CK(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost), "cudaMemcpy D2H");
    return JV_OK;
}
int jv_host_register(void *p, size_t bytes)
{
    NEED_INIT();
    CK(cudaHostRegister(p, bytes, cudaHostRegisterDefault), "cudaHostRegister");
    return JV_OK;
}
int jv_host_unregister(void *p)
{
    NEED_INIT();
    CK(cudaHostUnregister(p), "cudaHostUnregister");
    return JV_OK;
}
int jv_device_synchronize(void)
{
    NEED_INIT();
    CK(cudaDeviceSynchronize(), "cudaDeviceSynchronize");
    return JV_OK;
}

}  // extern "C"
