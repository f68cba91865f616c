/*
 * xm_api.cu -- the C ABI of libxenomapper_b200.so (include/xenomapper_b200.h):
 * context, device/pinned memory, the resident walk, the host-buffer walk with
 * pinned double-buffered staging, and the file-descriptor walk.
 *
 * There is no CPU classification path in this library.  If no CUDA device is
 * usable xm_create fails and every other entry point returns XM_ERR_CUDA.
 */
#include <cuda_runtime.h>
#include <errno.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <unistd.h>

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/xenomapper_b200.h"
#include "xm_common.h"
#include "xm_launch.h"
#include "xm_walk.h"
#include "xm_stream.h"
#include "xm_bam.h"
#include "xm_inflate.h"
#include "xm_bamchain.h"
#include "xm_deflate.h"
#include "xm_shard.h"
#include "xm_headers.h"
#include "xm_bgzf.h"
#include "xm_nccl.h"

using namespace xm;

static thread_local std::string g_create_error;

struct DeviceBackend {
    cudaStream_t st = nullptr;
    cudaStream_t up[2] = {nullptr, nullptr};      /* H2D lanes of the chunked walk, used alternately */
    int up_next = 0;
    int upload(void *d, const void *h, size_t n) { const int k = up_next; up_next ^= 1; return chk(cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, up[k])); }
    int upload_wait() { return chk(cudaStreamSynchronize(up[0])) || chk(cudaStreamSynchronize(up[1])); }
    int copy_dd(void *d, const void *s, size_t n) { return chk(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToDevice, st)) || chk(cudaStreamSynchronize(st)); }
    cudaEvent_t ev[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    std::string err;
    int chk(cudaError_t e)
    {
        if (e == cudaSuccess) return 0;
        err = cudaGetErrorString(e);
        return 1;
    }
    void *alloc(size_t n)
    {
        void *p = nullptr;
        if (chk(cudaMalloc(&p, n ? n : 16))) return nullptr;
        return p;
    }
    void release(void *p) { if (p) cudaFree(p); }
    int zero(void *p, size_t n) { return n ? chk(cudaMemsetAsync(p, 0, n, st)) : 0; }
    int write(void *d, const void *s, size_t n) { return chk(cudaMemcpyAsync(d, s, n, cudaMemcpyHostToDevice, st)) || chk(cudaStreamSynchronize(st)); }
    int read(void *d, const void *s, size_t n) { return chk(cudaMemcpyAsync(d, s, n, cudaMemcpyDeviceToHost, st)) || chk(cudaStreamSynchronize(st)); }
    unsigned long long *h_words = nullptr;        /* pinned landing place of read_words */
    int read_words(const void *const src[], int n, unsigned long long *dst)
    {
        if (!h_words && chk(cudaHostAlloc((void **)&h_words, 64 * 8, cudaHostAllocDefault))) return 1;
        for (int k = 0; k < n; ++k) if (chk(cudaMemcpyAsync(h_words + k, src[k], 8, cudaMemcpyDeviceToHost, st))) return 1;
        if (chk(cudaStreamSynchronize(st))) return 1;
        for (int k = 0; k < n; ++k) dst[k] = h_words[k];
        return 0;
    }
    int sync() { return chk(cudaStreamSynchronize(st)); }
    void tick(int k) { cudaEventRecord(ev[k], st); }
    float elapsed(int a, int b)
    {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ev[a], ev[b]);
        return ms;
    }
    std::string last_error() { return err; }
    int scan(const ScanArgs &a, bool small) { return chk(launch_scan(a, small, st)); }
    /* the barrier-free scan of clean inputs: 0 launched, -1 not to be used (XM_SCAN2=0), 1 launch error */
    int scan2(const ScanArgs &a)
    {
        static const bool off = [] { const char *e = getenv("XM_SCAN2"); return e && e[0] == '0'; }();
        if (off) return -1;
        return chk(launch_scan2(a, st));
    }
    int classify2(const ClassifyArgs &a)
    {
        static const bool off = [] { const char *e = getenv("XM_CLASSIFY2"); return e && e[0] == '0'; }();
        if (off) return -1;
        return chk(launch_classify2(a, st));
    }
    bool rows_enabled() { return true; }           /* the walk over rows (xm_emit.cuh), chosen with XM_DEBUG_ROWS */
    int size(const EmitArgs &a) { return chk(launch_size(a, st)); }
    int prefix(const EmitArgs &a) { return chk(launch_prefix(a, st)); }
    int emit(const EmitArgs &a) { return chk(launch_emit(a, st)); }
    int add64(void *p, uint64_t n, unsigned long long d) { return chk(launch_add_u64((unsigned long long *)p, d, n, st)) || chk(cudaStreamSynchronize(st)); }
    /* tiles the span kernels cut `len` bytes into at most, whatever geometry the launchers pick (look-back arrays are sized for it) */
    uint64_t scan2_tiles(uint64_t len) { const uint64_t t = span_tile_bytes_min(); return (len + t - 1) / t; }
    int classify(const ClassifyArgs &a, bool small) { return chk(launch_classify(a, small, st)); }
};

struct DevBuf {
    uint8_t *p = nullptr;
    uint64_t cap = 0;
};
/* two timing events that go away with the scope, whichever way it is left */
struct EventPair {
    cudaEvent_t a = nullptr, b = nullptr;
    EventPair() { cudaEventCreate(&a); cudaEventCreate(&b); }
    ~EventPair() { cudaEventDestroy(a); cudaEventDestroy(b); }
    EventPair(const EventPair &) = delete;
    EventPair &operator=(const EventPair &) = delete;
    float ms() const { float v = 0.f; cudaEventElapsedTime(&v, a, b); return v; }
};
struct HostBuf {
    uint8_t *p = nullptr;
    uint64_t cap = 0, len = 0;
};

/* the Comm of xm_shard.h over NCCL: small host vectors travel through a device staging buffer */
struct NcclComm_ {
    NcclComm comm = nullptr;
    int nranks = 1, my = 0;
    cudaStream_t st = nullptr;
    uint8_t *d_stage = nullptr;       /* [send | recv * nranks] */
    size_t stage_cap = 0;
    std::string err;
    int rank() const { return my; }
    int size() const { return nranks; }
    std::string last_error() const { return err; }
    int ck(int r, const char *what)
    {
        if (r == 0) return 0;
        const char *m = nccl_api().GetErrorString ? nccl_api().GetErrorString(r) : "?";
        err = std::string(what) + ": " + m;
        return 1;
    }
    int cu(cudaError_t e, const char *what)
    {
        if (e == cudaSuccess) return 0;
        err = std::string(what) + ": " + cudaGetErrorString(e);
        return 1;
    }
    int stage(size_t bytes)
    {
        const size_t need = bytes * ((size_t)nranks + 1) + 256;
        if (need <= stage_cap) return 0;
        if (d_stage) cudaFree(d_stage);
        d_stage = nullptr; stage_cap = 0;
        if (cu(cudaMalloc((void **)&d_stage, need), "cudaMalloc")) return 1;
        stage_cap = need;
        return 0;
    }
    int all_gather(const void *send, void *recv, size_t bytes)
    {
        if (nranks == 1) { memcpy(recv, send, bytes); return 0; }
        if (!comm) { err = "no communicator: call xm_comm_init_rank first"; return 1; }
        if (stage(bytes)) return 1;
        uint8_t *ds = d_stage, *dr = d_stage + ((bytes + 15) & ~(size_t)15);
        if (cu(cudaMemcpyAsync(ds, send, bytes, cudaMemcpyHostToDevice, st), "H2D copy")) return 1;
        if (ck(nccl_api().AllGather(ds, dr, bytes, NCCL_UINT8, comm, st), "ncclAllGather")) return 1;
        if (cu(cudaMemcpyAsync(recv, dr, bytes * (size_t)nranks, cudaMemcpyDeviceToHost, st), "D2H copy")) return 1;
        return cu(cudaStreamSynchronize(st), "all-gather");
    }
    int exchange(const Xfer *sends, int ns, const Xfer *recvs, int nr)
    {
        if (nranks == 1) return (ns || nr) ? (err = "exchange with one rank", 1) : 0;
        if (!comm) { err = "no communicator: call xm_comm_init_rank first"; return 1; }
        NcclApi &A = nccl_api();
        if (ck(A.GroupStart(), "ncclGroupStart")) return 1;
        int bad = 0;
        for (int k = 0; k < ns && !bad; ++k) bad = ck(A.Send(sends[k].ptr, (size_t)sends[k].bytes, NCCL_UINT8, sends[k].peer, comm, st), "ncclSend");
        for (int k = 0; k < nr && !bad; ++k) bad = ck(A.Recv(recvs[k].ptr, (size_t)recvs[k].bytes, NCCL_UINT8, recvs[k].peer, comm, st), "ncclRecv");
        if (ck(A.GroupEnd(), "ncclGroupEnd") || bad) return 1;
        return cu(cudaStreamSynchronize(st), "send/receive group");
    }
};

struct xm_ctx {
    int device = 0;
    DeviceBackend be;
    cudaStream_t copy_st[2] = {nullptr, nullptr};
    Scratch scratch;
    uint32_t debug = 0;
    std::string err;
    /* host-buffer walk: device staging and outputs, host outputs */
    DevBuf d_in[2][2], d_stage[2][2], d_out[2][6];     /* chunked walk: two walk and two staging buffers per stream, two sets of six bin buffers */
    HostBuf h_stage[2];      /* pinned blocks of the shard upload */
    HostBuf h_ring[2][3];    /* pinned slots descriptor sources are read ahead into */
    cudaStream_t dl = nullptr;          /* D2H lane */
    /* the six bins on the host: pinned blocks filled in order; reused from call to call */
    struct Block { uint8_t *p; uint64_t cap, len; };
    std::vector<Block> pool;            /* free blocks */
    std::vector<Block> bins[6];
    std::vector<uint8_t> flat[6];       /* xm_get_output of a bin that spans several blocks */
    uint64_t block_bytes = 0;
    /* BAM input: inflated windows, record tables, rendered SAM text */
    DevBuf d_bam[2], d_bam_rec[2], d_bam_ref[2], d_bam_len[2], d_bam_sum[2], d_bam_text[2];
    DevBuf d_bam_comp[2], d_bam_tab[2], d_bam_seg[2];      /* compressed window, its block table, the chain's segments */
    /* BGZF output deflated on the device (xm_deflate.h): member slots, sizes + offsets + plan, packed members per output set and bin */
    DevBuf d_zslot, d_zmeta, d_zout[2][6];
    void *bam_shard[2] = {nullptr, nullptr};      /* BamProducer of a rank's part of a BAM file (xm_bam_shard_*) */
    std::vector<uint8_t> z_host;
    xm_bgzf_stats bgzf_stats{};
    std::vector<uint8_t> bam_text_host;
    xm_bam_stats bam_stats{};
    /* the walk across GPUs (xm_shard.h): communicator, row scratch, shard staging of the host entry point */
    NcclComm_ comm;
    ShardScratch shard;
    DevBuf d_shard[2];
};
extern "C" { static void bam_shard_free(xm_ctx *c); }

static int fail(xm_ctx *c, int code, const std::string &msg)
{
    if (c) c->err = msg;
    return code;
}
static int cuda_fail(xm_ctx *c, cudaError_t e, const char *what)
{
    return fail(c, XM_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define XM_CUDA(c, call, what) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return cuda_fail((c), e_, (what)); } while (0)

int64_t xm::xm_pread_all(int fd, void *dst, uint64_t n, int64_t at)
{
    uint64_t got = 0;
    while (got < n) {
        const ssize_t r = pread(fd, (uint8_t *)dst + got, (size_t)std::min<uint64_t>(n - got, 1u << 30), (off_t)(at + (int64_t)got));
        if (r < 0) { if (errno == EINTR) continue; return -1; }
        if (r == 0) break;
        got += (uint64_t)r;
    }
    return (int64_t)got;
}

extern "C" {

int xm_abi_version(void) { return XM_ABI_VERSION; }

const char *xm_last_error(const xm_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

xm_ctx *xm_create(int device, uint32_t flags)
{
    (void)flags;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        g_create_error = std::string("no usable CUDA device: ") + (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                         " (this library has no CPU path)";
        return nullptr;
    }
    if (device < 0 || device >= n) { g_create_error = "device index out of range"; return nullptr; }
    cudaDeviceProp prop;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
        g_create_error = std::string("cudaSetDevice: ") + cudaGetErrorString(e);
        return nullptr;
    }
    if (prop.major != 10) {
        g_create_error = "kernels are built for sm_100a (B200) only; device is sm_" + std::to_string(prop.major) + std::to_string(prop.minor);
        return nullptr;
    }
    xm_ctx *c = new xm_ctx();
    c->device = device;
    if (cudaStreamCreateWithFlags(&c->be.st, cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&c->copy_st[0], cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&c->copy_st[1], cudaStreamNonBlocking) != cudaSuccess ||
        cudaStreamCreateWithFlags(&c->dl, cudaStreamNonBlocking) != cudaSuccess) {
        g_create_error = "cudaStreamCreate failed";
        delete c;
        return nullptr;
    }
    for (int k = 0; k < 6; ++k) cudaEventCreate(&c->be.ev[k]);
    c->be.up[0] = c->copy_st[0]; c->be.up[1] = c->copy_st[1];
    xm_set_debug(c, 0);
    return c;
}

void xm_destroy(xm_ctx *c)
{
    if (!c) return;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->be.st);
    scratch_release(c->be, c->scratch);
    shard_release(c->be, c->shard);
    xm_comm_destroy(c);
    for (auto &b : c->d_shard) if (b.p) cudaFree(b.p);
    for (auto &s : c->d_in) for (auto &b : s) if (b.p) cudaFree(b.p);
    for (auto &s : c->d_stage) for (auto &b : s) if (b.p) cudaFree(b.p);
    for (auto &s : c->h_ring) for (auto &b : s) if (b.p) cudaFreeHost(b.p);
    for (auto &s : c->d_out) for (auto &b : s) if (b.p) cudaFree(b.p);
    for (auto &b : c->h_stage) if (b.p) cudaFreeHost(b.p);
    bam_shard_free(c);
    if (c->d_zslot.p) cudaFree(c->d_zslot.p);
    if (c->d_zmeta.p) cudaFree(c->d_zmeta.p);
    for (auto *arr : {c->d_bam, c->d_bam_rec, c->d_bam_ref, c->d_bam_len, c->d_bam_sum, c->d_bam_text, c->d_bam_comp, c->d_bam_tab, c->d_bam_seg, c->d_zout[0], c->d_zout[0] + 2, c->d_zout[0] + 4, c->d_zout[1], c->d_zout[1] + 2, c->d_zout[1] + 4}) for (int k = 0; k < 2; ++k) if (arr[k].p) cudaFree(arr[k].p);
    for (auto &v : c->bins) for (auto &b : v) cudaFreeHost(b.p);
    for (auto &b : c->pool) cudaFreeHost(b.p);
    if (c->dl) cudaStreamDestroy(c->dl);
    for (int k = 0; k < 6; ++k) if (c->be.ev[k]) cudaEventDestroy(c->be.ev[k]);
    if (c->be.h_words) cudaFreeHost(c->be.h_words);
    if (c->be.st) cudaStreamDestroy(c->be.st);
    for (auto s : c->copy_st) if (s) cudaStreamDestroy(s);
    delete c;
}

int xm_set_debug(xm_ctx *c, uint32_t flags)
{
    if (!c) return XM_ERR_ARG;
    c->debug = flags;
    /* XM_ROWS=1 in the environment: every context walks over rows (benchmarks of the sharded walk's kernels) */
    static const bool rows = [] { const char *e = getenv("XM_ROWS"); return e && e[0] == '1'; }();
    if (rows) c->debug |= DBG_ROWS;
    static const bool exact = [] { const char *e = getenv("XM_EXACT_NAMES"); return e && e[0] == '1'; }();
    if (exact) c->debug |= DBG_EXACT_NAMES;
    return XM_OK;
}

/* ---- memory helpers ------------------------------------------------------ */
int xm_dev_alloc(xm_ctx *c, uint64_t bytes, void **d_ptr)
{
    if (!c || !d_ptr) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    cudaError_t e = cudaMalloc(d_ptr, bytes + 16);       /* readable up to the next multiple of 16 */
    if (e == cudaErrorMemoryAllocation) { cudaGetLastError(); return fail(c, XM_ERR_NOMEM, "cudaMalloc: out of memory"); }
    XM_CUDA(c, e, "cudaMalloc");
    return XM_OK;
}
int xm_dev_free(xm_ctx *c, void *d_ptr)
{
    if (!c) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    XM_CUDA(c, cudaFree(d_ptr), "cudaFree");
    return XM_OK;
}
int xm_host_alloc_pinned(xm_ctx *c, uint64_t bytes, void **h_ptr)
{
    if (!c || !h_ptr) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    cudaError_t e = cudaHostAlloc(h_ptr, bytes + 16, cudaHostAllocDefault);
    if (e == cudaErrorMemoryAllocation) { cudaGetLastError(); return fail(c, XM_ERR_NOMEM, "cudaHostAlloc: out of memory"); }
    XM_CUDA(c, e, "cudaHostAlloc");
    return XM_OK;
}
int xm_host_free_pinned(xm_ctx *c, void *h_ptr)
{
    if (!c) return XM_ERR_ARG;
    XM_CUDA(c, cudaFreeHost(h_ptr), "cudaFreeHost");
    return XM_OK;
}
int xm_memcpy_h2d(xm_ctx *c, void *d, const void *h, uint64_t n)
{
    if (!c) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    XM_CUDA(c, cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, c->be.st), "H2D copy");
    XM_CUDA(c, cudaStreamSynchronize(c->be.st), "H2D copy");
    return XM_OK;
}
int xm_memcpy_d2h(xm_ctx *c, void *h, const void *d, uint64_t n)
{
    if (!c) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    XM_CUDA(c, cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, c->be.st), "D2H copy");
    XM_CUDA(c, cudaStreamSynchronize(c->be.st), "D2H copy");
    return XM_OK;
}
int xm_memcpy_d2d(xm_ctx *c, void *dst, const void *src, uint64_t n)
{
    if (!c) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    XM_CUDA(c, cudaMemcpyAsync(dst, src, n, cudaMemcpyDeviceToDevice, c->be.st), "D2D copy");
    XM_CUDA(c, cudaStreamSynchronize(c->be.st), "D2D copy");
    return XM_OK;
}
int xm_dev_mem_info(xm_ctx *c, uint64_t *free_b, uint64_t *total_b)
{
    if (!c) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    size_t f = 0, t = 0;
    XM_CUDA(c, cudaMemGetInfo(&f, &t), "cudaMemGetInfo");
    if (free_b) *free_b = f;
    if (total_b) *total_b = t;
    return XM_OK;
}

/* ---- device-resident walk ---------------------------------------------------- */
int xm_classify_device(xm_ctx *c, const void *d_prim, uint64_t prim_len, const void *d_sec, uint64_t sec_len,
                       const xm_opts *opts, void *const d_out[6], const uint64_t out_cap[6], xm_result *res)
{
    if (!c || !opts || !res) return XM_ERR_ARG;
    if (((uintptr_t)d_prim | (uintptr_t)d_sec) & 15) return fail(c, XM_ERR_ARG, "device inputs must be 16-byte aligned");
    cudaSetDevice(c->device);
    uint8_t *o6[6];
    uint64_t cap6[6];
    for (int b = 0; b < 6; ++b) { o6[b] = d_out ? (uint8_t *)d_out[b] : nullptr; cap6[b] = (out_cap && o6[b]) ? out_cap[b] : 0; }
    std::string msg;
    WalkCtl ctl;
    ctl.halo = (opts->skip_repeated >> 1) & 1;
    xm_opts o = *opts;
    o.skip_repeated &= 1;
    const int rc = walk_resident(c->be, c->scratch, StreamBuf{(const uint8_t *)d_prim, prim_len}, StreamBuf{(const uint8_t *)d_sec, sec_len},
                                 o, o6, cap6, c->debug, res, msg, &ctl);
    if (ctl.halo && res->n_records) res->n_records -= 1;
    c->err = msg;
    return rc;
}

/* ---- host-buffer walk ----------------------------------------------------------- */
static int reserve_dev(xm_ctx *c, DevBuf &b, uint64_t n)
{
    if (n <= b.cap && b.p) return XM_OK;
    if (b.p) cudaFree(b.p);
    b.p = nullptr; b.cap = 0;
    cudaError_t e = cudaMalloc((void **)&b.p, n + 64);
    if (e != cudaSuccess) { cudaGetLastError(); b.p = nullptr; return fail(c, XM_ERR_NOMEM, std::string("cudaMalloc: ") + cudaGetErrorString(e)); }
    b.cap = n;
    return XM_OK;
}
static int reserve_host(xm_ctx *c, HostBuf &b, uint64_t n)
{
    if (n <= b.cap && b.p) return XM_OK;
    if (b.p) cudaFreeHost(b.p);
    b.p = nullptr; b.cap = 0;
    cudaError_t e = cudaHostAlloc((void **)&b.p, n + 64, cudaHostAllocDefault);
    if (e != cudaSuccess) { cudaGetLastError(); b.p = nullptr; return fail(c, XM_ERR_NOMEM, std::string("cudaHostAlloc: ") + cudaGetErrorString(e)); }
    b.cap = n;
    return XM_OK;
}

/* upper bounds of what each bin can receive from these inputs (xm.py:332-350, 423-448):
 * primary lines go to PS/PM/UA/UR, secondary lines to SS/SM/UR; an unterminated last
 * line gains a newline; overlapping pair units can emit a line twice. */
static void bin_bounds(uint64_t plen, uint64_t slen, int mode, uint32_t enabled, uint64_t cap[6])
{
    const uint64_t mul = mode == XM_MODE_SE ? 1 : 2;
    const uint64_t pb = (plen + 1) * mul, sb = (slen + 1) * mul;
    const uint64_t b[6] = {pb, sb, pb, sb, pb, pb + sb};
    for (int k = 0; k < 6; ++k) cap[k] = ((enabled >> k) & 1u) ? b[k] : 0;
}

/* ---- the chunked walk behind the host-buffer and the descriptor entry points ------------- */
static uint64_t chunk_bytes()
{
    const char *e = getenv("XM_CHUNK_BYTES");
    if (e && *e) { const long long v = atoll(e); if (v > 0) return (uint64_t)v; }
    e = getenv("XM_CHUNK_MB");
    if (e && *e) { const long long v = atoll(e); if (v > 0) return (uint64_t)v << 20; }
    return 256ull << 20;
}

static void recycle_bins(xm_ctx *c)
{
    for (auto &v : c->bins) { for (auto &b : v) { b.len = 0; c->pool.push_back(b); } v.clear(); }
    for (auto &f : c->flat) f.clear();
}

/* room for n more bytes of bin b: the tail of its last block, then fresh blocks */
static int bin_append_d2h(xm_ctx *c, int b, const uint8_t *d_src, uint64_t n)
{
    while (n) {
        if (c->bins[b].empty() || c->bins[b].back().len == c->bins[b].back().cap) {
            xm_ctx::Block blk{nullptr, 0, 0};
            for (size_t k = 0; k < c->pool.size(); ++k)
                if (c->pool[k].cap >= c->block_bytes) { blk = c->pool[k]; c->pool.erase(c->pool.begin() + (long)k); break; }
            if (!blk.p) {
                cudaError_t e = cudaHostAlloc((void **)&blk.p, c->block_bytes + 64, cudaHostAllocDefault);
                if (e != cudaSuccess) { cudaGetLastError(); return fail(c, XM_ERR_NOMEM, std::string("cudaHostAlloc: ") + cudaGetErrorString(e)); }
                blk.cap = c->block_bytes;
            }
            blk.len = 0;
            c->bins[b].push_back(blk);
        }
        xm_ctx::Block &k = c->bins[b].back();
        const uint64_t m = std::min<uint64_t>(n, k.cap - k.len);
        cudaError_t e = cudaMemcpyAsync(k.p + k.len, d_src, m, cudaMemcpyDeviceToHost, c->dl);
        if (e != cudaSuccess) return cuda_fail(c, e, "D2H copy");
        k.len += m; d_src += m; n -= m;
    }
    return XM_OK;
}

static int host_threads();
static int upload_shard(xm_ctx *c, uint8_t *d_dst, const uint8_t *src, uint64_t n);

static bool bgzf_on_host()
{
    const char *e = getenv("XM_BGZF_DEFLATE");
    return e && !strcmp(e, "host");
}

/* n bytes at d_src (device, 4-byte aligned, readable 8 bytes past the end) as BGZF members in `Z` (device): xm_deflate.h.
 * plan: the bin's code, made from a sample of these bytes when *have_plan is false.  The stream is synchronised on return. */
static int device_bgzf(xm_ctx *c, const uint8_t *d_src, uint64_t n, DevBuf &Z, uint64_t *z_len, DeflatePlan *plan, bool *have_plan)
{
    *z_len = 0;
    if (!n) return XM_OK;
    cudaStream_t st = c->be.st;
    int sm_count = 148;
    cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, c->device);
    const uint32_t in_per = deflate_member_bytes(n, (uint32_t)sm_count), slot_bytes = deflate_slot_bytes(in_per);
    const uint64_t members = (n + in_per - 1) / in_per;
    int rc;
    const uint64_t meta = members * 4 + 8 + (members + 1) * 8 + sizeof(DeflatePlan) + 316 * 4 + 16;
    if ((rc = reserve_dev(c, c->d_zslot, members * (uint64_t)slot_bytes + 64)) || (rc = reserve_dev(c, c->d_zmeta, meta + 64))) return rc;
    unsigned long long *d_offs = (unsigned long long *)c->d_zmeta.p;
    DeflatePlan *d_plan = (DeflatePlan *)(d_offs + members + 1);
    uint32_t *d_sizes = (uint32_t *)(d_plan + 1);
    if (!*have_plan) {
        /* the bin's code: a first guess from a sample of its bytes; the first members are deflated with it and the
         * symbols of the tokens that come out make the code that is used */
        std::vector<uint8_t> sample((size_t)std::min<uint64_t>(n, 256u << 10));
        XM_CUDA(c, cudaMemcpyAsync(sample.data(), d_src, sample.size(), cudaMemcpyDeviceToHost, st), "D2H copy");
        XM_CUDA(c, cudaStreamSynchronize(st), "D2H copy");
        deflate_plan(sample.data(), sample.size(), *plan);
        const uint32_t probe = (uint32_t)std::min<uint64_t>(members, 512);
        uint32_t *d_hist = (uint32_t *)(d_sizes + members + 1);
        uint32_t hist[316];
        cudaMemcpyAsync(d_plan, plan, sizeof *plan, cudaMemcpyHostToDevice, st);
        cudaMemsetAsync(d_hist, 0, sizeof hist, st);
        k_bgzf_deflate<<<(probe + DEF_WARPS - 1) / DEF_WARPS, DEF_WARPS * 32, 0, st>>>(d_src, std::min<uint64_t>(n, (uint64_t)probe * in_per), probe, in_per, slot_bytes, d_plan, c->d_zslot.p, d_sizes, d_hist);
        XM_CUDA(c, cudaMemcpyAsync(hist, d_hist, sizeof hist, cudaMemcpyDeviceToHost, st), "D2H copy");
        XM_CUDA(c, cudaStreamSynchronize(st), "BGZF deflate kernel");
        deflate_plan_hist(hist, *plan);
        c->bgzf_stats.n_launches += 1;
        *have_plan = true;
    }
    EventPair ev;
    cudaMemcpyAsync(d_plan, plan, sizeof *plan, cudaMemcpyHostToDevice, st);
    cudaEventRecord(ev.a, st);
    k_bgzf_deflate<<<(unsigned)((members + DEF_WARPS - 1) / DEF_WARPS), DEF_WARPS * 32, 0, st>>>(d_src, n, (uint32_t)members, in_per, slot_bytes, d_plan, c->d_zslot.p, d_sizes, nullptr);
    k_bgzf_offsets<<<1, 1024, 0, st>>>(d_sizes, (uint32_t)members, d_offs);
    unsigned long long total = 0;
    cudaMemcpyAsync(&total, d_offs + members, 8, cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(c, e, "BGZF deflate kernel");
    if ((rc = reserve_dev(c, Z, total + 64))) return rc;
    k_bgzf_pack<<<(unsigned)((members * 32 + 255) / 256), 256, 0, st>>>(c->d_zslot.p, slot_bytes, d_sizes, d_offs, (uint32_t)members, Z.p);
    cudaEventRecord(ev.b, st);
    e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(c, e, "BGZF pack kernel");
    c->bgzf_stats.in_bytes += n; c->bgzf_stats.out_bytes += total; c->bgzf_stats.members += members; c->bgzf_stats.kernel_ms += ev.ms();
    c->bgzf_stats.n_launches += 3;
    *z_len = total;
    return XM_OK;
}

/* The bins of a descriptor walk are written by a thread of their own: a step's blocks are queued behind the event
 * that marks the end of their D2H copies, written with write(2) in bin order, and handed back to the pool. */
struct BinWriter {
    struct Job { cudaEvent_t ev; std::vector<std::pair<int, xm_ctx::Block>> blocks; };
    xm_ctx *c;
    const int *fds;
    std::thread th;
    std::mutex mu;
    std::condition_variable cv;
    std::vector<Job> queue;
    std::vector<xm_ctx::Block> done;        /* written blocks, for the pool */
    size_t in_flight = 0;
    bool stop = false;
    int rc = XM_OK;
    std::string err;
    bool regular[6] = {false, false, false, false, false, false};      /* seekable regular files not opened for append */
    bool bgzf = false;                      /* XM_OUT_BGZF: the blocks leave as BGZF members */
    BinWriter(xm_ctx *ctx, const int *out_fds, bool as_bgzf = false) : c(ctx), fds(out_fds), bgzf(as_bgzf)
    {
        for (int b = 0; b < 6; ++b) {
            struct stat sb;
            if (fds[b] >= 0 && fstat(fds[b], &sb) == 0 && S_ISREG(sb.st_mode) && !(fcntl(fds[b], F_GETFL) & O_APPEND)) regular[b] = true;
        }
        th = std::thread([this] { run(); });
    }
    void run()
    {
        cudaSetDevice(c->device);
        for (;;) {
            Job j;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return stop || !queue.empty(); });
                if (queue.empty()) return;
                j = std::move(queue.front());
                queue.erase(queue.begin());
            }
            if (cudaEventSynchronize(j.ev) != cudaSuccess && rc == XM_OK) { rc = XM_ERR_CUDA; err = "D2H copy failed"; }
            cudaEventDestroy(j.ev);
            for (auto &kb : j.blocks) {
                uint64_t w0 = 0;
                const int fd = fds[kb.first];
                if (bgzf) {
                    if (rc == XM_OK && fd >= 0 && kb.second.len) {
                        std::vector<uint8_t> z;
                        if (!bgzf_compress(kb.second.p, kb.second.len, bgzf_level(), host_threads(), z)) { rc = XM_ERR_IO; err = "deflate failed"; }
                        uint64_t zw = 0;
                        while (rc == XM_OK && zw < z.size()) {
                            const ssize_t w = write(fd, z.data() + zw, (size_t)std::min<uint64_t>(z.size() - zw, 1u << 30));
                            if (w < 0) { if (errno == EINTR) continue; rc = XM_ERR_IO; err = std::string("write: ") + strerror(errno); break; }
                            zw += (uint64_t)w;
                        }
                    }
                    continue;
                }
                if (rc == XM_OK && fd >= 0 && regular[kb.first] && kb.second.len >= (32ull << 20)) {
                    /* a regular file: the block goes out as pwrites side by side behind the descriptor's position */
                    const off_t at = lseek(fd, 0, SEEK_CUR);
                    if (at >= 0) {
                        const int nt = std::max(1, std::min(8, host_threads() / 2));
                        const uint64_t per = ((kb.second.len + (uint64_t)nt - 1) / (uint64_t)nt + 4095) & ~4095ull;
                        std::vector<std::thread> th;
                        std::vector<int> bad((size_t)nt, 0);
                        for (int t = 0; t < nt; ++t)
                            th.emplace_back([&, t] {
                                uint64_t lo = (uint64_t)t * per;
                                const uint64_t hi = std::min<uint64_t>(lo + per, kb.second.len);
                                while (lo < hi) {
                                    const ssize_t w = pwrite(fd, kb.second.p + lo, (size_t)std::min<uint64_t>(hi - lo, 1u << 30), at + (off_t)lo);
                                    if (w < 0) { if (errno == EINTR) continue; bad[(size_t)t] = errno; return; }
                                    lo += (uint64_t)w;
                                }
                            });
                        for (auto &t : th) t.join();
                        for (int e : bad) if (e && rc == XM_OK) { rc = XM_ERR_IO; err = std::string("write: ") + strerror(e); }
                        if (rc == XM_OK && lseek(fd, at + (off_t)kb.second.len, SEEK_SET) < 0) { rc = XM_ERR_IO; err = std::string("lseek: ") + strerror(errno); }
                        w0 = kb.second.len;
                    }
                }
                while (rc == XM_OK && fd >= 0 && w0 < kb.second.len) {
                    const ssize_t w = write(fd, kb.second.p + w0, (size_t)std::min<uint64_t>(kb.second.len - w0, 1u << 30));
                    if (w < 0) { if (errno == EINTR) continue; rc = XM_ERR_IO; err = std::string("write: ") + strerror(errno); break; }
                    w0 += (uint64_t)w;
                }
            }
            {
                std::lock_guard<std::mutex> lk(mu);
                for (auto &kb : j.blocks) { kb.second.len = 0; done.push_back(kb.second); }
                --in_flight;
            }
            cv.notify_all();
        }
    }
    /* the blocks the bins hold now, to be written once the D2H lane has passed this point */
    void push(cudaStream_t dl)
    {
        Job j;
        cudaEventCreateWithFlags(&j.ev, cudaEventDisableTiming);
        cudaEventRecord(j.ev, dl);
        for (int b = 0; b < 6; ++b) { for (auto &k : c->bins[b]) j.blocks.push_back({b, k}); c->bins[b].clear(); }
        { std::lock_guard<std::mutex> lk(mu); queue.push_back(std::move(j)); ++in_flight; }
        cv.notify_all();
    }
    void reclaim()
    {
        std::lock_guard<std::mutex> lk(mu);
        for (auto &k : done) c->pool.push_back(k);
        done.clear();
    }
    /* at most `keep` steps' worth of blocks may be waiting for the descriptors */
    void wait_below(size_t keep)
    {
        std::unique_lock<std::mutex> lk(mu);
        cv.wait(lk, [&] { return in_flight <= keep; });
    }
    int finish()
    {
        wait_below(0);
        { std::lock_guard<std::mutex> lk(mu); stop = true; }
        cv.notify_all();
        if (th.joinable()) th.join();
        reclaim();
        return rc;
    }
};

/* out_fds == nullptr: keep the bins in host blocks (xm_get_output); else append each step's bytes to the descriptors */
static int stream_walk(xm_ctx *c, HostIn in[2], const int *out_fds, const xm_opts *opts, xm_result *res, uint32_t out_flags = 0)
{
    cudaSetDevice(c->device);
    recycle_bins(c);
    const uint64_t want = chunk_bytes();
    const uint64_t longest = std::max(in[0].len, in[1].len);
    StreamPlan plan;
    plan.chunk = std::max<uint64_t>(std::min<uint64_t>(want, longest + 64), 64);
    const uint64_t cap = 2 * plan.chunk + 64;
    DevIn dev[2];
    int rc;
    for (int s = 0; s < 2; ++s) {
        for (int k = 0; k < 2; ++k) {
            if ((rc = reserve_dev(c, c->d_in[k][s], cap)) || (rc = reserve_dev(c, c->d_stage[k][s], cap))) return rc;
            dev[s].buf[k] = c->d_in[k][s].p; dev[s].stage[k] = c->d_stage[k][s].p;
        }
        dev[s].cap = cap;
    }
    /* descriptor sources: a reader thread each, three pinned slots of one chunk */
    FdFeeder feeders[2];
    for (int s = 0; s < 2; ++s) {
        if (!in[s].feed) continue;
        FdFeeder &f = feeders[s];
        f.fd = in[s].feed->fd; f.off = in[s].feed->off; f.len = in[s].len;
        f.seekable = in[s].feed->seekable; f.pre.swap(in[s].feed->pre);
        f.slot_cap = std::max<uint64_t>(std::min<uint64_t>(plan.chunk, in[s].len + 64), 64);
        f.threads = std::max(1, host_threads() / 2);         /* page-cache reads are memcpy-bound per thread */
        f.ring.resize(3);
        for (int k = 0; k < 3; ++k) {
            if ((rc = reserve_host(c, c->h_ring[s][k], f.slot_cap))) return rc;
            f.ring[(size_t)k].p = c->h_ring[s][k].p;
        }
        in[s].feed = &f;
        f.start();
    }
    uint64_t ocap[6];
    bin_bounds(cap, cap, opts->mode, opts->enabled_bins, ocap);
    uint8_t *outs[2][6];
    for (int k = 0; k < 2; ++k)
        for (int b = 0; b < 6; ++b) { if ((rc = reserve_dev(c, c->d_out[k][b], ocap[b]))) { for (auto &f : feeders) f.shutdown(); return rc; } outs[k][b] = c->d_out[k][b].p; }
    /* host blocks: a step's worth per block at most, small inputs get small blocks */
    uint64_t bound[6];
    bin_bounds(in[0].len, in[1].len, opts->mode, opts->enabled_bins, bound);
    const uint64_t biggest = *std::max_element(bound, bound + 6);
    c->block_bytes = std::max<uint64_t>(std::min<uint64_t>(biggest, 256ull << 20), 4096);

    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0, c->be.st);
    const bool z_device = out_fds && (out_flags & XM_OUT_BGZF) && !bgzf_on_host();
    std::vector<DeflatePlan> z_plan(6);
    bool z_have[6] = {false, false, false, false, false, false};
    BinWriter *writer = out_fds ? new BinWriter(c, out_fds, (out_flags & XM_OUT_BGZF) != 0 && !z_device) : nullptr;
    int emit_rc = XM_OK;
    cudaEvent_t set_done[2];
    bool set_used[2] = {false, false};
    for (auto &e : set_done) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    auto emit = [&](int set, int b, const uint8_t *d_src, uint64_t n) {
        if (emit_rc) return;
        if (b < 0) {
            /* the step's D2H copies are all queued: mark the point, and let the writer have the blocks */
            cudaEventRecord(set_done[set], c->dl);
            set_used[set] = true;
            if (writer) writer->push(c->dl);
            return;
        }
        if (writer) writer->reclaim();
        if (z_device) {
            /* the bin leaves the device as BGZF members: deflated where it lies, then copied */
            uint64_t zn = 0;
            emit_rc = device_bgzf(c, d_src, n, c->d_zout[set][b], &zn, &z_plan[b], &z_have[b]);
            if (!emit_rc) emit_rc = bin_append_d2h(c, b, c->d_zout[set][b].p, zn);
            return;
        }
        emit_rc = bin_append_d2h(c, b, d_src, n);
    };
    int wait_rc = XM_OK;
    /* before output set `set` is written again: the D2H copies of the step that used it two steps ago are done (the
     * copies of the step in between go on), and at most two steps' blocks are waiting for the descriptors */
    auto emit_wait = [&](int set) {
        if (wait_rc) return;
        if (set_used[set] && cudaEventSynchronize(set_done[set]) != cudaSuccess) wait_rc = fail(c, XM_ERR_CUDA, "D2H copy failed");
        if (writer) writer->wait_below(2);
    };
    std::string msg;
    xm_opts o = *opts;
    o.skip_repeated &= 1;
    rc = walk_stream(c->be, c->scratch, in, dev, outs, ocap, o, c->debug, plan, emit, emit_wait, res, msg, (opts->skip_repeated >> 1) & 1);
    for (auto &f : feeders) f.shutdown();
    c->err = msg;
    if (emit_rc) rc = emit_rc;
    if (wait_rc) rc = wait_rc;
    for (auto &e : set_done) cudaEventDestroy(e);
    if (writer) {
        const int r2 = writer->finish();
        if (r2 && (rc == XM_OK || (rc != XM_ERR_CUDA && rc != XM_ERR_NOMEM))) { rc = r2; c->err = writer->err; }
        delete writer;
    } else if (rc != XM_ERR_CUDA && rc != XM_ERR_NOMEM) {
        if (cudaStreamSynchronize(c->dl) != cudaSuccess) rc = fail(c, XM_ERR_CUDA, "D2H copy failed");
    }
    cudaEventRecord(e1, c->be.st);
    cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    res->ms_total = ms;                 /* the whole call: staging, kernels, the bins back on the host (and written) */
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return rc;
}

int xm_classify_host(xm_ctx *c, const void *prim, uint64_t prim_len, const void *sec, uint64_t sec_len,
                     const xm_opts *opts, xm_result *res)
{
    if (!c || !opts || !res) return XM_ERR_ARG;
    HostIn in[2];
    in[0].mem = (const uint8_t *)prim; in[0].len = prim_len;
    in[1].mem = (const uint8_t *)sec; in[1].len = sec_len;
    static const uint8_t nothing = 0;
    if (!in[0].mem) in[0].mem = &nothing;
    if (!in[1].mem) in[1].mem = &nothing;
    return stream_walk(c, in, nullptr, opts, res);
}

int xm_get_output(xm_ctx *c, int bin, const void **data, uint64_t *len)
{
    if (!c || bin < 0 || bin > 5 || !data || !len) return XM_ERR_ARG;
    auto &v = c->bins[bin];
    if (v.empty()) { *data = nullptr; *len = 0; return XM_OK; }
    if (v.size() == 1) { *data = v[0].p; *len = v[0].len; return XM_OK; }
    if (c->flat[bin].empty()) {
        uint64_t n = 0;
        for (auto &b : v) n += b.len;
        c->flat[bin].resize(n);
        uint64_t at = 0;
        for (auto &b : v) { memcpy(c->flat[bin].data() + at, b.p, b.len); at += b.len; }
    }
    *data = c->flat[bin].data();
    *len = c->flat[bin].size();
    return XM_OK;
}

/* ---- file-descriptor walk ---------------------------------------------------------- */
int xm_classify_fds(xm_ctx *c, int fd_prim, int64_t off_prim, int fd_sec, int64_t off_sec, const int out_fds[6],
                    const xm_opts *opts, xm_result *res)
{
    return xm_classify_fds_ex(c, fd_prim, off_prim, fd_sec, off_sec, out_fds, opts, 0, res);
}

int xm_bgzf_deflate_host(xm_ctx *c, const void *data, uint64_t len, const void **out, uint64_t *out_len)
{
    if (!c || (!data && len) || !out || !out_len) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    *out = nullptr; *out_len = 0;
    int rc;
    if ((rc = reserve_dev(c, c->d_bam_text[0], len + 64))) return rc;           /* any idle device buffer will do for the input */
    if ((rc = upload_shard(c, c->d_bam_text[0].p, (const uint8_t *)data, len))) return rc;
    DeflatePlan plan;
    bool have = false;
    uint64_t zn = 0;
    if ((rc = device_bgzf(c, c->d_bam_text[0].p, len, c->d_zout[0][0], &zn, &plan, &have))) return rc;
    c->z_host.resize(zn);
    if (zn) {
        XM_CUDA(c, cudaMemcpyAsync(c->z_host.data(), c->d_zout[0][0].p, zn, cudaMemcpyDeviceToHost, c->be.st), "D2H copy");
        XM_CUDA(c, cudaStreamSynchronize(c->be.st), "D2H copy");
    }
    *out = c->z_host.data();
    *out_len = zn;
    return XM_OK;
}

int xm_bgzf_get_stats(xm_ctx *c, xm_bgzf_stats *out, int reset)
{
    if (!c || !out) return XM_ERR_ARG;
    *out = c->bgzf_stats;
    if (reset) c->bgzf_stats = xm_bgzf_stats{};
    return XM_OK;
}

int xm_bgzf_write(int fd, const void *data, uint64_t len, int eof)
{
    if (fd < 0 || (!data && len)) return XM_ERR_ARG;
    std::vector<uint8_t> z;
    if (len && !bgzf_compress((const uint8_t *)data, len, bgzf_level(), host_threads(), z)) { g_create_error = "deflate failed"; return XM_ERR_IO; }
    if (eof) z.insert(z.end(), BGZF_EOF, BGZF_EOF + sizeof BGZF_EOF);
    uint64_t at = 0;
    while (at < z.size()) {
        const ssize_t w = write(fd, z.data() + at, (size_t)std::min<uint64_t>(z.size() - at, 1u << 30));
        if (w < 0) { if (errno == EINTR) continue; g_create_error = std::string("write: ") + strerror(errno); return XM_ERR_IO; }
        at += (uint64_t)w;
    }
    return XM_OK;
}

int xm_classify_fds_ex(xm_ctx *c, int fd_prim, int64_t off_prim, int fd_sec, int64_t off_sec, const int out_fds[6],
                       const xm_opts *opts, uint32_t out_flags, xm_result *res)
{
    if (!c || !opts || !res || !out_fds) return XM_ERR_ARG;
    HostIn in[2];
    FdFeeder where[2];                  /* descriptor and offset only: stream_walk sets the readers up */
    const int fds[2] = {fd_prim, fd_sec};
    const int64_t offs[2] = {off_prim, off_sec};
    for (int s = 0; s < 2; ++s) {
        const off_t end = lseek(fds[s], 0, SEEK_END);
        if (end < 0) return fail(c, XM_ERR_IO, std::string("input must be seekable: ") + strerror(errno));
        where[s].fd = fds[s]; where[s].off = offs[s];
        in[s].feed = &where[s];
        in[s].len = (uint64_t)end > (uint64_t)offs[s] ? (uint64_t)end - (uint64_t)offs[s] : 0;
    }
    xm_opts o = *opts;
    uint32_t en = 0;
    for (int b = 0; b < 6; ++b) if (out_fds[b] >= 0) en |= 1u << b;
    o.enabled_bins = en;
    return stream_walk(c, in, out_fds, &o, res, out_flags);
}

/* ---- BAM input (xm_bam.h) ------------------------------------------------------------------ */
static int host_threads()
{
    const char *e = getenv("XM_HOST_THREADS");
    if (e && *e) { const int v = atoi(e); if (v > 0) return v; }
    const unsigned h = std::thread::hardware_concurrency();
    return (int)std::min<unsigned>(h ? h : 1, 32);
}

/* one BAM file as SAM text in device memory (slot s); defined behind BamProducer */
static int bam_to_device_text(xm_ctx *c, const void *bam, uint64_t len, int s, uint8_t **d_text, uint64_t *text_len);

/* the header and reference names of a BAM file (blocks: its bgzf_scan table): 4, 16, 64 ... leading blocks inflated on
 * `threads` host threads until the header is complete */
static bool bam_read_header(const uint8_t *bam, const std::vector<BgzfBlock> &blocks, uint64_t total, int threads, BamIndex &ix, std::string &err)
{
    for (size_t take = std::min<size_t>(blocks.size(), 4);; take = std::min(blocks.size(), take * 4)) {
        const uint64_t bytes = take < blocks.size() ? blocks[take].out_off : total;
        std::vector<uint8_t> buf(bytes + 16);
        if (!bgzf_inflate(bam, blocks, 0, take, buf.data(), threads, err)) return false;
        ix = BamIndex();
        if (bam_index(buf.data(), bytes, ix, true, err)) return true;
        if (take == blocks.size()) return false;
    }
}

int xm_bam_header_text(const void *bam, uint64_t len, char *dst, uint64_t cap, uint64_t *needed)
{
    if (!bam || !needed) return XM_ERR_ARG;
    std::string err;
    std::vector<BgzfBlock> blocks;
    uint64_t total = 0;
    BamIndex ix;
    if (!bgzf_scan((const uint8_t *)bam, len, blocks, total, err) || !bam_read_header((const uint8_t *)bam, blocks, total, 1, ix, err)) {
        g_create_error = "BAM input: " + err;
        return XM_ERR_IO;
    }
    *needed = ix.text.size();
    if (dst && cap >= ix.text.size()) memcpy(dst, ix.text.data(), ix.text.size());
    return XM_OK;
}

int xm_bam_render_host(xm_ctx *c, const void *bam, uint64_t len, const void **text, uint64_t *text_len)
{
    if (!c || !bam || !text || !text_len) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    uint8_t *d = nullptr;
    uint64_t n = 0;
    const int rc = bam_to_device_text(c, bam, len, 0, &d, &n);
    if (rc) return rc;
    c->bam_text_host.resize(n);
    if (n) {
        XM_CUDA(c, cudaMemcpyAsync(c->bam_text_host.data(), d, n, cudaMemcpyDeviceToHost, c->be.st), "D2H copy");
        XM_CUDA(c, cudaStreamSynchronize(c->be.st), "D2H copy");
    }
    *text = c->bam_text_host.data();
    *text_len = n;
    return XM_OK;
}

static uint64_t bam_window_bytes()
{
    const char *e = getenv("XM_BAM_WINDOW");
    if (e && *e) { const long long v = atoll(e); if (v > 0) return (uint64_t)v; }
    return 1ull << 30;
}
static uint64_t bam_seg_bytes()
{
    const char *e = getenv("XM_BAM_SEG");
    if (e && *e) { const long long v = atoll(e); if (v >= 64) return (uint64_t)v; }
    return 16384;
}
static bool bam_inflate_on_host()
{
    const char *e = getenv("XM_BAM_INFLATE");
    return e && !strcmp(e, "host");
}

/* BAM as a source of the chunked walk.  The file is taken a window of BGZF blocks at a time (XM_BAM_WINDOW): the blocks
 * are inflated into device memory (k_bgzf_inflate; XM_BAM_INFLATE=host: zlib on the host threads, then uploaded), the
 * record chain is followed by k_bam_chain, and each call renders records of the window as SAM text straight into the
 * walk's staging buffer.  What is resident at any time is one window, not the file: the inflated size of a BAM does not
 * have to fit the GPU. */
struct BamProducer : DevSource {
    xm_ctx *c = nullptr;
    int s = 0;
    const uint8_t *bam = nullptr;
    uint64_t bam_len = 0;
    std::vector<BgzfBlock> blocks;
    size_t blk = 0;
    uint32_t n_ref = 0;
    uint8_t *d_names = nullptr;
    uint64_t full_cap = 0;              /* the walk's whole staging step: a record that does not fit it is refused */

    bool host_mode = false;             /* XM_BAM_INFLATE=host: blocks inflated by zlib on the host threads */
    std::vector<uint8_t> h_piece;       /* host mode: inflated blocks on their way to d_bam[s] */
    uint64_t inflated_total = 0;
    uint64_t skip = 0;                  /* header bytes of the inflated stream that are still ahead */
    uint64_t have_d = 0, win_end = 0;   /* inflated bytes in d_bam[s]; end of the last whole record among them */
    uint64_t n_rec = 0, r_next = 0;     /* records of the window; the next one to render */
    uint64_t cut_off = 0;               /* text bytes of r_next's group of 1024 that are rendered already */
    std::vector<ChainSeg> seg0;         /* the segments' guesses of the current window */
    bool seg_valid = false;
    uint64_t skip_abs = 0;              /* offset of the first record in the inflated stream */
    std::vector<unsigned long long> sums;      /* text bytes of each group of 1024 records of the window */

    /* block table, header (leading blocks inflated on the host: a few KiB), reference names to the device */
    int open(std::string &err)
    {
        host_mode = bam_inflate_on_host();
        std::string e;
        if (!bgzf_scan(bam, bam_len, blocks, inflated_total, e)) { err = "BAM input: " + e; return XM_ERR_IO; }
        c->bam_stats.bam_bytes += bam_len;
        BamIndex ix;
        if (!bam_read_header(bam, blocks, inflated_total, host_threads(), ix, e)) { err = "BAM input: " + e; return XM_ERR_IO; }
        skip = ix.first_record;
        skip_abs = ix.first_record;
        n_ref = (uint32_t)ix.ref_off.size() - 1;
        const uint64_t ref_bytes = ix.ref_off.size() * 4 + ix.ref_names.size() + 16;
        int rc;
        if ((rc = reserve_dev(c, c->d_bam_ref[s], ref_bytes))) { err = c->err; return rc; }
        cudaMemcpyAsync(c->d_bam_ref[s].p, ix.ref_off.data(), ix.ref_off.size() * 4, cudaMemcpyHostToDevice, c->be.st);
        d_names = c->d_bam_ref[s].p + ix.ref_off.size() * 4;
        if (!ix.ref_names.empty()) cudaMemcpyAsync(d_names, ix.ref_names.data(), ix.ref_names.size(), cudaMemcpyHostToDevice, c->be.st);
        if (cudaStreamSynchronize(c->be.st) != cudaSuccess) { err = "H2D copy failed"; return XM_ERR_CUDA; }
        return XM_OK;
    }

    /* blocks [lo, hi) inflated behind the `left` bytes at the front of d_bam[s] (which holds them all) */
    int inflate_blocks(size_t lo, size_t hi, uint64_t left, std::string &err)
    {
        cudaStream_t st = c->be.st;
        const size_t nblk = hi - lo;
        if (!nblk) return XM_OK;
        int rc;
        if (host_mode) {
            /* 64 MiB of inflated bytes at a time through one host buffer: the host memory stays small whatever the window.
             * The upload runs on the copy streams: the move of the last window's tail to the front (on st) ends first. */
            if (cudaStreamSynchronize(st) != cudaSuccess) { err = "D2D copy failed"; return XM_ERR_CUDA; }
            for (size_t a = lo, b; a < hi; a = b) {
                uint64_t n = 0;
                for (b = a; b < hi && (b == a || n + blocks[b].out_len <= (64ull << 20)); ++b) n += blocks[b].out_len;
                if (!n) continue;                                  /* empty blocks only */
                if (h_piece.size() < n) h_piece.resize(n);
                std::string e;
                if (!bgzf_inflate(bam, blocks, a, b, h_piece.data() - blocks[a].out_off, host_threads(), e)) { err = "BAM input: " + e; return XM_ERR_IO; }
                const auto tu = std::chrono::steady_clock::now();
                if ((rc = upload_shard(c, c->d_bam[s].p + left + (blocks[a].out_off - blocks[lo].out_off), h_piece.data(), n))) { err = c->err; return rc; }
                c->bam_stats.upload_s += std::chrono::duration<double>(std::chrono::steady_clock::now() - tu).count();
            }
            return XM_OK;
        }
        const uint64_t c0 = blocks[lo].in_off, c1 = blocks[hi - 1].in_off + blocks[hi - 1].in_len;
        if ((rc = reserve_dev(c, c->d_bam_comp[s], c1 - c0 + 64)) || (rc = reserve_dev(c, c->d_bam_tab[s], nblk * sizeof(BgzfDev) + 16))) { err = c->err; return rc; }
        const auto tu = std::chrono::steady_clock::now();
        if ((rc = upload_shard(c, c->d_bam_comp[s].p, bam + c0, c1 - c0))) { err = c->err; return rc; }
        c->bam_stats.upload_s += std::chrono::duration<double>(std::chrono::steady_clock::now() - tu).count();
        std::vector<BgzfDev> tab(nblk);
        for (size_t k = 0; k < nblk; ++k) {
            const BgzfBlock &b = blocks[lo + k];
            tab[k].in_off = b.in_off - c0 + b.hdr_len;
            tab[k].in_len = b.in_len - b.hdr_len - 8;
            tab[k].out_off = left + (b.out_off - blocks[lo].out_off);
            tab[k].out_len = b.out_len;
            tab[k].crc = rd_u32(bam + b.in_off + b.in_len - 8);
            tab[k].pad = 0;
        }
        EventPair ev;
        cudaMemcpyAsync(c->d_bam_tab[s].p, tab.data(), nblk * sizeof(BgzfDev), cudaMemcpyHostToDevice, st);
        unsigned long long *d_status = (unsigned long long *)(c->d_bam_tab[s].p + nblk * sizeof(BgzfDev));
        const unsigned long long none = ~0ull;
        cudaMemcpyAsync(d_status, &none, 8, cudaMemcpyHostToDevice, st);
        cudaEventRecord(ev.a, st);
        k_bgzf_inflate<<<(unsigned)((nblk + INF_WARPS - 1) / INF_WARPS), INF_WARPS * 32, 0, st>>>(c->d_bam_comp[s].p, (const BgzfDev *)c->d_bam_tab[s].p,
                                                                                               (uint32_t)nblk, c->d_bam[s].p, d_status, 1);
        cudaEventRecord(ev.b, st);
        unsigned long long status = 0;
        cudaMemcpyAsync(&status, d_status, 8, cudaMemcpyDeviceToHost, st);
        if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) { err = "the BGZF inflate kernel failed"; return XM_ERR_CUDA; }
        if (status != ~0ull) { err = "BAM input: BGZF block does not inflate (corrupt data or CRC mismatch)"; return XM_ERR_IO; }
        c->bam_stats.inflate_ms += ev.ms();
        c->bam_stats.n_launches += 1;
        return XM_OK;
    }

    /* The record chain over d_bam[s][0, have_d) (xm_bamchain.h) and the text length of every record.  first: offset of a
     * known record start, or CHAIN_NONE (a rank's part of a file: the chain starts at the first guess, reported in *guess).
     * stop: only records that start before it are taken.  Sets n_rec, win_end (where the chain ended), sums. */
    int chain_records(uint64_t first, uint64_t stop, uint64_t *guess, std::string &err)
    {
        cudaStream_t st = c->be.st;
        DevBuf &D = c->d_bam[s];
        int rc;
        n_rec = 0; r_next = 0; win_end = 0; cut_off = 0;
        if (guess) *guess = CHAIN_NONE;
        const uint64_t SEG = bam_seg_bytes();
        const uint32_t n_seg = (uint32_t)((have_d + SEG - 1) / SEG);
        if (!n_seg) return XM_OK;
        if ((rc = reserve_dev(c, c->d_bam_seg[s], (uint64_t)(n_seg + 1) * (sizeof(ChainSeg) + 8) + 64))) { err = c->err; return rc; }
        ChainSeg *d_seg = (ChainSeg *)c->d_bam_seg[s].p, *d_one = d_seg + n_seg;
        uint64_t *d_base = (uint64_t *)(d_one + 1);
        if (!seg_valid) {
            k_bam_chain<<<(n_seg + 127) / 128, 128, 0, st>>>(D.p, have_d, SEG, first, n_seg, n_ref, nullptr, d_seg);
            seg0.resize(n_seg);
            cudaMemcpyAsync(seg0.data(), d_seg, (size_t)n_seg * sizeof(ChainSeg), cudaMemcpyDeviceToHost, st);
            if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) { err = "the BAM chain kernel failed"; return XM_ERR_CUDA; }
            c->bam_stats.n_launches += 1;
        }
        std::vector<ChainSeg> seg(seg0);                  /* the confirmation changes them; the guesses are kept for another try */
        std::vector<uint64_t> base(n_seg);
        if (first == CHAIN_NONE) {
            for (uint32_t k = 0; k < n_seg && first == CHAIN_NONE; ++k) first = seg[k].entry;
            if (first == CHAIN_NONE) { win_end = have_d; return XM_OK; }        /* no record starts in these bytes */
        }
        if (guess) *guess = first;
        auto repair = [&](uint32_t k, uint64_t entry, uint64_t hi) {
            ChainSeg r;
            k_bam_chain_one<<<1, 32, 0, st>>>(D.p, have_d, (uint64_t)k * SEG, hi, entry, n_ref, d_one);
            cudaMemcpyAsync(&r, d_one, sizeof r, cudaMemcpyDeviceToHost, st);
            if (cudaStreamSynchronize(st) != cudaSuccess) { r.entry = entry; r.exit = entry; r.count = 0; r.flag = CHAIN_CORRUPT; }
            return r;
        };
        uint64_t end = 0, nr = 0;
        uint32_t nrep = 0;
        if (!chain_confirm(seg.data(), base.data(), n_seg, SEG, first, have_d, std::min(stop, have_d), repair, end, nr, nrep)) { err = "corrupt BAM record"; return XM_ERR_IO; }
        c->bam_stats.chain_repairs += nrep;
        c->bam_stats.n_launches += nrep;
        n_rec = nr; win_end = end;
        if (!n_rec) return XM_OK;
        const uint64_t nb = (n_rec + 1023) / 1024;
        if ((rc = reserve_dev(c, c->d_bam_rec[s], n_rec * 8)) || (rc = reserve_dev(c, c->d_bam_len[s], n_rec * 8 + 16)) ||
            (rc = reserve_dev(c, c->d_bam_sum[s], nb * 8 + 16))) { err = c->err; return rc; }
        cudaMemcpyAsync(d_seg, seg.data(), (size_t)n_seg * sizeof(ChainSeg), cudaMemcpyHostToDevice, st);
        cudaMemcpyAsync(d_base, base.data(), (size_t)n_seg * 8, cudaMemcpyHostToDevice, st);
        k_bam_chain_emit<<<(n_seg + 127) / 128, 128, 0, st>>>(D.p, have_d, SEG, n_seg, d_seg, d_base, (uint64_t *)c->d_bam_rec[s].p);
        unsigned long long *d_err = (unsigned long long *)(c->d_bam_sum[s].p + nb * 8);
        const unsigned long long no_err = BAM_NO_ERROR;
        cudaMemcpyAsync(d_err, &no_err, 8, cudaMemcpyHostToDevice, st);
        BamDev B = dev_view(0, n_rec);
        uint32_t *d_len = (uint32_t *)c->d_bam_len[s].p, *d_loff = d_len + n_rec + (n_rec & 1);
        EventPair rv;
        cudaEventRecord(rv.a, st);
        k_bam_len<<<(unsigned)((n_rec + 255) / 256), 256, 0, st>>>(B, d_len, d_err);
        k_bam_scan_blocks<<<(unsigned)nb, 1024, 0, st>>>(d_len, n_rec, d_loff, (unsigned long long *)c->d_bam_sum[s].p);
        cudaEventRecord(rv.b, st);
        sums.assign(nb + 1, 0);
        cudaMemcpyAsync(sums.data(), c->d_bam_sum[s].p, (nb + 1) * 8, cudaMemcpyDeviceToHost, st);
        if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) { err = "BAM length kernels failed"; return XM_ERR_CUDA; }
        c->bam_stats.render_ms += rv.ms();
        c->bam_stats.n_launches += 4;
        if (sums[nb] != BAM_NO_ERROR) { err = "corrupt BAM record"; return XM_ERR_IO; }
        c->bam_stats.records += n_rec;
        return XM_OK;
    }

    /* the next window: what is left of the last one moves to the front, the next blocks are inflated behind it, the chain is
     * followed and the text length of every record is found */
    int load_window(std::string &err)
    {
        cudaStream_t st = c->be.st;
        const auto t0 = std::chrono::steady_clock::now();
        int rc;
        const uint64_t left = have_d - win_end;
        size_t last = blk;
        uint64_t add = 0;
        const uint64_t W = bam_window_bytes();
        while (last < blocks.size() && (last == blk || add + blocks[last].out_len <= W)) add += blocks[last++].out_len;
        DevBuf &D = c->d_bam[s];
        if (left && left + add + 64 <= D.cap && left <= win_end) {
            cudaMemcpyAsync(D.p, D.p + win_end, left, cudaMemcpyDeviceToDevice, st);
        } else {
            uint8_t *tmp = nullptr;
            if (left) {
                if (cudaMalloc((void **)&tmp, left) != cudaSuccess) { cudaGetLastError(); err = "cudaMalloc: out of memory"; return XM_ERR_NOMEM; }
                cudaMemcpyAsync(tmp, D.p + win_end, left, cudaMemcpyDeviceToDevice, st);
                cudaStreamSynchronize(st);
            }
            if ((rc = reserve_dev(c, D, std::max<uint64_t>(left + add + 64, std::min<uint64_t>(W, inflated_total) + 64)))) { if (tmp) cudaFree(tmp); err = c->err; return rc; }
            if (left) { cudaMemcpyAsync(D.p, tmp, left, cudaMemcpyDeviceToDevice, st); cudaStreamSynchronize(st); cudaFree(tmp); }
        }
        if ((rc = inflate_blocks(blk, last, left, err))) return rc;
        have_d = left + add;
        blk = last;
        c->bam_stats.inflated_bytes += add;
        n_rec = 0; r_next = 0; win_end = 0; cut_off = 0;
        seg_valid = false;
        uint64_t first = 0;
        if (skip) {
            if (skip >= have_d) {            /* nothing but header so far */
                skip -= have_d; have_d = 0;
                c->bam_stats.inflate_s += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
                return XM_OK;
            }
            first = skip; skip = 0;
        }
        if ((rc = chain_records(first, have_d, nullptr, err))) return rc;
        if (blk == blocks.size() && win_end != have_d) { err = "truncated BAM record at the end of the file"; return XM_ERR_IO; }
        c->bam_stats.inflate_s += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        return XM_OK;
    }

    /* ---- a rank's part of the file, for the walk across GPUs ------------------------------------------------------------
     * Rank r of W takes the BGZF blocks that START in bytes [len r / W, len (r + 1) / W) of the file and, of the records,
     * those that start in these blocks' inflated bytes [so0, so1).  It inflates its blocks and as many of the next ones as
     * its last record reaches into (every rank maps the whole file: nothing is exchanged but two numbers per rank).  */
    size_t sb0 = 0, sb1 = 0, sbx = 0;
    uint64_t so0 = 0, so1 = 0;
    int shard_open(int rank, int world, uint64_t &guess_abs, uint64_t &exit_abs, std::string &err)
    {
        auto first_block_at = [&](uint64_t byte) {
            size_t lo = 0, hi = blocks.size();
            while (lo < hi) { const size_t mid = (lo + hi) / 2; if (blocks[mid].in_off < byte) lo = mid + 1; else hi = mid; }
            return lo;
        };
        sb0 = rank == 0 ? 0 : first_block_at(bam_len / (uint64_t)world * (uint64_t)rank);
        sb1 = rank + 1 == world ? blocks.size() : first_block_at(bam_len / (uint64_t)world * (uint64_t)(rank + 1));
        so0 = sb0 < blocks.size() ? blocks[sb0].out_off : inflated_total;
        so1 = sb1 < blocks.size() ? blocks[sb1].out_off : inflated_total;
        sbx = sb1;
        return shard_chain(CHAIN_NONE, guess_abs, exit_abs, err);
    }
    /* (Re)do the chain of the rank's part.  entry_abs: the true start of its first record (the exit the rank before
     * reports), or CHAIN_NONE for the first attempt: rank 0 knows its start, the others guess.  exit_abs: the first record
     * start at or behind so1 -- the next rank's true entry. */
    int shard_chain(uint64_t entry_abs, uint64_t &guess_abs, uint64_t &exit_abs, std::string &err)
    {
        const uint64_t data0 = std::max(so0, skip_abs);                       /* records start behind the header */
        guess_abs = exit_abs = CHAIN_NONE;
        if (so1 <= data0 || sb0 >= sb1) { n_rec = 0; have_d = 0; return XM_OK; }          /* header only, or no blocks: passes the entry on */
        int rc;
        for (size_t extra = 2;; extra *= 4) {
            const size_t want = std::min(blocks.size(), sb1 + extra);
            if (want != sbx || !have_d) {
                uint64_t add = 0;
                for (size_t k = sb0; k < want; ++k) add += blocks[k].out_len;
                if ((rc = reserve_dev(c, c->d_bam[s], add + 64))) { err = c->err; return rc; }
                if ((rc = inflate_blocks(sb0, want, 0, err))) return rc;
                c->bam_stats.inflated_bytes += add;
                have_d = add; sbx = want; seg_valid = false;
            }
            uint64_t first = entry_abs != CHAIN_NONE ? entry_abs - so0 : (so0 < skip_abs ? skip_abs - so0 : CHAIN_NONE);
            if (first != CHAIN_NONE && first >= so1 - so0) { n_rec = 0; guess_abs = entry_abs; exit_abs = entry_abs; return XM_OK; }     /* one record covers the whole part */
            uint64_t guess = CHAIN_NONE;
            if ((rc = chain_records(first, so1 - so0, &guess, err))) return rc;
            seg_valid = true;
            guess_abs = guess == CHAIN_NONE ? CHAIN_NONE : so0 + guess;
            if (guess == CHAIN_NONE) { exit_abs = CHAIN_NONE; return XM_OK; }     /* nothing that looks like a record: passes the entry on */
            if (win_end >= so1 - so0 || (sbx == blocks.size() && win_end == have_d)) { exit_abs = so0 + win_end; return XM_OK; }
            if (sbx == blocks.size()) { err = "truncated BAM record at the end of the file"; return XM_ERR_IO; }
            /* the last record of the part runs past the blocks inflated so far: take more */
        }
    }
    /* the part's records as SAM text at T.p + front_room (room behind it as well) */
    int shard_text(uint64_t front_room, uint64_t back_room, DevBuf &T, uint64_t &text_len, std::string &err)
    {
        text_len = n_rec ? window_text_left() : 0;
        int rc;
        if ((rc = reserve_dev(c, T, front_room + text_len + back_room + 64))) { err = c->err; return rc; }
        uint64_t off = 0;
        while (r_next < n_rec) {
            uint64_t n = 0;
            if ((rc = render_window(T.p + front_room + off, text_len - off, n, err))) return rc;
            if (!n) { err = "BAM shard rendering made no progress"; return XM_ERR_IO; }
            off += n;
        }
        return XM_OK;
    }

    BamDev dev_view(uint64_t r0, uint64_t n) const
    {
        BamDev B;
        B.data = c->d_bam[s].p; B.rec = (const uint64_t *)c->d_bam_rec[s].p + r0; B.n = n;
        B.ref_off = (const uint32_t *)c->d_bam_ref[s].p; B.ref_names = d_names; B.n_ref = n_ref;
        return B;
    }
    /* text bytes the rest of the window renders to (0: the window is spent) */
    uint64_t window_text_left() const
    {
        uint64_t t = 0;
        if (r_next == n_rec) return 0;
        for (uint64_t g = r_next / 1024, nb = (n_rec + 1023) / 1024; g < nb; ++g) t += sums[g];
        return t - cut_off;
    }

    /* Up to max_bytes of text of the current window's records from r_next on into dev_dst (r_next < n_rec); n_out = 0:
     * not even the next record fits.  Whole groups of 1024 records while they fit, then the records of the next group
     * that still do (its offsets are read back: 4 KiB).  cut_off: text bytes of r_next's group that earlier calls
     * rendered. */
    int render_window(uint8_t *dev_dst, uint64_t max_bytes, uint64_t &n_out, std::string &err)
    {
        n_out = 0;
        cudaStream_t st = c->be.st;
        const uint64_t g0 = r_next >> 10, nbw = (n_rec + 1023) / 1024;
        const uint32_t *d_len = (const uint32_t *)c->d_bam_len[s].p, *d_loff = d_len + n_rec + (n_rec & 1);
        uint64_t g = g0, bytes = 0, r_end = r_next, cut_end = cut_off;
        while (g < nbw) {
            const uint64_t rem = sums[g] - (g == g0 ? cut_off : 0);
            if (bytes + rem > max_bytes) break;
            bytes += rem; ++g;
            r_end = std::min(n_rec, g * 1024); cut_end = 0;
        }
        if (g < nbw && bytes < max_bytes) {
            const uint64_t lo = g * 1024, cnt_g = std::min<uint64_t>(1024, n_rec - lo);
            uint32_t loff[1024];
            cudaMemcpyAsync(loff, d_loff + lo, cnt_g * 4, cudaMemcpyDeviceToHost, st);
            if (cudaStreamSynchronize(st) != cudaSuccess) { err = "D2H copy failed"; return XM_ERR_CUDA; }
            const uint64_t start = g == g0 ? cut_off : 0, room = max_bytes - bytes;
            uint64_t j = r_end - lo;                                   /* records [lo + j0, lo + j) of this group are taken */
            while (j + 1 < cnt_g && loff[j + 1] - start <= room) ++j;  /* loff[j + 1] - start: text of the records up to j */
            if (lo + j > r_end) { bytes += loff[j] - start; r_end = lo + j; cut_end = loff[j]; }
        }
        if (r_end == r_next) return XM_OK;
        const uint64_t cnt = r_end - r_next, ng = ((r_end - 1) >> 10) - g0 + 1;
        std::vector<unsigned long long> bases(ng);
        unsigned long long run = 0ull - cut_off;                       /* wraps: the first group's base lies before dev_dst */
        for (uint64_t k = 0; k < ng; ++k) { bases[k] = run; run += sums[g0 + k]; }
        cudaMemcpyAsync(c->d_bam_sum[s].p, bases.data(), bases.size() * 8, cudaMemcpyHostToDevice, st);
        EventPair ev;
        cudaEventRecord(ev.a, st);
        k_bam_render<<<(unsigned)((cnt * 32 + 255) / 256), 256, 0, st>>>(dev_view(0, n_rec), r_next, cnt, d_loff, (const unsigned long long *)c->d_bam_sum[s].p, dev_dst);
        cudaEventRecord(ev.b, st);
        if (cudaStreamSynchronize(st) != cudaSuccess || cudaGetLastError() != cudaSuccess) { err = "BAM render kernel failed"; return XM_ERR_CUDA; }
        c->bam_stats.render_ms += ev.ms();
        c->bam_stats.text_bytes += bytes;
        c->bam_stats.n_launches += 1;
        cut_off = cut_end;
        r_next = r_end;
        n_out = bytes;
        return XM_OK;
    }

    /* the walk's source: windows are loaded while the current one is spent */
    int next(uint8_t *dev_dst, uint64_t max_bytes, uint64_t &n_out, bool &final, std::string &err) override
    {
        n_out = 0; final = false;
        if (max_bytes == 0) return XM_OK;
        int rc;
        while (r_next == n_rec) {
            if (blk == blocks.size()) { final = true; return XM_OK; }
            if ((rc = load_window(err))) return rc;
        }
        if ((rc = render_window(dev_dst, max_bytes, n_out, err))) return rc;
        if (!n_out && max_bytes >= full_cap) { err = "a BAM record renders to more text than a staging step holds"; return XM_ERR_UNSUPPORTED; }
        final = r_next == n_rec && blk == blocks.size();      /* n_out = 0 and not final: the walk buffer is full of carried records */
        return XM_OK;
    }
};

/* one BAM file as SAM text in device memory (slot s): the producer's windows rendered one behind the other */
static int bam_to_device_text(xm_ctx *c, const void *bam, uint64_t len, int s, uint8_t **d_text, uint64_t *text_len)
{
    *d_text = nullptr; *text_len = 0;
    BamProducer p;
    p.c = c; p.s = s; p.bam = (const uint8_t *)bam; p.bam_len = len;
    std::string err;
    int rc = p.open(err);
    if (rc) return fail(c, rc, err);
    DevBuf &T = c->d_bam_text[s];
    uint64_t off = 0;
    for (;;) {
        while (p.r_next == p.n_rec && p.blk < p.blocks.size()) if ((rc = p.load_window(err))) return fail(c, rc, err);
        const uint64_t want = p.window_text_left();
        if (!want) break;
        if (off + want > T.cap || !T.p) {                   /* grow, keeping what is rendered */
            uint8_t *np_ = nullptr;
            const uint64_t cap = std::max<uint64_t>(off + want, T.cap * 2);
            if (cudaMalloc((void **)&np_, cap + 64) != cudaSuccess) { cudaGetLastError(); return fail(c, XM_ERR_NOMEM, "cudaMalloc: out of memory"); }
            if (off) { cudaMemcpyAsync(np_, T.p, off, cudaMemcpyDeviceToDevice, c->be.st); cudaStreamSynchronize(c->be.st); }
            if (T.p) cudaFree(T.p);
            T.p = np_; T.cap = cap;
        }
        uint64_t n = 0;                                     /* offered the whole rest of the window: renders all of it */
        if ((rc = p.render_window(T.p + off, want, n, err))) return fail(c, rc, err);
        off += n;
    }
    if (!T.p && (rc = reserve_dev(c, T, 64))) return rc;
    *d_text = T.p;
    *text_len = off;
    return XM_OK;
}

static int classify_bam(xm_ctx *c, const void *prim_bam, uint64_t prim_len, const void *sec_bam, uint64_t sec_len,
                        const int *out_fds, const xm_opts *opts, uint32_t out_flags, xm_result *res)
{
    cudaSetDevice(c->device);
    memset(res, 0, sizeof *res);
    BamProducer prod[2];
    HostIn in[2];
    const void *src[2] = {prim_bam, sec_bam};
    const uint64_t len[2] = {prim_len, sec_len};
    const uint32_t launches0 = c->bam_stats.n_launches;
    for (int s = 0; s < 2; ++s) {
        prod[s].c = c; prod[s].s = s; prod[s].bam = (const uint8_t *)src[s]; prod[s].bam_len = len[s];
        std::string err;
        const int rc = prod[s].open(err);
        if (rc) return res->status = fail(c, rc, err);
        in[s].prod = &prod[s];
        in[s].len = prod[s].inflated_total * 3 + 4096;  /* an estimate of the text: sizes the staging steps of small files */
    }
    const uint64_t step = std::max<uint64_t>(std::min<uint64_t>(chunk_bytes(), std::max(in[0].len, in[1].len) + 64), 64);     /* stream_walk's chunk */
    prod[0].full_cap = prod[1].full_cap = step;
    const int rc = stream_walk(c, in, out_fds, opts, res, out_flags);
    res->n_launches += c->bam_stats.n_launches - launches0;
    return rc;
}

int xm_classify_bam_host(xm_ctx *c, const void *prim_bam, uint64_t prim_len, const void *sec_bam, uint64_t sec_len,
                         const xm_opts *opts, xm_result *res)
{
    if (!c || !opts || !res || !prim_bam || !sec_bam) return XM_ERR_ARG;
    return classify_bam(c, prim_bam, prim_len, sec_bam, sec_len, nullptr, opts, 0, res);
}

int xm_classify_bam_fds(xm_ctx *c, const void *prim_bam, uint64_t prim_len, const void *sec_bam, uint64_t sec_len,
                        const int out_fds[6], const xm_opts *opts, uint32_t out_flags, xm_result *res)
{
    if (!c || !opts || !res || !prim_bam || !sec_bam || !out_fds) return XM_ERR_ARG;
    return classify_bam(c, prim_bam, prim_len, sec_bam, sec_len, out_fds, opts, out_flags, res);
}

/* ---- a rank's part of a BAM file as SAM text on the device (the walk across GPUs on BAM input) ------------------------- */
static void bam_shard_free(xm_ctx *c)
{
    for (auto &p : c->bam_shard) { delete (BamProducer *)p; p = nullptr; }
}

int xm_bam_shard_open(xm_ctx *c, int stream, const void *bam, uint64_t len, int rank, int world, uint64_t *guess, uint64_t *exit_off)
{
    if (!c || stream < 0 || stream > 1 || !bam || rank < 0 || world < 1 || rank >= world || !guess || !exit_off) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    delete (BamProducer *)c->bam_shard[stream];
    BamProducer *p = new BamProducer;
    c->bam_shard[stream] = p;
    p->c = c; p->s = stream; p->bam = (const uint8_t *)bam; p->bam_len = len;
    std::string err;
    int rc = p->open(err);
    if (rc) return fail(c, rc, err);
    if (p->host_mode) return fail(c, XM_ERR_UNSUPPORTED, "the sharded BAM walk inflates on the device (unset XM_BAM_INFLATE)");
    if ((rc = p->shard_open(rank, world, *guess, *exit_off, err))) return fail(c, rc, err);
    return XM_OK;
}

int xm_bam_shard_chain(xm_ctx *c, int stream, uint64_t entry, uint64_t *exit_off)
{
    if (!c || stream < 0 || stream > 1 || !c->bam_shard[stream] || !exit_off) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    BamProducer *p = (BamProducer *)c->bam_shard[stream];
    std::string err;
    uint64_t guess = 0;
    const int rc = p->shard_chain(entry, guess, *exit_off, err);
    if (rc) return fail(c, rc, err);
    return XM_OK;
}

int xm_bam_shard_text(xm_ctx *c, int stream, uint64_t front_room, uint64_t back_room, void **d_text, uint64_t *text_len)
{
    if (!c || stream < 0 || stream > 1 || !c->bam_shard[stream] || !d_text || !text_len) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    BamProducer *p = (BamProducer *)c->bam_shard[stream];
    std::string err;
    front_room = (front_room + 15) & ~15ull;
    const int rc = p->shard_text(front_room, back_room, c->d_bam_text[stream], *text_len, err);
    if (rc) return fail(c, rc, err);
    *d_text = c->d_bam_text[stream].p + front_room;
    return XM_OK;
}

int xm_get_walk_kernels(xm_ctx *c, uint32_t *mask)
{
    if (!c || !mask) return XM_ERR_ARG;
    *mask = c->scratch.last_kernels;
    return XM_OK;
}

int xm_bam_get_stats(xm_ctx *c, xm_bam_stats *out, int reset)
{
    if (!c || !out) return XM_ERR_ARG;
    *out = c->bam_stats;
    if (reset) c->bam_stats = xm_bam_stats{};
    return XM_OK;
}

/* ---- index pass of the sharded walk (xm_walk.h index_resident) ---------------------------- */
int xm_count_device(xm_ctx *c, const void *d_buf, uint64_t len, int skip_repeated, xm_shard_info *info)
{
    if (!c || !info) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    std::string msg;
    const int rc = index_resident(c->be, c->scratch, StreamBuf{(const uint8_t *)d_buf, len}, skip_repeated != 0, c->debug, 0, nullptr, nullptr, info, msg);
    c->err = msg;
    return rc;
}

int xm_locate_device(xm_ctx *c, const void *d_buf, uint64_t len, int skip_repeated, uint32_t n_queries,
                     const uint64_t *record_index, uint64_t *byte_offset)
{
    if (!c || (n_queries && (!record_index || !byte_offset))) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    xm_shard_info info;
    std::string msg;
    const int rc = index_resident(c->be, c->scratch, StreamBuf{(const uint8_t *)d_buf, len}, skip_repeated != 0, c->debug, n_queries, record_index, byte_offset, &info, msg);
    c->err = msg;
    return rc;
}

/* ---- the walk across GPUs (xm_shard.h) ------------------------------------------------------------------------ */
int xm_comm_unique_id(void *id128)
{
    if (!id128) return XM_ERR_ARG;
    NcclApi &A = nccl_api();
    if (!A.load()) { g_create_error = A.err; return XM_ERR_CUDA; }
    NcclId id;
    const int r = A.GetUniqueId(&id);
    if (r) { g_create_error = std::string("ncclGetUniqueId: ") + A.GetErrorString(r); return XM_ERR_CUDA; }
    memcpy(id128, &id, sizeof id);
    return XM_OK;
}

int xm_comm_init_rank(xm_ctx *c, int nranks, int rank, const void *id128)
{
    if (!c || nranks < 1 || rank < 0 || rank >= nranks || (nranks > 1 && !id128)) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    xm_comm_destroy(c);
    c->comm.nranks = nranks; c->comm.my = rank; c->comm.st = c->be.st;
    if (nranks == 1) return XM_OK;
    NcclApi &A = nccl_api();
    if (!A.load()) return fail(c, XM_ERR_CUDA, A.err);
    NcclId id;
    memcpy(&id, id128, sizeof id);
    const int r = A.CommInitRank(&c->comm.comm, nranks, id, rank);
    if (r) { c->comm.comm = nullptr; c->comm.nranks = 1; c->comm.my = 0; return fail(c, XM_ERR_CUDA, std::string("ncclCommInitRank: ") + A.GetErrorString(r)); }
    return XM_OK;
}

int xm_comm_destroy(xm_ctx *c)
{
    if (!c) return XM_ERR_ARG;
    if (c->comm.comm) { cudaStreamSynchronize(c->be.st); nccl_api().CommDestroy(c->comm.comm); c->comm.comm = nullptr; }
    if (c->comm.d_stage) { cudaFree(c->comm.d_stage); c->comm.d_stage = nullptr; c->comm.stage_cap = 0; }
    c->comm.nranks = 1; c->comm.my = 0;
    return XM_OK;
}

int xm_comm_barrier(xm_ctx *c)
{
    if (!c) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    if (cudaStreamSynchronize(c->be.st) != cudaSuccess) return fail(c, XM_ERR_CUDA, "stream synchronize failed");
    uint64_t one = 1;
    std::vector<uint64_t> all((size_t)c->comm.nranks);
    if (c->comm.all_gather(&one, all.data(), 8)) return fail(c, XM_ERR_CUDA, c->comm.err);
    return XM_OK;
}

int xm_comm_allreduce_f64(xm_ctx *c, double *values, int n, int op)
{
    if (!c || !values || n < 0) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    std::vector<double> all((size_t)n * (size_t)c->comm.nranks);
    if (n && c->comm.all_gather(values, all.data(), (size_t)n * 8)) return fail(c, XM_ERR_CUDA, c->comm.err);
    for (int k = 0; k < n; ++k) {
        double v = all[(size_t)k];
        for (int q = 1; q < c->comm.nranks; ++q) { const double w = all[(size_t)q * (size_t)n + (size_t)k]; v = op == 1 ? std::max(v, w) : v + w; }
        values[k] = v;
    }
    return XM_OK;
}

int xm_classify_sharded_device(xm_ctx *c, void *d_prim, uint64_t prim_len, void *d_sec, uint64_t sec_len, uint64_t front_room,
                               uint64_t back_room, const xm_opts *opts, void *const d_out[6], const uint64_t out_cap[6],
                               xm_result *res, xm_shard_stats *stats)
{
    if (!c || !opts || !res || !stats) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    c->comm.st = c->be.st;
    ShardBuf in[2] = {{(uint8_t *)d_prim, prim_len, front_room, back_room}, {(uint8_t *)d_sec, sec_len, front_room, back_room}};
    uint8_t *o6[6];
    uint64_t cap6[6];
    for (int b = 0; b < 6; ++b) { o6[b] = d_out ? (uint8_t *)d_out[b] : nullptr; cap6[b] = (out_cap && o6[b]) ? out_cap[b] : 0; }
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0, c->be.st);
    std::string msg;
    int rc = walk_sharded(c->be, c->comm, c->shard, in, *opts, o6, cap6, c->debug, res, stats, msg);
    cudaEventRecord(e1, c->be.st);
    cudaEventSynchronize(e1);
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    res->ms_total = ms;                     /* device time of the whole call: alignment, scans, exchanges, emit */
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    c->err = msg;
    if (rc == XM_SHARD_DECLINED) { rc = XM_ERR_UNSUPPORTED; c->err = "the sharded device walk handles clean SAM only: " + msg; res->status = rc; }
    return rc;
}

/* one memcpy by several threads (a single core moves ~10 GB/s, less than the PCIe link takes) */
static void memcpy_threads(uint8_t *dst, const uint8_t *src, size_t n, int threads)
{
    if (threads <= 1 || n < (8u << 20)) { memcpy(dst, src, n); return; }
    const size_t part = ((n + (size_t)threads - 1) / (size_t)threads + 4095) & ~(size_t)4095;
    std::vector<std::thread> pool;
    for (size_t at = part; at < n; at += part) pool.emplace_back([=]() { memcpy(dst + at, src + at, std::min(part, n - at)); });
    memcpy(dst, src, std::min(part, n));
    for (auto &t : pool) t.join();
}

/* pageable host memory -> device through two pinned blocks, the memcpy of one overlapping the H2D of the other */
static int upload_shard(xm_ctx *c, uint8_t *d_dst, const uint8_t *src, uint64_t n)
{
    const uint64_t blk = 64ull << 20;
    const int nt = std::max(1, std::min(8, host_threads() / 2));
    int rc;
    for (int k = 0; k < 2; ++k) if ((rc = reserve_host(c, c->h_stage[k], std::min<uint64_t>(blk, n ? n : 1)))) return rc;
    cudaEvent_t ev[2];
    cudaEventCreate(&ev[0]); cudaEventCreate(&ev[1]);
    uint64_t done = 0;
    for (int k = 0; done < n; ++k) {
        const int b = k & 1;
        const uint64_t m = std::min<uint64_t>(std::min<uint64_t>(blk, c->h_stage[b].cap), n - done);
        if (k >= 2) cudaEventSynchronize(ev[b]);
        memcpy_threads(c->h_stage[b].p, src + done, (size_t)m, nt);
        cudaMemcpyAsync(d_dst + done, c->h_stage[b].p, (size_t)m, cudaMemcpyHostToDevice, c->copy_st[b]);
        cudaEventRecord(ev[b], c->copy_st[b]);
        done += m;
    }
    cudaError_t e = cudaStreamSynchronize(c->copy_st[0]);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->copy_st[1]);
    cudaEventDestroy(ev[0]); cudaEventDestroy(ev[1]);
    if (e != cudaSuccess) return cuda_fail(c, e, "H2D copy");
    return XM_OK;
}

int xm_classify_sharded_host(xm_ctx *c, const void *prim, uint64_t prim_len, const void *sec, uint64_t sec_len,
                             const xm_opts *opts, xm_result *res, xm_shard_stats *stats)
{
    if (!c || !opts || !res || !stats) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    c->comm.st = c->be.st;
    recycle_bins(c);
    uint64_t room = 1ull << 20;
    if (const char *e = getenv("XM_SHARD_ROOM_MB")) { const long long v = atoll(e); if (v > 0) room = (uint64_t)v << 20; }
    const void *src[2] = {prim, sec};
    const uint64_t len[2] = {prim_len, sec_len};
    ShardBuf in[2];
    int rc;
    for (int s = 0; s < 2; ++s) {
        if ((rc = reserve_dev(c, c->d_shard[s], len[s] + 2 * room + 64))) return res->status = rc;
        in[s] = ShardBuf{c->d_shard[s].p + room, len[s], room, room};
        if (len[s] && (rc = upload_shard(c, in[s].p, (const uint8_t *)src[s], len[s]))) return res->status = rc;
    }
    uint8_t *none[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    uint64_t nocap[6] = {0, 0, 0, 0, 0, 0};
    auto alloc_out = [&](const uint64_t *want, uint8_t **ptr, uint64_t *cap) -> int {
        for (int b = 0; b < 6; ++b) {
            if (reserve_dev(c, c->d_out[0][b], want[b] + 16)) return 1;
            ptr[b] = c->d_out[0][b].p; cap[b] = want[b];
        }
        return 0;
    };
    struct Alloc {
        decltype(alloc_out) &f;
        int operator()(const uint64_t *w, uint8_t **p, uint64_t *cp) const { return f(w, p, cp); }
        explicit operator bool() const { return true; }
    } al{alloc_out};
    std::string msg;
    rc = walk_sharded(c->be, c->comm, c->shard, in, *opts, none, nocap, c->debug, res, stats, msg, al);
    c->err = msg;
    if (rc == XM_SHARD_DECLINED) {
        /* some rank's shard needs the exact kernels: every rank sends its (untouched) bytes to rank 0, which walks the
         * whole streams alone; the other ranks contribute empty bins */
        const int W = c->comm.size(), r = c->comm.rank();
        std::vector<uint64_t> mine = {len[0], len[1]}, all((size_t)2 * (size_t)W);
        if (c->comm.all_gather(mine.data(), all.data(), 16)) return res->status = fail(c, XM_ERR_CUDA, c->comm.err);
        for (int s = 0; s < 2; ++s) if (len[s] && (rc = upload_shard(c, in[s].p, (const uint8_t *)src[s], len[s]))) return res->status = rc;
        uint64_t total[2] = {0, 0};
        for (int q = 0; q < W; ++q) { total[0] += all[(size_t)2 * q]; total[1] += all[(size_t)2 * q + 1]; }
        DevBuf whole[2];
        int alloc_rc = XM_OK;
        if (r == 0) for (int s = 0; s < 2; ++s) if (!alloc_rc) alloc_rc = reserve_dev(c, whole[s], total[s] + 64);
        std::vector<uint64_t> ok = {(uint64_t)alloc_rc}, allok((size_t)W);
        c->comm.all_gather(ok.data(), allok.data(), 8);
        if (allok[0]) { for (auto &w : whole) if (w.p) cudaFree(w.p); return res->status = fail(c, XM_ERR_NOMEM, "rank 0 cannot hold the whole streams for the exact walk"); }
        std::vector<Xfer> sends, recvs;
        for (int s = 0; s < 2; ++s) {
            if (r > 0 && len[s]) sends.push_back(Xfer{0, in[s].p, len[s]});
            if (r == 0) {
                uint64_t at = len[s];
                if (len[s]) cudaMemcpyAsync(whole[s].p, in[s].p, len[s], cudaMemcpyDeviceToDevice, c->be.st);
                for (int q = 1; q < W; ++q) { const uint64_t n = all[(size_t)2 * q + s]; if (n) recvs.push_back(Xfer{q, whole[s].p + at, n}); at += n; }
            }
        }
        if ((!sends.empty() || !recvs.empty()) && c->comm.exchange(sends.data(), (int)sends.size(), recvs.data(), (int)recvs.size())) {
            for (auto &w : whole) if (w.p) cudaFree(w.p);
            return res->status = fail(c, XM_ERR_CUDA, c->comm.err);
        }
        xm_result rr;
        memset(&rr, 0, sizeof rr);
        int wrc = XM_OK;
        std::string wmsg;
        if (r == 0) {
            xm_opts o = *opts;
            o.skip_repeated &= 1;
            uint8_t *no[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
            uint64_t cap[6] = {0, 0, 0, 0, 0, 0};
            xm_result dry;
            wrc = walk_resident(c->be, c->scratch, StreamBuf{whole[0].p, total[0]}, StreamBuf{whole[1].p, total[1]}, o, no, cap, c->debug, &dry, wmsg);
            if (wrc != XM_ERR_CUDA && wrc != XM_ERR_NOMEM) {
                uint8_t *outs[6];
                for (int b = 0; b < 6; ++b) {
                    cap[b] = ((o.enabled_bins >> b) & 1u) ? dry.out_len[b] : 0;
                    if (reserve_dev(c, c->d_out[0][b], cap[b] + 16)) wrc = XM_ERR_NOMEM;
                    outs[b] = c->d_out[0][b].p;
                }
                if (wrc != XM_ERR_NOMEM) wrc = walk_resident(c->be, c->scratch, StreamBuf{whole[0].p, total[0]}, StreamBuf{whole[1].p, total[1]}, o, outs, cap, c->debug, &rr, wmsg);
            }
        }
        for (auto &w : whole) if (w.p) cudaFree(w.p);
        /* rank 0's result is everybody's */
        std::vector<uint64_t> g((size_t)4 + 6 + 36, 0), allg(g.size() * (size_t)W);
        if (r == 0) {
            g[0] = (uint64_t)wrc; g[1] = rr.n_records; g[2] = rr.err_record; g[3] = (uint64_t)(int64_t)rr.err_stream;
            for (int b = 0; b < 6; ++b) g[(size_t)4 + b] = rr.out_len[b];
            for (int k = 0; k < 36; ++k) g[(size_t)10 + k] = rr.counts[k];
        }
        if (c->comm.all_gather(g.data(), allg.data(), g.size() * 8)) return res->status = fail(c, XM_ERR_CUDA, c->comm.err);
        memset(res, 0, sizeof *res);
        memset(stats, 0, sizeof *stats);
        res->status = (int32_t)allg[0]; res->n_records = allg[1]; res->err_record = allg[2]; res->err_stream = (int32_t)(int64_t)allg[3];
        for (int k = 0; k < 36; ++k) res->counts[k] = allg[(size_t)10 + k];
        for (int b = 0; b < 6; ++b) { stats->out_total[b] = allg[(size_t)4 + b]; stats->out_offset[b] = r == 0 ? 0 : allg[(size_t)4 + b]; res->out_len[b] = r == 0 ? allg[(size_t)4 + b] : 0; }
        stats->n_records_total = allg[1]; stats->rec_lo = 0; stats->rec_hi = r == 0 ? allg[1] : 0;
        stats->first_bad_rank = allg[0] ? 0 : -1;
        rc = (int)allg[0];
        c->err = r == 0 ? wmsg : (rc ? "the exact walk on rank 0 failed" : "");
        if (rc == XM_ERR_CUDA || rc == XM_ERR_NOMEM) return rc;
    } else if (rc == XM_ERR_CUDA || rc == XM_ERR_NOMEM || rc == XM_ERR_ARG) return rc;
    /* this rank's bins back to host blocks */
    uint64_t biggest = 4096;
    for (int b = 0; b < 6; ++b) biggest = std::max<uint64_t>(biggest, res->out_len[b]);
    c->block_bytes = std::min<uint64_t>(biggest, 256ull << 20);
    for (int b = 0; b < 6; ++b)
        if (((opts->enabled_bins >> b) & 1u) && res->out_len[b]) { const int r2 = bin_append_d2h(c, b, c->d_out[0][b].p, res->out_len[b]); if (r2) return r2; }
    if (cudaStreamSynchronize(c->dl) != cudaSuccess) return fail(c, XM_ERR_CUDA, "D2H copy failed");
    return rc;
}

int xm_copy_ceiling(xm_ctx *c, uint64_t h2d_bytes, uint64_t d2h_bytes, int reps, float *ms)
{
    if (!c || !ms || reps < 1) return XM_ERR_ARG;
    cudaSetDevice(c->device);
    const uint64_t piece = 256ull << 20, span = 1ull << 30;
    uint8_t *h[2] = {nullptr, nullptr}, *d[2] = {nullptr, nullptr};
    int rc = XM_OK;
    for (int k = 0; k < 2 && rc == XM_OK; ++k) {
        if (cudaHostAlloc((void **)&h[k], span, cudaHostAllocDefault) != cudaSuccess || cudaMalloc((void **)&d[k], span) != cudaSuccess) { cudaGetLastError(); rc = fail(c, XM_ERR_NOMEM, "out of memory for the copy buffers"); }
        else memset(h[k], 0x41 + k, span);
    }
    cudaEvent_t e0[2], e1[2];
    for (int k = 0; k < 2; ++k) { cudaEventCreate(&e0[k]); cudaEventCreate(&e1[k]); }
    float best = 0.f;
    for (int r = 0; r < reps && rc == XM_OK; ++r) {
        cudaStreamSynchronize(c->copy_st[0]); cudaStreamSynchronize(c->dl);
        cudaEventRecord(e0[0], c->copy_st[0]); cudaEventRecord(e0[1], c->dl);
        for (uint64_t at = 0; at < std::max(h2d_bytes, d2h_bytes); at += piece) {
            const uint64_t o = at % span;
            if (at < h2d_bytes) cudaMemcpyAsync(d[0] + o, h[0] + o, (size_t)std::min<uint64_t>(piece, h2d_bytes - at), cudaMemcpyHostToDevice, c->copy_st[0]);
            if (at < d2h_bytes) cudaMemcpyAsync(h[1] + o, d[1] + o, (size_t)std::min<uint64_t>(piece, d2h_bytes - at), cudaMemcpyDeviceToHost, c->dl);
        }
        cudaEventRecord(e1[0], c->copy_st[0]); cudaEventRecord(e1[1], c->dl);
        if (cudaEventSynchronize(e1[0]) != cudaSuccess || cudaEventSynchronize(e1[1]) != cudaSuccess) { rc = fail(c, XM_ERR_CUDA, "copy failed"); break; }
        float a = 0.f, b = 0.f;
        cudaEventElapsedTime(&a, e0[0], e1[0]); cudaEventElapsedTime(&b, e0[1], e1[1]);
        const float t = std::max(a, b);
        if (r == 0 || t < best) best = t;
    }
    for (int k = 0; k < 2; ++k) { cudaEventDestroy(e0[k]); cudaEventDestroy(e1[k]); if (h[k]) cudaFreeHost(h[k]); if (d[k]) cudaFree(d[k]); }
    *ms = best;
    return rc;
}

/* ---- headers (xm_headers.h) ------------------------------------------------------------------------------------ */
static thread_local HeaderPlan g_header_plan;

static int headers_finish(std::vector<std::string> h[2], const char *version, xm_headers *out)
{
    for (int k = 0; k < 2; ++k)
        for (auto &l : h[k])
            if (!utf8_valid((const unsigned char *)l.data(), l.size())) { out->failed_input = k; g_create_error = "invalid UTF-8 in the header"; return XM_ERR_UNICODE; }
    plan_headers(h, version && *version ? version : "1.0.2", g_header_plan);
    for (int b = 0; b < 6; ++b) {
        out->text[b] = g_header_plan.text[b].data();
        out->text_len[b] = g_header_plan.text[b].size();
        out->status[b] = g_header_plan.status[b];
    }
    return XM_OK;
}

int xm_process_headers_mem(const void *prim, uint64_t prim_len, const void *sec, uint64_t sec_len, const char *version, xm_headers *out)
{
    if (!out || (!prim && prim_len) || (!sec && sec_len)) return XM_ERR_ARG;
    memset(out, 0, sizeof *out);
    out->failed_input = -1;
    const void *src[2] = {prim, sec};
    const uint64_t len[2] = {prim_len, sec_len};
    std::vector<std::string> h[2];
    for (int k = 0; k < 2; ++k) {
        const int rc = sam_header_scan((const uint8_t *)src[k], len[k], true, h[k], out->record_offset[k]);
        if (rc != HDR_OK) { out->failed_input = k; g_create_error = "no record after the header lines"; return rc; }
    }
    return headers_finish(h, version, out);
}

int xm_process_headers_fds(int fd_prim, int fd_sec, const char *version, xm_headers *out)
{
    if (!out) return XM_ERR_ARG;
    memset(out, 0, sizeof *out);
    out->failed_input = -1;
    const int fds[2] = {fd_prim, fd_sec};
    std::vector<std::string> h[2];
    for (int k = 0; k < 2; ++k) {
        std::vector<uint8_t> buf;
        for (uint64_t want = 1 << 16;; want *= 4) {
            buf.resize(want);
            const int64_t got = xm_pread_all(fds[k], buf.data(), want, 0);
            if (got < 0) { out->failed_input = k; g_create_error = std::string("read failed: ") + strerror(errno); return XM_ERR_IO; }
            const int rc = sam_header_scan(buf.data(), (uint64_t)got, (uint64_t)got < want, h[k], out->record_offset[k]);
            if (rc == HDR_MORE) continue;
            if (rc != HDR_OK) { out->failed_input = k; g_create_error = "no record after the header lines"; return rc; }
            break;
        }
    }
    return headers_finish(h, version, out);
}

/* ---- two streams in, six bins out (pipes) --------------------------------------------------------------------- */
static int write_all(int fd, const void *p, uint64_t n)
{
    uint64_t at = 0;
    while (at < n) {
        const ssize_t w = write(fd, (const uint8_t *)p + at, (size_t)std::min<uint64_t>(n - at, 1u << 30));
        if (w < 0) { if (errno == EINTR) continue; return -1; }
        at += (uint64_t)w;
    }
    return 0;
}

int xm_classify_streams(xm_ctx *c, int fd_prim, int fd_sec, const int out_fds[6], const xm_opts *opts, uint32_t out_flags,
                        const char *version, xm_result *res)
{
    if (!c || !opts || !res || !out_fds) return XM_ERR_ARG;
    memset(res, 0, sizeof *res);
    const int fds[2] = {fd_prim, fd_sec};
    FdFeeder where[2];
    HostIn in[2];
    std::vector<std::string> h[2];
    /* the headers come off the descriptors themselves; what was read behind them opens the record stream */
    for (int s = 0; s < 2; ++s) {
        std::vector<uint8_t> buf;
        bool eof = false;
        uint64_t offset = 0;
        for (;;) {
            const size_t at = buf.size();
            buf.resize(at + (1 << 16));
            ssize_t r;
            do { r = read(fds[s], buf.data() + at, 1 << 16); } while (r < 0 && errno == EINTR);
            if (r < 0) return res->status = fail(c, XM_ERR_IO, std::string("read failed: ") + strerror(errno));
            buf.resize(at + (size_t)r);
            if (r == 0) eof = true;
            const int rc = sam_header_scan(buf.data(), buf.size(), eof, h[s], offset);
            if (rc == HDR_MORE) continue;
            if (rc != HDR_OK) return res->status = fail(c, rc, "no record after the header lines of input " + std::to_string(s + 1));
            break;
        }
        for (auto &l : h[s]) if (!utf8_valid((const unsigned char *)l.data(), l.size())) return res->status = fail(c, XM_ERR_UNICODE, "invalid UTF-8 in the header");
        where[s].fd = fds[s]; where[s].off = 0; where[s].seekable = false;
        where[s].pre.assign(buf.begin() + (long)offset, buf.end());
        in[s].feed = &where[s];
        in[s].len = eof ? (uint64_t)where[s].pre.size() : (~0ull >> 2);        /* unknown until the writer closes its end */
    }
    HeaderPlan plan;
    plan_headers(h, version && *version ? version : "1.0.2", plan);
    uint32_t en = 0;
    for (int b = 0; b < 6; ++b) {
        if (out_fds[b] < 0) continue;
        en |= 1u << b;
        if (plan.status[b] != HDR_OK) return res->status = fail(c, plan.status[b], "header of output " + std::to_string(b) + " cannot be made (xm.py:124-127)");
        const int w = (out_flags & XM_OUT_BGZF) ? xm_bgzf_write(out_fds[b], plan.text[b].data(), plan.text[b].size(), 0)
                                                : write_all(out_fds[b], plan.text[b].data(), plan.text[b].size());
        if (w) return res->status = fail(c, XM_ERR_IO, std::string("write: ") + strerror(errno));
    }
    xm_opts o = *opts;
    o.enabled_bins = en;
    const int rc = stream_walk(c, in, out_fds, &o, res, out_flags);
    if (out_flags & XM_OUT_BGZF)
        for (int b = 0; b < 6; ++b) if (out_fds[b] >= 0) xm_bgzf_write(out_fds[b], nullptr, 0, 1);
    return rc;
}

}  // extern "C"
