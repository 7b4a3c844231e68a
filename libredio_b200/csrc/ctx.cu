// ctx.cu -- context, status strings, pinned host memory (placed on the GPU's NUMA node).
#include "common.cuh"
#include <cctype>
#include <sched.h>
#include <string>
#include <sys/syscall.h>
#include <unistd.h>

// ---- NUMA placement without libnuma (not in the image): sysfs + the raw set_mempolicy / sched_setaffinity calls ---------
static int read_int_file(const char *path, int dflt)
{
    FILE *f = fopen(path, "r");
    if (!f) return dflt;
    int v = dflt;
    if (fscanf(f, "%d", &v) != 1) v = dflt;
    fclose(f);
    return v;
}

// "0-15,32-47" -> cpu_set_t; returns the number of CPUs
static int parse_cpulist(const char *path, cpu_set_t *set)
{
    CPU_ZERO(set);
    FILE *f = fopen(path, "r");
    if (!f) return 0;
    char buf[4096];
    const size_t n = fread(buf, 1, sizeof(buf) - 1, f);
    fclose(f);
    buf[n] = 0;
    int count = 0;
    for (char *p = buf; *p;) {
        while (*p && !isdigit((unsigned char)*p)) ++p;
        if (!*p) break;
        long a = strtol(p, &p, 10), b = a;
        if (*p == '-') b = strtol(p + 1, &p, 10);
        for (long c = a; c <= b && c < CPU_SETSIZE; ++c) { CPU_SET((int)c, set); ++count; }
    }
    return count;
}

static int gpu_numa_node(int device)
{
    char id[32] = "";
    if (cudaDeviceGetPCIBusId(id, sizeof(id), device) != cudaSuccess) return -1;
    for (char *p = id; *p; ++p) *p = (char)tolower((unsigned char)*p);
    const std::string path = std::string("/sys/bus/pci/devices/") + id + "/numa_node";
    return read_int_file(path.c_str(), -1);
}

static int online_numa_nodes(void)
{
    cpu_set_t dummy;                                    // the node list has the cpulist syntax
    return parse_cpulist("/sys/devices/system/node/online", &dummy);
}

static thread_local char g_err[512] = "";

void lrc_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" int lrc_version(void) { return LRC_VERSION; }

extern "C" const char *lrc_last_error(void) { return g_err; }

extern "C" const char *lrc_strerror(int status)
{
    switch (status) {
        case LRC_OK:              return "ok";
        case LRC_ERR_INVALID:     return "invalid argument";
        case LRC_ERR_CUDA:        return "CUDA error (no usable GPU or a runtime failure); there is no CPU fallback";
        case LRC_ERR_UNSUPPORTED: return "valid for the reference but not implemented by this library";
        case LRC_ERR_NOMEM:       return "out of memory";
        case LRC_ERR_CAPACITY:    return "output capacity too small";
        case LRC_ERR_ODD_LENGTH:  return "odd byte count into the u8 IQ unpack";
        case LRC_ERR_LENGTH:      return "frame length does not match block_size";
    }
    return "unknown status";
}

extern "C" int lrc_ctx_create(int device, lrc_ctx **out)
{
    LRC_REQUIRE(out != nullptr, LRC_ERR_INVALID, "lrc_ctx_create: null out");
    int n = 0;
    LRC_CUDA(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) {
        lrc_set_error("lrc_ctx_create: device %d out of range (%d visible)", device, n);
        return LRC_ERR_INVALID;
    }
    LRC_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    LRC_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10 || prop.minor != 0) {
        // the build emits sm_100a SASS only (arch-specific, no PTX): any other device, sm_103 (B300) included, would
        // fail at the first launch with "no kernel image" instead of this message
        lrc_set_error("lrc_ctx_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only",
                      device, prop.major, prop.minor);
        return LRC_ERR_UNSUPPORTED;
    }
    lrc_ctx *c = new (std::nothrow) lrc_ctx();
    LRC_REQUIRE(c != nullptr, LRC_ERR_NOMEM, "out of host memory");
    c->device = device;
    c->n_sm = prop.multiProcessorCount;
    c->numa_node = gpu_numa_node(device);
    c->numa_nodes = online_numa_nodes();
    cudaError_t e = cudaSuccess;
    for (cudaStream_t *s : {&c->stream, &c->copy_stream, &c->out_stream})
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(s, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        lrc_set_error("lrc_ctx_create: cudaStreamCreateWithFlags -> %s", cudaGetErrorString(e));
        lrc_ctx_destroy(c);
        return LRC_ERR_CUDA;
    }
    *out = c;
    return LRC_OK;
}

extern "C" int lrc_ctx_destroy(lrc_ctx *c)
{
    if (!c) return LRC_OK;
    cudaSetDevice(c->device);
    for (cudaStream_t s : {c->stream, c->copy_stream, c->out_stream})
        if (s) cudaStreamDestroy(s);
    delete c;
    return LRC_OK;
}

extern "C" int lrc_ctx_sync(lrc_ctx *c)
{
    LRC_BIND(c);
    LRC_CUDA(cudaStreamSynchronize(c->stream));
    return LRC_OK;
}

extern "C" int lrc_ctx_sm_count(lrc_ctx *c, int *n_sm)
{
    LRC_REQUIRE(c && n_sm, LRC_ERR_INVALID, "null argument");
    *n_sm = c->n_sm;
    return LRC_OK;
}

extern "C" int lrc_ctx_numa_node(lrc_ctx *c, int *node, int *n_nodes)
{
    LRC_REQUIRE(c != nullptr, LRC_ERR_INVALID, "null context");
    if (node) *node = c->numa_node;
    if (n_nodes) *n_nodes = c->numa_nodes;
    return LRC_OK;
}

// Pin the CALLING thread to the CPUs of the GPU's NUMA node (a KPN block thread that packs chunks into the pinned ring,
// or a one-process-per-GPU rank).  No-op (status OK, *n_cpus = 0) on a single-node host or when sysfs does not say.
extern "C" int lrc_ctx_bind_thread(lrc_ctx *c, int *n_cpus)
{
    LRC_REQUIRE(c != nullptr, LRC_ERR_INVALID, "null context");
    if (n_cpus) *n_cpus = 0;
    if (c->numa_node < 0 || c->numa_nodes < 2) return LRC_OK;
    char path[128];
    snprintf(path, sizeof(path), "/sys/devices/system/node/node%d/cpulist", c->numa_node);
    cpu_set_t set;
    const int n = parse_cpulist(path, &set);
    if (n == 0) return LRC_OK;
    if (sched_setaffinity(0, sizeof(set), &set) != 0) return LRC_OK;      // cgroup-restricted: keep the inherited mask
    if (n_cpus) *n_cpus = n;
    return LRC_OK;
}

extern "C" int lrc_host_alloc(lrc_ctx *c, size_t bytes, void **h_ptr)
{
    LRC_BIND(c);
    LRC_REQUIRE(h_ptr != nullptr, LRC_ERR_INVALID, "null out pointer");
    // the pages are allocated and pinned inside cudaHostAlloc, under the calling thread's memory policy: prefer the GPU's
    // own node for the duration of the call, so that H2D reads do not cross the socket interconnect (at 8 GPUs the
    // per-GPU copy rate fell from 55 to 24 GB/s with every rank's ring on whatever node its process started on)
    bool policy = false;
    if (c->numa_node >= 0 && c->numa_nodes > 1 && c->numa_node < 1024) {
        unsigned long mask[16] = {0};
        mask[c->numa_node / (8 * sizeof(unsigned long))] |= 1ul << (c->numa_node % (8 * sizeof(unsigned long)));
        policy = syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, mask, (unsigned long)(8 * sizeof(mask))) == 0;
    }
    const cudaError_t e = cudaHostAlloc(h_ptr, bytes ? bytes : 1, cudaHostAllocDefault);
    if (policy) syscall(SYS_set_mempolicy, 0 /* MPOL_DEFAULT */, nullptr, 0ul);
    if (e != cudaSuccess) {
        lrc_set_error("lrc_host_alloc: cudaHostAlloc(%zu) -> %s", bytes, cudaGetErrorString(e));
        return LRC_ERR_CUDA;
    }
    return LRC_OK;
}

extern "C" int lrc_host_free(lrc_ctx *c, void *h_ptr)
{
    LRC_BIND(c);
    if (h_ptr) LRC_CUDA(cudaFreeHost(h_ptr));
    return LRC_OK;
}

// ---- device memory, streams and asynchronous copies for FFI hosts without CUDA bindings of their own (rust/kpn-gpu): with
// lrc_host_alloc these are what a KPN block needs to run a pinned, double-buffered ring around the plan entry points --------
extern "C" int lrc_dev_alloc(lrc_ctx *c, size_t bytes, void **d_ptr)
{
    LRC_BIND(c);
    LRC_REQUIRE(d_ptr != nullptr, LRC_ERR_INVALID, "null out pointer");
    LRC_CUDA(cudaMalloc(d_ptr, bytes ? bytes : 1));
    return LRC_OK;
}

extern "C" int lrc_dev_free(lrc_ctx *c, void *d_ptr)
{
    LRC_BIND(c);
    if (d_ptr) LRC_CUDA(cudaFree(d_ptr));
    return LRC_OK;
}

extern "C" int lrc_dev_memset(lrc_ctx *c, void *d_ptr, int value, size_t bytes, void *stream)
{
    LRC_BIND(c);
    if (bytes) LRC_CUDA(cudaMemsetAsync(d_ptr, value, bytes, lrc_stream(c, stream)));
    return LRC_OK;
}

extern "C" int lrc_stream_create(lrc_ctx *c, void **stream)
{
    LRC_BIND(c);
    LRC_REQUIRE(stream != nullptr, LRC_ERR_INVALID, "null out pointer");
    cudaStream_t s = nullptr;
    LRC_CUDA(cudaStreamCreateWithFlags(&s, cudaStreamNonBlocking));
    *stream = s;
    return LRC_OK;
}

extern "C" int lrc_stream_destroy(lrc_ctx *c, void *stream)
{
    LRC_BIND(c);
    if (stream) LRC_CUDA(cudaStreamDestroy(reinterpret_cast<cudaStream_t>(stream)));
    return LRC_OK;
}

extern "C" int lrc_stream_sync(lrc_ctx *c, void *stream)
{
    LRC_BIND(c);
    LRC_CUDA(cudaStreamSynchronize(lrc_stream(c, stream)));
    return LRC_OK;
}

extern "C" int lrc_event_create(lrc_ctx *c, void **event)
{
    LRC_BIND(c);
    LRC_REQUIRE(event != nullptr, LRC_ERR_INVALID, "null out pointer");
    cudaEvent_t e = nullptr;
    LRC_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    *event = e;
    return LRC_OK;
}

extern "C" int lrc_event_destroy(lrc_ctx *c, void *event)
{
    LRC_BIND(c);
    if (event) LRC_CUDA(cudaEventDestroy(reinterpret_cast<cudaEvent_t>(event)));
    return LRC_OK;
}

extern "C" int lrc_event_record(lrc_ctx *c, void *event, void *stream)
{
    LRC_BIND(c);
    LRC_REQUIRE(event != nullptr, LRC_ERR_INVALID, "null event");
    LRC_CUDA(cudaEventRecord(reinterpret_cast<cudaEvent_t>(event), lrc_stream(c, stream)));
    return LRC_OK;
}

extern "C" int lrc_event_sync(lrc_ctx *c, void *event)
{
    LRC_BIND(c);
    LRC_REQUIRE(event != nullptr, LRC_ERR_INVALID, "null event");
    LRC_CUDA(cudaEventSynchronize(reinterpret_cast<cudaEvent_t>(event)));
    return LRC_OK;
}

extern "C" int lrc_copy_h2d_async(lrc_ctx *c, void *d_dst, const void *h_src, size_t bytes, void *stream)
{
    LRC_BIND(c);
    if (bytes == 0) return LRC_OK;
    LRC_REQUIRE(d_dst && h_src, LRC_ERR_INVALID, "lrc_copy_h2d_async: null pointer");
    LRC_CUDA(cudaMemcpyAsync(d_dst, h_src, bytes, cudaMemcpyHostToDevice, lrc_stream(c, stream)));
    return LRC_OK;
}

extern "C" int lrc_copy_d2h_async(lrc_ctx *c, void *h_dst, const void *d_src, size_t bytes, void *stream)
{
    LRC_BIND(c);
    if (bytes == 0) return LRC_OK;
    LRC_REQUIRE(h_dst && d_src, LRC_ERR_INVALID, "lrc_copy_d2h_async: null pointer");
    LRC_CUDA(cudaMemcpyAsync(h_dst, d_src, bytes, cudaMemcpyDeviceToHost, lrc_stream(c, stream)));
    return LRC_OK;
}

extern "C" int lrc_copy_to_host(lrc_ctx *c, void *h_dst, const void *d_src, size_t bytes)
{
    LRC_BIND(c);
    if (bytes == 0) return LRC_OK;
    LRC_REQUIRE(h_dst && d_src, LRC_ERR_INVALID, "lrc_copy_to_host: null pointer");
    LRC_CUDA(cudaDeviceSynchronize());
    LRC_CUDA(cudaMemcpy(h_dst, d_src, bytes, cudaMemcpyDeviceToHost));
    return LRC_OK;
}
