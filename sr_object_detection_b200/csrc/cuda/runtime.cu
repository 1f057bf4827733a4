// Device runtime behind the C-ABI: memory, streams, events, CUDA-graph capture.
// Replaces the reference's cuda.c:12-158 (cuda_set_device / cuda_make_array /
// cuda_push_array / cuda_pull_array / cuda_free) and the per-predict
// cudaMalloc+cudaFree of network_kernels.cu:392-407.
#include "y2_common.cuh"

#include <ctype.h>
#include <sched.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

namespace y2 {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int sm_count()
{
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev < 0 || dev >= 64) return 148;
    if (!cached[dev]) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
            n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

// CPUs next to a GPU: /sys/bus/pci/devices/<bus id>/local_cpulist ("0-31,64-95"), intersected with the CPUs this
// thread may run on.  False when the topology is not visible (containers without sysfs) or the intersection is empty.
static bool device_local_cpus(int dev, cpu_set_t *out)
{
    char bus[64] = "";
    if (cudaDeviceGetPCIBusId(bus, (int)sizeof(bus), dev) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    for (char *c = bus; *c; ++c) *c = (char)tolower(*c);
    char path[160];
    snprintf(path, sizeof(path), "/sys/bus/pci/devices/%s/local_cpulist", bus);
    FILE *f = fopen(path, "r");
    if (!f) return false;
    char line[1024] = "";
    const bool got = fgets(line, sizeof(line), f) != nullptr;
    fclose(f);
    if (!got) return false;
    cpu_set_t allowed, local;
    CPU_ZERO(&local);
    if (sched_getaffinity(0, sizeof(allowed), &allowed) != 0) return false;
    for (char *tok = strtok(line, ",\n"); tok; tok = strtok(nullptr, ",\n")) {
        int lo = 0, hi = 0;
        const int n = sscanf(tok, "%d-%d", &lo, &hi);
        if (n < 1) continue;
        if (n == 1) hi = lo;
        for (int c = lo; c <= hi && c < CPU_SETSIZE; ++c)
            if (c >= 0 && CPU_ISSET(c, &allowed)) CPU_SET(c, &local);
    }
    if (CPU_COUNT(&local) == 0) return false;
    *out = local;
    return true;
}

} // namespace y2

using namespace y2;

// Keep the calling host thread on the CPUs next to `dev` (its NUMA node): the pinned staging buffers it allocates
// afterwards land in that node's memory and its H2D copies do not cross the socket interconnect.  Returns the
// number of CPUs in the new mask, 0 when the topology is unknown (nothing changed).
extern "C" int y2_bind_thread_to_device(int dev)
{
    cpu_set_t local;
    if (getenv("Y2_NO_NUMA_BIND") || !device_local_cpus(dev, &local)) return 0;
    if (sched_setaffinity(0, sizeof(local), &local) != 0) return 0;
    return CPU_COUNT(&local);
}

extern "C" const char *y2_last_error(void) { return g_err; }
extern "C" const char *y2_version(void) { return "yolo2-b200 0.1 (sm_100a)"; }

extern "C" int y2_device_count(int *count)
{
    if (!count) return Y2_EINVAL;
    Y2_CUDA_CHECK(cudaGetDeviceCount(count));
    return Y2_OK;
}
extern "C" int y2_set_device(int dev)
{
    Y2_CUDA_CHECK(cudaSetDevice(dev));
    return Y2_OK;
}
extern "C" int y2_get_device(int *dev)
{
    if (!dev) return Y2_EINVAL;
    Y2_CUDA_CHECK(cudaGetDevice(dev));
    return Y2_OK;
}
extern "C" int y2_malloc(void **dptr, size_t bytes)
{
    if (!dptr) return Y2_EINVAL;
    Y2_CUDA_CHECK(cudaMalloc(dptr, bytes ? bytes : 16));
    return Y2_OK;
}
// cudaPointerGetAttributes tells device, managed and host memory apart; the driver's cuMemGetAddressRange gives the
// allocation around the address, so a range that runs past its allocation is refused too.
extern "C" int y2_pointer_device(const void *p, size_t bytes)
{
    typedef int (*AddressRangeFn)(unsigned long long *base, size_t *size, unsigned long long ptr);
    static AddressRangeFn range_fn = nullptr;
    if (!p || !bytes) return -1;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    if (a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) return -1;
    if (!range_fn) {
        void *fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &fn, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess || !fn) {
            cudaGetLastError();
            return -1;
        }
        range_fn = (AddressRangeFn)fn;
    }
    unsigned long long base = 0;
    size_t size = 0;
    const unsigned long long at = (unsigned long long)(uintptr_t)p;
    if (range_fn(&base, &size, at) != 0) return -1;
    if (at < base || bytes > size - (at - base)) return -1;
    return a.device;
}

extern "C" int y2_free(void *dptr)
{
    if (dptr) Y2_CUDA_CHECK(cudaFree(dptr));
    return Y2_OK;
}
extern "C" int y2_memset(void *dptr, int value, size_t bytes, y2_stream_t s)
{
    Y2_CUDA_CHECK(cudaMemsetAsync(dptr, value, bytes, to_stream(s)));
    return Y2_OK;
}
extern "C" int y2_host_alloc(void **hptr, size_t bytes)
{
    if (!hptr) return Y2_EINVAL;
    // page-lock the buffer from a CPU of the current device's NUMA node (first touch decides where the pages live);
    // the caller's affinity mask is restored afterwards
    int dev = 0;
    cpu_set_t saved, local;
    bool moved = false;
    if (bytes >= (1u << 20) && !getenv("Y2_NO_NUMA_BIND") && cudaGetDevice(&dev) == cudaSuccess &&
        sched_getaffinity(0, sizeof(saved), &saved) == 0 && device_local_cpus(dev, &local))
        moved = sched_setaffinity(0, sizeof(local), &local) == 0;
    const cudaError_t e = cudaHostAlloc(hptr, bytes ? bytes : 16, cudaHostAllocDefault);
    if (moved) sched_setaffinity(0, sizeof(saved), &saved);
    Y2_CUDA_CHECK(e);
    return Y2_OK;
}
extern "C" int y2_host_free(void *hptr)
{
    if (hptr) Y2_CUDA_CHECK(cudaFreeHost(hptr));
    return Y2_OK;
}
extern "C" int y2_memcpy_h2d(void *dst, const void *src, size_t bytes, y2_stream_t s)
{
    Y2_CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, to_stream(s)));
    return Y2_OK;
}
extern "C" int y2_memcpy_d2h(void *dst, const void *src, size_t bytes, y2_stream_t s)
{
    Y2_CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, to_stream(s)));
    return Y2_OK;
}
extern "C" int y2_stream_create(y2_stream_t *s)
{
    if (!s) return Y2_EINVAL;
    cudaStream_t st;
    Y2_CUDA_CHECK(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
    *s = (y2_stream_t)st;
    return Y2_OK;
}
extern "C" int y2_stream_destroy(y2_stream_t s)
{
    if (s) Y2_CUDA_CHECK(cudaStreamDestroy(to_stream(s)));
    return Y2_OK;
}
extern "C" int y2_stream_sync(y2_stream_t s)
{
    Y2_CUDA_CHECK(cudaStreamSynchronize(to_stream(s)));
    return Y2_OK;
}
extern "C" int y2_device_sync(void)
{
    Y2_CUDA_CHECK(cudaDeviceSynchronize());
    return Y2_OK;
}

extern "C" int y2_graph_begin(y2_stream_t s)
{
    Y2_CUDA_CHECK(cudaStreamBeginCapture(to_stream(s), cudaStreamCaptureModeThreadLocal));
    return Y2_OK;
}
extern "C" int y2_graph_end(y2_stream_t s, y2_graph_t *g)
{
    if (!g) return Y2_EINVAL;
    cudaGraph_t graph = nullptr;
    Y2_CUDA_CHECK(cudaStreamEndCapture(to_stream(s), &graph));
    cudaGraphExec_t exec = nullptr;
    cudaError_t e = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) {
        set_error("cudaGraphInstantiate -> %s", cudaGetErrorString(e));
        return Y2_ECUDA;
    }
    *g = (y2_graph_t)exec;
    return Y2_OK;
}
extern "C" int y2_graph_launch(y2_graph_t g, y2_stream_t s)
{
    Y2_CUDA_CHECK(cudaGraphLaunch((cudaGraphExec_t)g, to_stream(s)));
    return Y2_OK;
}
extern "C" int y2_graph_destroy(y2_graph_t g)
{
    if (g) Y2_CUDA_CHECK(cudaGraphExecDestroy((cudaGraphExec_t)g));
    return Y2_OK;
}

extern "C" int y2_event_create(y2_event_t *e)
{
    if (!e) return Y2_EINVAL;
    cudaEvent_t ev;
    Y2_CUDA_CHECK(cudaEventCreate(&ev));
    *e = (y2_event_t)ev;
    return Y2_OK;
}
extern "C" int y2_event_record(y2_event_t e, y2_stream_t s)
{
    Y2_CUDA_CHECK(cudaEventRecord((cudaEvent_t)e, to_stream(s)));
    return Y2_OK;
}
extern "C" int y2_event_elapsed_ms(y2_event_t a, y2_event_t b, float *ms)
{
    Y2_CUDA_CHECK(cudaEventSynchronize((cudaEvent_t)b));
    Y2_CUDA_CHECK(cudaEventElapsedTime(ms, (cudaEvent_t)a, (cudaEvent_t)b));
    return Y2_OK;
}
extern "C" int y2_event_sync(y2_event_t e)
{
    Y2_CUDA_CHECK(cudaEventSynchronize((cudaEvent_t)e));
    return Y2_OK;
}
extern "C" int y2_stream_wait_event(y2_stream_t s, y2_event_t e)
{
    Y2_CUDA_CHECK(cudaStreamWaitEvent(to_stream(s), (cudaEvent_t)e, 0));
    return Y2_OK;
}
extern "C" int y2_event_destroy(y2_event_t e)
{
    if (e) Y2_CUDA_CHECK(cudaEventDestroy((cudaEvent_t)e));
    return Y2_OK;
}

/* cudaGetErrorString for the reference's check_error(cudaError_t) (cuda.c:27-49) */
extern "C" const char *y2_cuda_error_string(int cuda_status)
{
    return cudaGetErrorString((cudaError_t)cuda_status);
}

/* cudaGetLastError, cleared: what check_error is usually fed (cuda.c: check_error(cudaPeekAtLastError())) */
extern "C" int y2_cuda_last_status(void)
{
    return (int)cudaGetLastError();
}
