// Runtime plumbing of libpolus_b200.so: device selection, memory, streams/events, CUDA-graph capture.
// Replaces what TensorFlow's runtime does for the reference (polus/__init__.py:107-122 device pinning,
// polus/training.py:150-151 tf.function graph).
#include "common.cuh"
#include <cuda_profiler_api.h>
#include <nvtx3/nvToolsExt.h>   // header-only: ranges are no-ops unless a profiler injected itself
#include <atomic>
#include <stdarg.h>
#include <stdlib.h>
#include <unordered_map>

std::atomic<long long> g_launch_count{0};

static thread_local char g_err[1024] = "";
static int g_num_sms = 0;
static long long g_capture_start = 0;
static std::unordered_map<void*, long long> g_graph_kernels;  // kernels recorded per captured graph

void polus_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int polus_num_sms() {
    if (g_num_sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
        if (g_num_sms <= 0) g_num_sms = 148;
    }
    return g_num_sms;
}

bool polus_pdl_enabled() {
    static const bool on = !(getenv("POLUS_PDL") && atoi(getenv("POLUS_PDL")) == 0);
    return on;
}

extern "C" {

const char* polus_last_error(void) { return g_err; }
int polus_version(void) { return 101; }

int polus_device_count(int* n) {
    POLUS_CHECK_CUDA(cudaGetDeviceCount(n));
    return 0;
}

int polus_init(int device) {
    int n = 0;
    POLUS_CHECK_CUDA(cudaGetDeviceCount(&n));
    POLUS_REQUIRE(device >= 0 && device < n, "polus_init: device %d out of range (have %d)", device, n);
    POLUS_CHECK_CUDA(cudaSetDevice(device));
    int major = 0, minor = 0;
    POLUS_CHECK_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    POLUS_CHECK_CUDA(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device));
    POLUS_REQUIRE(major == 10, "polus_init: this library is built for sm_100a only; device %d is sm_%d%d",
                  device, major, minor);
    g_num_sms = 0;
    polus_num_sms();
    POLUS_CHECK_CUDA(cudaFree(0));
    return 0;
}

int polus_device_info(int* sm_count, int* cc_major, int* cc_minor, size_t* total_mem) {
    int dev = 0;
    POLUS_CHECK_CUDA(cudaGetDevice(&dev));
    POLUS_CHECK_CUDA(cudaDeviceGetAttribute(sm_count, cudaDevAttrMultiProcessorCount, dev));
    POLUS_CHECK_CUDA(cudaDeviceGetAttribute(cc_major, cudaDevAttrComputeCapabilityMajor, dev));
    POLUS_CHECK_CUDA(cudaDeviceGetAttribute(cc_minor, cudaDevAttrComputeCapabilityMinor, dev));
    size_t free_b = 0;
    POLUS_CHECK_CUDA(cudaMemGetInfo(&free_b, total_mem));
    return 0;
}

int polus_malloc(void** d_ptr, size_t bytes) {
    cudaError_t e = cudaMalloc(d_ptr, bytes ? bytes : 16);
    if (e == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        polus_set_error("polus_malloc: out of device memory requesting %zu bytes", bytes);
        return POLUS_ERR_OOM;
    }
    POLUS_CHECK_CUDA(e);
    return 0;
}
int polus_free(void* d_ptr) {
    POLUS_CHECK_CUDA(cudaFree(d_ptr));
    return 0;
}
int polus_host_alloc(void** h_ptr, size_t bytes) {
    POLUS_CHECK_CUDA(cudaMallocHost(h_ptr, bytes ? bytes : 16));
    return 0;
}
int polus_host_free(void* h_ptr) {
    POLUS_CHECK_CUDA(cudaFreeHost(h_ptr));
    return 0;
}
int polus_memcpy_h2d(void* d, const void* h, size_t bytes, void* stream) {
    if (bytes == 0) return 0;
    POLUS_CHECK_CUDA(cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, (cudaStream_t)stream));
    return 0;
}
int polus_memcpy_d2h(void* h, const void* d, size_t bytes, void* stream) {
    if (bytes == 0) return 0;
    POLUS_CHECK_CUDA(cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    return 0;
}
int polus_memcpy_d2d(void* d, const void* s, size_t bytes, void* stream) {
    if (bytes == 0) return 0;
    POLUS_CHECK_CUDA(cudaMemcpyAsync(d, s, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return 0;
}
int polus_memset(void* d, int value, size_t bytes, void* stream) {
    if (bytes == 0) return 0;
    POLUS_CHECK_CUDA(cudaMemsetAsync(d, value, bytes, (cudaStream_t)stream));
    return 0;
}
int polus_stream_create(void** stream, int high_priority) {
    int lo = 0, hi = 0;
    POLUS_CHECK_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    cudaStream_t s;
    // 0 = normal (one level above the lowest when the device has more than two levels), 1 = highest (collectives),
    // 2 = background (lowest: weight-gradient GEMMs that fill the tails of the main chain)
    int prio = lo;
    if (high_priority == 1) prio = hi;
    else if (high_priority == 0 && lo - hi >= 2) prio = lo - 1;
    POLUS_CHECK_CUDA(cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, prio));
    *stream = s;
    return 0;
}
int polus_stream_destroy(void* stream) {
    POLUS_CHECK_CUDA(cudaStreamDestroy((cudaStream_t)stream));
    return 0;
}
int polus_stream_sync(void* stream) {
    POLUS_CHECK_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return 0;
}
int polus_device_sync(void) {
    POLUS_CHECK_CUDA(cudaDeviceSynchronize());
    return 0;
}
int polus_event_create(void** event) {
    cudaEvent_t e;
    POLUS_CHECK_CUDA(cudaEventCreate(&e));
    *event = e;
    return 0;
}
int polus_event_destroy(void* event) {
    POLUS_CHECK_CUDA(cudaEventDestroy((cudaEvent_t)event));
    return 0;
}
int polus_event_record(void* event, void* stream) {
    POLUS_CHECK_CUDA(cudaEventRecord((cudaEvent_t)event, (cudaStream_t)stream));
    return 0;
}
int polus_event_sync(void* event) {
    POLUS_CHECK_CUDA(cudaEventSynchronize((cudaEvent_t)event));
    return 0;
}
int polus_event_elapsed_ms(void* start, void* stop, float* ms) {
    POLUS_CHECK_CUDA(cudaEventElapsedTime(ms, (cudaEvent_t)start, (cudaEvent_t)stop));
    return 0;
}
int polus_stream_wait_event(void* stream, void* event) {
    POLUS_CHECK_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, (cudaEvent_t)event, 0));
    return 0;
}

int polus_graph_begin(void* stream) {
    // relaxed mode: the host may cudaMalloc activation buffers while the step is being traced
    POLUS_CHECK_CUDA(cudaStreamBeginCapture((cudaStream_t)stream, cudaStreamCaptureModeRelaxed));
    g_capture_start = g_launch_count.load();
    return 0;
}
int polus_graph_end(void* stream, void** graph_exec) {
    cudaGraph_t g = nullptr;
    POLUS_CHECK_CUDA(cudaStreamEndCapture((cudaStream_t)stream, &g));
    cudaGraphExec_t ge = nullptr;
    cudaError_t e = cudaGraphInstantiate(&ge, g, 0);
    cudaGraphDestroy(g);
    POLUS_CHECK_CUDA(e);
    *graph_exec = ge;
    const long long recorded = g_launch_count.load() - g_capture_start;
    g_graph_kernels[ge] = recorded;
    g_launch_count -= recorded;  // recorded, not executed; each replay adds them back
    return 0;
}
int polus_graph_launch(void* graph_exec, void* stream) {
    POLUS_CHECK_CUDA(cudaGraphLaunch((cudaGraphExec_t)graph_exec, (cudaStream_t)stream));
    auto it = g_graph_kernels.find(graph_exec);
    if (it != g_graph_kernels.end()) g_launch_count += it->second;
    return 0;
}
int polus_graph_destroy(void* graph_exec) {
    POLUS_CHECK_CUDA(cudaGraphExecDestroy((cudaGraphExec_t)graph_exec));
    g_graph_kernels.erase(graph_exec);
    return 0;
}

int64_t polus_launch_count(void) { return (int64_t)g_launch_count.load(); }

int polus_profiler_start(void) {
    POLUS_CHECK_CUDA(cudaProfilerStart());
    return 0;
}
int polus_profiler_stop(void) {
    POLUS_CHECK_CUDA(cudaProfilerStop());
    return 0;
}
// Named, nestable ranges on the calling thread (NVTX): what tf.profiler.experimental.Trace('step', step_num=...) marks in
// the reference (polus/callbacks.py:442-470).  nsys / ncu --nvtx show them; without a profiler attached they cost nothing.
int polus_profiler_range_push(const char* name) {
    POLUS_REQUIRE(name != nullptr, "polus_profiler_range_push: name required");
    nvtxRangePushA(name);
    return 0;
}
int polus_profiler_range_pop(void) {
    nvtxRangePop();
    return 0;
}

}  // extern "C"
