// extern "C" boundary of libcpi_b200.so (declared in include/cpi_b200.h).  Plain pointers and sizes only.
#include <atomic>
#include <chrono>
#include <cstdlib>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>

#include "cpi_common.cuh"
#include "cpi_kernels.h"


namespace {

thread_local std::string g_err;
std::atomic<int64_t> g_launches{0};

int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    g_err = buf;
    return code;
}
}  // namespace
namespace cpi {
int capi_fail(int code, const char* fmt, ...) {      // same per-thread error slot, for the other translation units of the C ABI
    char buf[512];
    va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    g_err = buf;
    return code;
}
}  // namespace cpi
namespace {
#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(CPI_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); } while (0)

struct DevInfo { int sms = 0; int max_smem = 0; bool ok = false; };
int device_info(DevInfo& d) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return fail(CPI_ENODEVICE, "no CUDA device: %s", cudaGetErrorString(e));
    static std::mutex mu;
    static DevInfo cache[64];
    std::lock_guard<std::mutex> lk(mu);
    if (dev < 64 && cache[dev].ok) { d = cache[dev]; return CPI_OK; }
    int major = 0;
    CU(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    if (major != 10) return fail(CPI_ENODEVICE, "device %d is sm_%d*, this library is built for sm_100a (B200) only", dev, major * 10);
    CU(cudaDeviceGetAttribute(&d.sms, cudaDevAttrMultiProcessorCount, dev));
    CU(cudaDeviceGetAttribute(&d.max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    d.ok = true;
    if (dev < 64) cache[dev] = d;
    return CPI_OK;
}

// grow-only scratch buffers for the *_host entry points (per process; guarded by one mutex: host calls serialise)
struct Scratch {
    static constexpr int NSTREAM = 8;
    void* dev[8] = {nullptr}; size_t dev_sz[8] = {0};
    cudaStream_t stream = nullptr;            // copy-in / general stream
    cudaStream_t work[NSTREAM] = {nullptr};   // one per pipeline chunk (kernel + copy-out)
    cudaEvent_t ev[NSTREAM] = {nullptr};
    int device = -1;
};
std::mutex g_scratch_mu;
double g_host_submit_ms = 0.0, g_host_total_ms = 0.0;   // last cpi_preintegrate_batch_host call: time to enqueue everything / until drained
Scratch g_scratch;

int scratch_prepare() {
    int dev = 0;
    CU(cudaGetDevice(&dev));
    if (g_scratch.device != dev) {
        // buffers belong to the device they were allocated on; drop them if the caller switched device
        for (int i = 0; i < 8; i++) { if (g_scratch.dev[i]) cudaFree(g_scratch.dev[i]); g_scratch.dev[i] = nullptr; g_scratch.dev_sz[i] = 0; }
        if (g_scratch.stream) { cudaStreamDestroy(g_scratch.stream); g_scratch.stream = nullptr; }
        for (int i = 0; i < Scratch::NSTREAM; i++) {
            if (g_scratch.work[i]) { cudaStreamDestroy(g_scratch.work[i]); g_scratch.work[i] = nullptr; }
            if (g_scratch.ev[i]) { cudaEventDestroy(g_scratch.ev[i]); g_scratch.ev[i] = nullptr; }
        }
        g_scratch.device = dev;
    }
    if (!g_scratch.stream) CU(cudaStreamCreateWithFlags(&g_scratch.stream, cudaStreamNonBlocking));
    for (int i = 0; i < Scratch::NSTREAM; i++) {
        if (!g_scratch.work[i]) CU(cudaStreamCreateWithFlags(&g_scratch.work[i], cudaStreamNonBlocking));
        if (!g_scratch.ev[i]) CU(cudaEventCreateWithFlags(&g_scratch.ev[i], cudaEventDisableTiming));
    }
    return CPI_OK;
}
int dev_buf(int slot, size_t bytes, void** out) {
    if (bytes == 0) bytes = 8;
    if (g_scratch.dev_sz[slot] < bytes) {
        if (g_scratch.dev[slot]) CU(cudaFree(g_scratch.dev[slot]));
        g_scratch.dev[slot] = nullptr; g_scratch.dev_sz[slot] = 0;
        cudaError_t e = cudaMalloc(&g_scratch.dev[slot], bytes);
        if (e != cudaSuccess) return fail(CPI_ENOMEM, "cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
        g_scratch.dev_sz[slot] = bytes;
    }
    *out = g_scratch.dev[slot];
    return CPI_OK;
}

int preintegrate_dev(int model, int dtype, int64_t n_windows, const int64_t* sample_offsets, int64_t ns_uniform,
                            const void* samples, const void* lin, const double* sigmas, int flags, void* out_records, void* stream, int wpb,
                            const void* init_records = nullptr) {
    if (model != 1 && model != 2) return fail(CPI_EINVAL, "model must be 1 or 2 (got %d)", model);
    if (dtype != 64 && dtype != 32) return fail(CPI_EINVAL, "dtype must be 64 or 32 (got %d)", dtype);
    if (n_windows < 0 || (!sample_offsets && ns_uniform < 0)) return fail(CPI_EINVAL, "negative count");
    if (n_windows == 0) return CPI_OK;
    if (!lin || !sigmas || !out_records) return fail(CPI_EINVAL, "null pointer argument");
    // device-resident CSR offsets cannot be inspected here: a NULL samples pointer is only rejected when the layout is uniform and
    // non-empty (an all-empty CSR shard legitimately has no sample buffer)
    if (!samples && !sample_offsets && ns_uniform > 0) return fail(CPI_EINVAL, "samples is null");
    if (model == 1 && (flags & CPI_FLAG_ANALYTIC_JACOBIANS)) flags &= ~CPI_FLAG_ANALYTIC_JACOBIANS;   // model 1 is always analytic
    DevInfo d;
    int rc = device_info(d);
    if (rc) return rc;
    cpi::PreintParams p;
    p.n_windows = n_windows; p.offsets = sample_offsets; p.ns_uniform = ns_uniform;
    p.samples = samples; p.lin = lin; p.out = out_records; p.init = init_records;
    if (init_records && (!cpi::preint_tri_supported(model, flags) || getenv("CPI_B200_LEGACY")))
        return fail(CPI_EINVAL, "continuation is implemented for the default modes only (no imu_avg, model 2 with state_transition_jacobians)");
    p.q_w = sigmas[0] * sigmas[0]; p.q_wb = sigmas[1] * sigmas[1]; p.q_a = sigmas[2] * sigmas[2]; p.q_ab = sigmas[3] * sigmas[3];
    p.wpb = wpb;
    int launches = 0;
    CU(cpi::preint_launch(model, dtype, flags, p, d.sms, d.max_smem, (cudaStream_t)stream, &launches));
    g_launches += launches;
    return CPI_OK;
}

}  // namespace

extern "C" {

const char* cpi_last_error(void) { return g_err.c_str(); }
const char* cpi_version(void) { return "cpi_b200 0.2 (sm_100a)"; }
int cpi_record_doubles(int model) { return model == 1 ? CPI_REC_V1_DOUBLES : (model == 2 ? CPI_REC_V2_DOUBLES : CPI_EINVAL); }
int64_t cpi_launch_count(void) { return g_launches.load(); }

int cpi_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) return fail(CPI_ENODEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    int ok = 0;
    for (int i = 0; i < n; i++) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, i) == cudaSuccess && major == 10) ok++;
    }
    return ok;
}

int cpi_preintegrate_batch(int model, int dtype, int64_t n_windows, const int64_t* sample_offsets, int64_t ns_uniform,
                           const void* samples, const void* lin, const double* sigmas, int flags, void* out_records, void* stream) {
    return preintegrate_dev(model, dtype, n_windows, sample_offsets, ns_uniform, samples, lin, sigmas, flags, out_records, stream, 0);
}

int cpi_preintegrate_batch_continue(int model, int dtype, int64_t n_windows, const int64_t* sample_offsets, int64_t ns_uniform,
                                    const void* samples, const void* lin, const double* sigmas, int flags, void* records, void* stream) {
    return preintegrate_dev(model, dtype, n_windows, sample_offsets, ns_uniform, samples, lin, sigmas, flags, records, stream, 0, records);
}

int cpi_preintegrate_batch_host(int model, int dtype, int64_t n_windows, const int64_t* sample_offsets, int64_t ns_uniform,
                                const void* samples, const void* lin, const double* sigmas, int flags, void* out_records) {
    if (model != 1 && model != 2) return fail(CPI_EINVAL, "model must be 1 or 2 (got %d)", model);
    if (dtype != 64 && dtype != 32) return fail(CPI_EINVAL, "dtype must be 64 or 32 (got %d)", dtype);
    if (n_windows < 0) return fail(CPI_EINVAL, "negative count");
    if (n_windows == 0) return CPI_OK;
    if (!lin || !sigmas || !out_records) return fail(CPI_EINVAL, "null pointer argument");
    const int avg = (flags & CPI_FLAG_IMU_AVG) ? 1 : 0;
    const int64_t ent_w = ns_uniform + avg;
    const int64_t entries = sample_offsets ? sample_offsets[n_windows] : n_windows * ent_w;
    if (entries > 0 && !samples) return fail(CPI_EINVAL, "samples is null");
    if (sample_offsets) {                       // the host copy of the CSR layout can be validated before anything reaches the device
        if (sample_offsets[0] < 0) return fail(CPI_EINVAL, "sample_offsets[0] is negative");
        for (int64_t w = 0; w < n_windows; w++)
            if (sample_offsets[w + 1] < sample_offsets[w])     // an empty window is legal (also with imu_avg: it simply has no step)
                return fail(CPI_EINVAL, "sample_offsets must be non-decreasing (window %lld)", (long long)w);
    } else if (ns_uniform < 0) return fail(CPI_EINVAL, "negative count");
    const int rd = cpi_record_doubles(model);
    const size_t es = dtype == 32 ? 4 : 8;
    DevInfo d;
    int rc = device_info(d);
    if (rc) return rc;
    std::lock_guard<std::mutex> lk(g_scratch_mu);
    if ((rc = scratch_prepare())) return rc;
    void *d_s, *d_l, *d_o, *d_off = nullptr;
    if ((rc = dev_buf(0, (size_t)entries * CPI_SAMPLE_DOUBLES * es + 16, &d_s))) return rc;
    if ((rc = dev_buf(1, (size_t)n_windows * CPI_LIN_DOUBLES * es, &d_l))) return rc;
    if ((rc = dev_buf(2, (size_t)n_windows * rd * es, &d_o))) return rc;
    if (sample_offsets && (rc = dev_buf(3, (size_t)(n_windows + 1) * 8, &d_off))) return rc;

    // Chunked pipeline: H2D of chunk k+1 runs under the kernel of chunk k, D2H of chunk k under the kernel of chunk k+1.  The
    // default kernels are one-warp CTAs, so chunk kernels of different streams co-reside on the SMs and a batch can be cut into
    // many small chunks.  The lane-per-window kernels (imu_avg / analytic modes) are launched with the windows-per-block the WHOLE
    // batch would use, so that a chunk occupies only its share of the SMs.
    //
    // Wavefront schedule (uniform layout, fp64, default modes).  A window is a chain of ns DEPENDENT samples (~3.7 us each on B200,
    // whatever the occupancy), so a chunk that travels whole finishes ~ns x 3.7 us after it arrived, however small it is: 0.74 ms
    // behind the last byte of H2D for 200-sample windows, a quarter of the PCIe time of the whole 10k-window batch.  Instead the batch
    // is cut into G window groups x S sample segments, and the (group, segment) tiles are sent along ANTI-DIAGONALS: tile (g, s) is a
    // strided copy (cudaMemcpy2DAsync: rows = windows of the group, row = samples [s ns/S, (s+1) ns/S)) followed, on the group's stream,
    // by a CONTINUATION kernel over the group (cpi_preintegrate_batch_continue).  Every group's chain then runs WHILE its samples
    // arrive, S other groups keep the SMs busy in between, groups finish (and copy out) one after the other, and what is left behind
    // the last byte is one segment of one group + that group's D2H.  fp64 only: a float record would round the fp64-accumulated
    // covariance state at every segment.
    const size_t in_bytes = (size_t)entries * CPI_SAMPLE_DOUBLES * es;
    const int cap = cpi::preint_cap(model, dtype, flags, d.sms);     // windows per CTA of the kernel preint_launch will select
    const bool small_ctas = cap <= 16;
    const bool big = in_bytes >= ((size_t)16 << 20) && n_windows >= 8 * (int64_t)d.sms;
    int nchunk = 1;
    if (big) {
        nchunk = small_ctas ? (int)(in_bytes >> 23) : 4;             // ~8 MB of samples per chunk
        if (nchunk < 4) nchunk = 4;
        if (nchunk > 16) nchunk = 16;
    }
    if (const char* e = getenv("CPI_B200_HOST_CHUNKS")) { int v = atoi(e); if (v >= 1 && v <= 64) nchunk = v; }   // A/B measurements
    int64_t need = (n_windows + d.sms - 1) / d.sms;
    const int wpb = (int)(need < cap ? (need < 1 ? 1 : need) : cap);
    const int64_t blocks = (n_windows + wpb - 1) / wpb;
    // wavefront geometry: the first wave_H % of the windows travel as whole-window chunks, the rest as G groups x S segments.
    // Defaults (measured on B200, tools/host_pipeline_probe.py, profiles/r02_host_pipeline_probe.json): every copy costs ~3.5 us of dead
    // time on the copy engine, so few large tiles beat a fine wavefront -- ONE group of 4 segments, sized so that its transfer lasts
    // about as long as its sample chain (ns x ~4.6 us incl. the per-segment record reload, x ~50 GB/s of PCIe; model 2 chains are
    // ~1.5x longer), behind whole-window chunks for everything before it.
    int wave_G = 0, wave_S = 0, wave_H = 0;
    if (big) {
        wave_G = 1;
        wave_S = (int)(ns_uniform / 8 < 4 ? ns_uniform / 8 : 4);
        const double tail_bytes = (double)ns_uniform * (model == 1 ? 231e3 : 344e3);
        const double frac = tail_bytes / (double)in_bytes;
        wave_H = frac >= 1.0 ? 0 : (int)(100.0 * (1.0 - frac));
        if (wave_H > 95) wave_H = 95;
    }
    if (const char* e = getenv("CPI_B200_HOST_WAVE")) {              // "G,S[,H]": A/B measurements and tests ("0,0" = whole-window chunks only)
        int a_ = 0, b_ = 0, c_ = 0;
        const int nf = sscanf(e, "%d,%d,%d", &a_, &b_, &c_);
        if (nf >= 2 && a_ >= 0 && a_ <= 256 && b_ >= 0 && b_ <= 64 && c_ >= 0 && c_ < 100) { wave_G = a_; wave_S = b_; wave_H = nf == 3 ? c_ : 0; }
    }
    const bool wave = dtype == 64 && !sample_offsets && !avg && small_ctas && cpi::preint_tri_supported(model, flags) && !getenv("CPI_B200_LEGACY") &&
                      wave_G >= 1 && wave_S >= 2 && ns_uniform >= 2 * (int64_t)wave_S;
    const int64_t head_blocks = wave ? blocks * wave_H / 100 : blocks;
    const int64_t head_hi = wave ? head_blocks * wpb : n_windows;    // windows [0, head_hi) travel whole, [head_hi, n) as the wavefront
    if (wave && head_blocks > 0) { nchunk = (int)((int64_t)nchunk * wave_H / 100); if (nchunk < 1) nchunk = 1; }
    const int64_t blocks_per_chunk = (head_blocks + nchunk - 1) / nchunk > 0 ? (head_blocks + nchunk - 1) / nchunk : 1;
    const auto t_start = std::chrono::steady_clock::now();
    int used = 0;                                                    // streams handed out so far (round robin)

    cudaStream_t s_in = g_scratch.stream;
    rc = CPI_OK;
    // every error path drains the streams before returning: async copies into the caller's buffers must not outlive the call
#define CUX(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { rc = fail(CPI_ECUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); goto drain; } } while (0)
    if (sample_offsets) CUX(cudaMemcpyAsync(d_off, sample_offsets, (size_t)(n_windows + 1) * 8, cudaMemcpyHostToDevice, s_in));
    for (int k = 0; k < nchunk; k++) {
        const int64_t lo = (int64_t)k * blocks_per_chunk * wpb;
        if (lo >= head_hi) break;
        const int64_t hi = (lo + blocks_per_chunk * wpb < head_hi) ? lo + blocks_per_chunk * wpb : head_hi;
        used = k + 1;
        const int64_t e_lo = sample_offsets ? sample_offsets[lo] : lo * ent_w, e_hi = sample_offsets ? sample_offsets[hi] : hi * ent_w;
        const int si = k % Scratch::NSTREAM;
        cudaStream_t sk = g_scratch.work[si];
        CUX(cudaMemcpyAsync((char*)d_l + (size_t)lo * CPI_LIN_DOUBLES * es, (const char*)lin + (size_t)lo * CPI_LIN_DOUBLES * es,
                            (size_t)(hi - lo) * CPI_LIN_DOUBLES * es, cudaMemcpyHostToDevice, s_in));
        if (e_hi > e_lo)
            CUX(cudaMemcpyAsync((char*)d_s + (size_t)e_lo * CPI_SAMPLE_DOUBLES * es, (const char*)samples + (size_t)e_lo * CPI_SAMPLE_DOUBLES * es,
                                (size_t)(e_hi - e_lo) * CPI_SAMPLE_DOUBLES * es, cudaMemcpyHostToDevice, s_in));
        CUX(cudaEventRecord(g_scratch.ev[si], s_in));
        CUX(cudaStreamWaitEvent(sk, g_scratch.ev[si], 0));
        {
            // offsets are absolute entry indices, so CSR chunks keep the global sample base; uniform chunks shift it
            const void* s_base = sample_offsets ? d_s : (const void*)((const char*)d_s + (size_t)e_lo * CPI_SAMPLE_DOUBLES * es);
            rc = preintegrate_dev(model, dtype, hi - lo, sample_offsets ? (const int64_t*)d_off + lo : nullptr, ns_uniform, s_base,
                                  (const char*)d_l + (size_t)lo * CPI_LIN_DOUBLES * es, sigmas, flags, (char*)d_o + (size_t)lo * rd * es, sk, wpb);
            if (rc) goto drain;
        }
        CUX(cudaMemcpyAsync((char*)out_records + (size_t)lo * rd * es, (const char*)d_o + (size_t)lo * rd * es, (size_t)(hi - lo) * rd * es,
                            cudaMemcpyDeviceToHost, sk));
    }
    if (wave && head_hi < n_windows) {
        const size_t sb = (size_t)CPI_SAMPLE_DOUBLES * es;            // bytes per sample
        const int64_t wblocks = blocks - head_blocks;
        const int64_t bpg = (wblocks + wave_G - 1) / wave_G;          // blocks per group
        const int64_t G = (wblocks + bpg - 1) / bpg;
        const int64_t seg_len = (ns_uniform + wave_S - 1) / wave_S;
        const int64_t S = (ns_uniform + seg_len - 1) / seg_len;
        for (int64_t t = 0; t < G + S - 1; t++) {
            for (int64_t g = t - S + 1 > 0 ? t - S + 1 : 0; g <= t && g < G; g++) {      // oldest group (latest segment) first
                const int64_t sidx = t - g, s0 = sidx * seg_len;
                const int64_t len = s0 + seg_len <= ns_uniform ? seg_len : ns_uniform - s0;
                const int64_t lo = head_hi + g * bpg * wpb, hi = (lo + bpg * wpb < n_windows) ? lo + bpg * wpb : n_windows, ng = hi - lo;
                const int si = (int)((used + g) % Scratch::NSTREAM);
                cudaStream_t sk = g_scratch.work[si];
                char* d_lg = (char*)d_l + (size_t)lo * CPI_LIN_DOUBLES * es;
                char* d_og = (char*)d_o + (size_t)lo * rd * es;
                if (sidx == 0)
                    CUX(cudaMemcpyAsync(d_lg, (const char*)lin + (size_t)lo * CPI_LIN_DOUBLES * es, (size_t)ng * CPI_LIN_DOUBLES * es, cudaMemcpyHostToDevice, s_in));
                // the tiles of a group are compact ([window][len]) and together fill the group's share of the device sample buffer
                char* d_seg = (char*)d_s + ((size_t)lo * ns_uniform + (size_t)ng * s0) * sb;
                CUX(cudaMemcpy2DAsync(d_seg, (size_t)len * sb, (const char*)samples + ((size_t)lo * ns_uniform + (size_t)s0) * sb, (size_t)ns_uniform * sb,
                                      (size_t)len * sb, (size_t)ng, cudaMemcpyHostToDevice, s_in));
                CUX(cudaEventRecord(g_scratch.ev[si], s_in));
                CUX(cudaStreamWaitEvent(sk, g_scratch.ev[si], 0));
                rc = preintegrate_dev(model, dtype, ng, nullptr, len, d_seg, d_lg, sigmas, flags, d_og, sk, wpb, sidx > 0 ? d_og : nullptr);
                if (rc) goto drain;
                if (sidx == S - 1)
                    CUX(cudaMemcpyAsync((char*)out_records + (size_t)lo * rd * es, d_og, (size_t)ng * rd * es, cudaMemcpyDeviceToHost, sk));
            }
        }
    }
drain:
#undef CUX
    g_host_submit_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count();
    for (int k = 0; k < Scratch::NSTREAM; k++) {
        cudaError_t e_ = cudaStreamSynchronize(g_scratch.work[k]);
        if (e_ != cudaSuccess && rc == CPI_OK) rc = fail(CPI_ECUDA, "cudaStreamSynchronize failed: %s", cudaGetErrorString(e_));
    }
    {
        cudaError_t e_ = cudaStreamSynchronize(s_in);
        if (e_ != cudaSuccess && rc == CPI_OK) rc = fail(CPI_ECUDA, "cudaStreamSynchronize failed: %s", cudaGetErrorString(e_));
    }
    g_host_total_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count();
    return rc;
}

int cpi_host_last_timing(double* submit_ms, double* total_ms) {
    if (submit_ms) *submit_ms = g_host_submit_ms;
    if (total_ms) *total_ms = g_host_total_ms;
    return CPI_OK;
}

int cpi_host_register(void* ptr, size_t bytes) {
    if (!ptr || bytes == 0) return fail(CPI_EINVAL, "null pointer argument");
    CU(cudaHostRegister(ptr, bytes, cudaHostRegisterDefault));
    return CPI_OK;
}
int cpi_host_unregister(void* ptr) {
    if (!ptr) return fail(CPI_EINVAL, "null pointer argument");
    CU(cudaHostUnregister(ptr));
    return CPI_OK;
}

int cpi_imu_factor_eval_batch(int model, int64_t n_factors, const double* states, const int64_t* idx_i, const int64_t* idx_j,
                              const double* records, const double* lin, double* e, double* H1, double* H2, void* stream) {
    if (model != 1 && model != 2) return fail(CPI_EINVAL, "model must be 1 or 2 (got %d)", model);
    if (n_factors < 0) return fail(CPI_EINVAL, "negative count");
    if (n_factors == 0) return CPI_OK;
    if (!states || !records || !lin || !e) return fail(CPI_EINVAL, "null pointer argument");
    if ((idx_i == nullptr) != (idx_j == nullptr)) return fail(CPI_EINVAL, "idx_i and idx_j must both be given or both be null");
    DevInfo d;
    int rc = device_info(d);
    if (rc) return rc;
    cpi::FactorParams p{n_factors, states, idx_i, idx_j, records, lin, e, H1, H2};
    CU(cpi::factor_launch(model, p, (cudaStream_t)stream));
    g_launches += 1;
    return CPI_OK;
}

int cpi_imu_factor_eval_batch_host(int model, int64_t n_factors, int64_t n_states, const double* states, const int64_t* idx_i,
                                   const int64_t* idx_j, const double* records, const double* lin, double* e, double* H1, double* H2) {
    if (model != 1 && model != 2) return fail(CPI_EINVAL, "model must be 1 or 2 (got %d)", model);
    if (n_factors < 0 || n_states < 0) return fail(CPI_EINVAL, "negative count");
    if (n_factors == 0) return CPI_OK;
    if (!states || !records || !lin || !e) return fail(CPI_EINVAL, "null pointer argument");
    if (!idx_i && n_states < n_factors + 1) return fail(CPI_EINVAL, "chain indexing needs n_states >= n_factors + 1");
    if ((idx_i == nullptr) != (idx_j == nullptr)) return fail(CPI_EINVAL, "idx_i and idx_j must both be given or both be null");
    if (idx_i)
        for (int64_t f = 0; f < n_factors; f++)
            if (idx_i[f] < 0 || idx_i[f] >= n_states || idx_j[f] < 0 || idx_j[f] >= n_states)
                return fail(CPI_EINVAL, "factor %lld: state index out of range [0, %lld)", (long long)f, (long long)n_states);
    const int rd = cpi_record_doubles(model);
    std::lock_guard<std::mutex> lk(g_scratch_mu);
    int rc = scratch_prepare();
    if (rc) return rc;
    cudaStream_t st = g_scratch.stream;
    void *d_x, *d_r, *d_l, *d_e, *d_h1 = nullptr, *d_h2 = nullptr, *d_i = nullptr, *d_j = nullptr;
    if ((rc = dev_buf(0, (size_t)n_states * CPI_STATE_DOUBLES * 8, &d_x))) return rc;
    if ((rc = dev_buf(1, (size_t)n_factors * CPI_LIN_DOUBLES * 8, &d_l))) return rc;
    if ((rc = dev_buf(2, (size_t)n_factors * rd * 8, &d_r))) return rc;
    if ((rc = dev_buf(4, (size_t)n_factors * 15 * 8, &d_e))) return rc;
    if (H1 && (rc = dev_buf(5, (size_t)n_factors * 225 * 8, &d_h1))) return rc;
    if (H2 && (rc = dev_buf(6, (size_t)n_factors * 225 * 8, &d_h2))) return rc;
    if (idx_i) {
        if ((rc = dev_buf(3, (size_t)n_factors * 8, &d_i))) return rc;
        if ((rc = dev_buf(7, (size_t)n_factors * 8, &d_j))) return rc;
        CU(cudaMemcpyAsync(d_i, idx_i, (size_t)n_factors * 8, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(d_j, idx_j, (size_t)n_factors * 8, cudaMemcpyHostToDevice, st));
    }
    CU(cudaMemcpyAsync(d_x, states, (size_t)n_states * CPI_STATE_DOUBLES * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_l, lin, (size_t)n_factors * CPI_LIN_DOUBLES * 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_r, records, (size_t)n_factors * rd * 8, cudaMemcpyHostToDevice, st));
    rc = cpi_imu_factor_eval_batch(model, n_factors, (const double*)d_x, (const int64_t*)d_i, (const int64_t*)d_j, (const double*)d_r,
                                   (const double*)d_l, (double*)d_e, (double*)d_h1, (double*)d_h2, st);
    if (rc) return rc;
    CU(cudaMemcpyAsync(e, d_e, (size_t)n_factors * 15 * 8, cudaMemcpyDeviceToHost, st));
    if (H1) CU(cudaMemcpyAsync(H1, d_h1, (size_t)n_factors * 225 * 8, cudaMemcpyDeviceToHost, st));
    if (H2) CU(cudaMemcpyAsync(H2, d_h2, (size_t)n_factors * 225 * 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return CPI_OK;
}

int cpi_imu_factor_hessian_batch(int model, int64_t n_factors, const double* records, const double* e, const double* H1, const double* H2,
                                 double* G11, double* G12, double* G22, double* g1, double* g2, double* f, void* stream) {
    if (model != 1 && model != 2) return fail(CPI_EINVAL, "model must be 1 or 2 (got %d)", model);
    if (n_factors < 0) return fail(CPI_EINVAL, "negative count");
    if (n_factors == 0) return CPI_OK;
    if (!records || !e || !H1 || !H2 || !G11 || !G12 || !G22 || !g1 || !g2 || !f) return fail(CPI_EINVAL, "null pointer argument");
    DevInfo d;
    int rc = device_info(d);
    if (rc) return rc;
    CU(cpi::hessian_launch(cpi_record_doubles(model), n_factors, records, e, H1, H2, G11, G12, G22, g1, g2, f, (cudaStream_t)stream));
    g_launches += 1;
    return CPI_OK;
}

int cpi_imu_factor_whiten_batch(int model, int64_t n_factors, const double* records, const double* e, const double* H1, const double* H2,
                                double* A1, double* A2, double* b, void* stream) {
    if (model != 1 && model != 2) return fail(CPI_EINVAL, "model must be 1 or 2 (got %d)", model);
    if (n_factors < 0) return fail(CPI_EINVAL, "negative count");
    if (n_factors == 0) return CPI_OK;
    if (!records || !e || !H1 || !H2 || !A1 || !A2 || !b) return fail(CPI_EINVAL, "null pointer argument");
    DevInfo d;
    int rc = device_info(d);
    if (rc) return rc;
    CU(cpi::whiten_launch(cpi_record_doubles(model), n_factors, records, e, H1, H2, A1, A2, b, (cudaStream_t)stream));
    g_launches += 1;
    return CPI_OK;
}

int cpi_imu_chain_assemble(int64_t n_factors, const double* G11, const double* G12, const double* G22, const double* g1, const double* g2, double lambda,
                           int diagonal_damping, const double* prior_info0, const double* prior_rhs0, double* D, double* E, double* rhs, void* stream) {
    if (n_factors < 0) return fail(CPI_EINVAL, "negative count");
    if (n_factors > 0 && (!G11 || !G12 || !G22 || !g1 || !g2 || !E)) return fail(CPI_EINVAL, "null pointer argument");
    if (!D || !rhs) return fail(CPI_EINVAL, "null pointer argument");
    if (n_factors >= 2147483647) return fail(CPI_EINVAL, "chain too long");
    if (!(lambda >= 0.0)) return fail(CPI_EINVAL, "lambda must be >= 0 (got %g)", lambda);
    DevInfo d;
    int rc = device_info(d);
    if (rc) return rc;
    CU(cpi::chain_assemble_launch(n_factors, G11, G12, G22, g1, g2, lambda, diagonal_damping != 0, prior_info0, prior_rhs0, D, E, rhs, (cudaStream_t)stream));
    g_launches += 1;
    return CPI_OK;
}

int64_t cpi_imu_chain_solve_workspace(int64_t n_states) { return n_states < 0 ? (int64_t)CPI_EINVAL : cpi::chain_solve_workspace_bytes(n_states); }

int cpi_imu_chain_solve(int64_t n_states, const double* D, const double* E, const double* rhs, double* x, void* workspace, void* stream) {
    if (n_states < 0) return fail(CPI_EINVAL, "negative count");
    if (n_states == 0) return CPI_OK;
    if (!D || !rhs || !x || (n_states > 1 && (!E || !workspace))) return fail(CPI_EINVAL, "null pointer argument");
    DevInfo d;
    int rc = device_info(d);
    if (rc) return rc;
    int launches = 0;
    CU(cpi::chain_solve_launch(n_states, D, E, rhs, x, (double*)workspace, (cudaStream_t)stream, &launches));
    g_launches += launches;
    return CPI_OK;
}

int64_t cpi_imu_chain_marginals_workspace(int64_t n_states) { return n_states < 0 ? (int64_t)CPI_EINVAL : cpi::chain_solve_workspace_bytes(n_states); }

int cpi_imu_chain_marginals(int64_t n_states, const double* D, const double* E, double* S_diag, double* S_off, void* workspace, void* stream) {
    if (n_states < 0) return fail(CPI_EINVAL, "negative count");
    if (n_states == 0) return CPI_OK;
    if (!D || !S_diag || (n_states > 1 && (!E || !workspace))) return fail(CPI_EINVAL, "null pointer argument");
    DevInfo d;
    int rc = device_info(d);
    if (rc) return rc;
    int launches = 0;
    CU(cpi::chain_marginals_launch(n_states, D, E, S_diag, S_off, (double*)workspace, (cudaStream_t)stream, &launches));
    g_launches += launches;
    return CPI_OK;
}

int cpi_predict_state_batch(int model, int64_t n, const double* states_k, const double* records, const double* lin, double* states_k1, void* stream) {
    if (model != 1 && model != 2) return fail(CPI_EINVAL, "model must be 1 or 2 (got %d)", model);
    if (n < 0) return fail(CPI_EINVAL, "negative count");
    if (n == 0) return CPI_OK;
    if (!states_k || !records || !lin || !states_k1) return fail(CPI_EINVAL, "null pointer argument");
    DevInfo d;
    int rc = device_info(d);
    if (rc) return rc;
    CU(cpi::predict_launch(model, n, states_k, records, lin, states_k1, (cudaStream_t)stream));
    g_launches += 1;
    return CPI_OK;
}

int cpi_retract_batch(int64_t n, const double* states, const double* xi, double* states_out, void* stream) {
    if (n < 0) return fail(CPI_EINVAL, "negative count");
    if (n == 0) return CPI_OK;
    if (!states || !xi || !states_out) return fail(CPI_EINVAL, "null pointer argument");
    DevInfo d;
    int rc = device_info(d);
    if (rc) return rc;
    CU(cpi::retract_launch(n, states, xi, states_out, (cudaStream_t)stream));
    g_launches += 1;
    return CPI_OK;
}

}  // extern "C"
