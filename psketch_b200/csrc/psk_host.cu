// psk_host.cu — host-buffer entry points of the C ABI (include/psk_craft.h, "host_" section).
//
// A caller that keeps its environments in host memory (as the reference does: every CraftState
// is a numpy object on the CPU) hands whole batches to psk_craft_host_tick.  The batch is cut
// into chunks; chunk i runs on stream i % PSK_HOST_STREAMS as  H2D(state) -> fused tick kernel
// -> D2H(features, teacher actions, flags, new state), so the copy engines and the SMs overlap
// across chunks.  Pass pinned memory (psk_host_alloc, or any cudaHostRegister'ed / torch-pinned
// buffer) or the copies degrade to staged synchronous ones.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>

#include <cuda_runtime.h>

#include "../../include/psk_craft.h"
#include "psk_common.cuh"
#include "psk_hostcpu.h"

#define PSK_HOST_STREAMS 3
#define PSK_WIDEN_BLOCK (64u << 10)     // bytes of u8 per widening job (256 KB of f32 written)

struct psk_craft_host_ctx {
    psk_craft_tables tables;
    int64_t max_envs, chunk;
    int cell_stride, nf;
    int device;
    cudaStream_t streams[PSK_HOST_STREAMS];
    // per-stream chunk buffers
    uint8_t *d_grid[PSK_HOST_STREAMS], *d_agent[PSK_HOST_STREAMS], *d_action[PSK_HOST_STREAMS];
    uint8_t *d_expert[PSK_HOST_STREAMS], *d_done[PSK_HOST_STREAMS], *d_success[PSK_HOST_STREAMS];
    float *d_feat[PSK_HOST_STREAMS];
    // device-resident episode tables (static per context)
    uint8_t *d_scen_grid, *d_init_agent;
    int32_t *d_scen_idx;
    int64_t n_scen, n_eps;
    unsigned long long *d_stats;   // d_stats[0..3] and d_err live in ONE 64-byte allocation (d_stats) so that
    int32_t *d_err;                // both come down with a single copy into the pinned mailbox below
    unsigned long long *h_mail;    // pinned, 64 bytes: stats u64[4] | err i32
    // resident mode (psk_craft_host_tick_resident): the working state and the per-env byte outputs
    // of the whole batch stay on the device; allocated on first use
    uint8_t *r_grid, *r_agent, *r_action, *r_expert, *r_done, *r_success;
    cudaEvent_t ev_in, ev_chunk[PSK_HOST_STREAMS];
    bool resident_ready;
    // PSK_FEATURES_F32_WIRE_U8: pinned u8 landing zone for the whole batch, one event per chunk,
    // host threads that widen to the caller's f32 buffer; allocated on first use
    uint8_t *h_wire;
    cudaEvent_t *ev_wire;
    int64_t n_wire_events;
    PskWidenPool *pool;
    int host_threads;           // psk_craft_host_set_threads; 0 = PskWidenPool::default_threads()
    // PSK_FEATURES_F32_WIRE_U8, split frame: the LAST `wire_direct` chunks of a call cross PCIe as f32
    // straight into the caller's (pinned) buffer while the host threads are still widening the byte
    // chunks that landed before them.  wire_direct_fixed < 0: the count follows the two measured
    // rates (per-chunk PCIe time, per-chunk widening time) from call to call.
    int wire_direct, wire_direct_fixed;
    double wire_pcie_us, wire_widen_us;     // smoothed per-u8-chunk times, 0 = not measured yet
    cudaEvent_t ev_end;
    // small batches: the fused kernel reads the actions from and writes every output into the caller's
    // pinned buffers itself (unified addressing) — one launch, one 40-byte copy, one synchronize
    int64_t zerocopy_max;               // env PSK_HOST_ZEROCOPY_MAX, psk_craft_host_set_zerocopy_max
};

static inline double now_us() {
    return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

#define CK(x)                                   \
    do {                                        \
        if ((x) != cudaSuccess) return PSK_ERR_CUDA; \
    } while (0)

// A context belongs to the device that was current when it was created; calls made while another
// device is current switch to it for their duration.
struct DeviceScope {
    int prev = -1;
    explicit DeviceScope(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev); else prev = -1;
    }
    ~DeviceScope() {
        if (prev >= 0) cudaSetDevice(prev);
    }
};

extern "C" {

void *psk_host_alloc(size_t bytes) {
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}

void psk_host_free(void *p) {
    if (p) cudaFreeHost(p);
}

static int host_ctx_alloc(psk_craft_host_ctx *c) {
    CK(cudaGetDevice(&c->device));
    for (int i = 0; i < PSK_HOST_STREAMS; i++) {
        CK(cudaStreamCreateWithFlags(&c->streams[i], cudaStreamNonBlocking));
        CK(cudaMalloc(&c->d_grid[i], (size_t)c->chunk * c->cell_stride));
        CK(cudaMalloc(&c->d_agent[i], (size_t)c->chunk * PSK_AGENT_BYTES));
        CK(cudaMalloc(&c->d_action[i], (size_t)c->chunk));
        CK(cudaMalloc(&c->d_expert[i], (size_t)c->chunk));
        CK(cudaMalloc(&c->d_done[i], (size_t)c->chunk));
        CK(cudaMalloc(&c->d_success[i], (size_t)c->chunk));
        CK(cudaMalloc(&c->d_feat[i], (size_t)c->chunk * c->nf * sizeof(float)));
    }
    CK(cudaMalloc(&c->d_stats, 64));
    CK(cudaMemset(c->d_stats, 0, 64));
    c->d_err = reinterpret_cast<int32_t *>(c->d_stats + 4);
    CK(cudaHostAlloc(reinterpret_cast<void **>(&c->h_mail), 64, cudaHostAllocDefault));
    return PSK_OK;
}

void psk_craft_host_destroy(psk_craft_host_ctx *c);

int psk_craft_host_create(const psk_craft_tables *t, int64_t max_envs, int64_t chunk_envs,
                          psk_craft_host_ctx **out) {
    if (!t || !out || max_envs <= 0) return PSK_ERR_BADARG;
    if (!psk_craft_supported(t)) return PSK_ERR_UNSUPPORTED;
    psk_craft_host_ctx *c = new (std::nothrow) psk_craft_host_ctx();
    if (!c) return PSK_ERR_BADARG;
    memset(c, 0, sizeof(*c));
    c->tables = *t;
    c->max_envs = max_envs;
    if (chunk_envs <= 0) chunk_envs = 16384;
    if (chunk_envs > max_envs) chunk_envs = max_envs;
    c->chunk = (chunk_envs + 127) / 128 * 128;
    c->cell_stride = ((t->width * t->height + 63) / 64) * 64;
    c->nf = psk_craft_n_features(t);
    c->wire_direct_fixed = -1;
    if (const char *e = getenv("PSK_WIRE_DIRECT")) c->wire_direct_fixed = atoi(e);
    c->zerocopy_max = 2048;
    if (const char *e = getenv("PSK_HOST_ZEROCOPY_MAX")) c->zerocopy_max = atoll(e);
    const int rc = host_ctx_alloc(c);
    if (rc != PSK_OK) {             // release whatever was allocated before the failure
        psk_craft_host_destroy(c);
        return rc;
    }
    *out = c;
    return PSK_OK;
}

void psk_craft_host_destroy(psk_craft_host_ctx *c) {
    if (!c) return;
    DeviceScope scope(c->device);
    for (int i = 0; i < PSK_HOST_STREAMS; i++) {
        if (c->streams[i]) cudaStreamSynchronize(c->streams[i]);
        cudaFree(c->d_grid[i]); cudaFree(c->d_agent[i]); cudaFree(c->d_action[i]);
        cudaFree(c->d_expert[i]); cudaFree(c->d_done[i]); cudaFree(c->d_success[i]);
        cudaFree(c->d_feat[i]);
        if (c->streams[i]) cudaStreamDestroy(c->streams[i]);
    }
    cudaFree(c->d_scen_grid); cudaFree(c->d_init_agent); cudaFree(c->d_scen_idx);
    cudaFree(c->d_stats);
    if (c->h_mail) cudaFreeHost(c->h_mail);
    cudaFree(c->r_grid); cudaFree(c->r_agent); cudaFree(c->r_action);
    cudaFree(c->r_expert); cudaFree(c->r_done); cudaFree(c->r_success);
    if (c->ev_in) cudaEventDestroy(c->ev_in);
    if (c->ev_end) cudaEventDestroy(c->ev_end);
    for (int i = 0; i < PSK_HOST_STREAMS; i++)
        if (c->ev_chunk[i]) cudaEventDestroy(c->ev_chunk[i]);
    delete c->pool;
    if (c->h_wire) cudaFreeHost(c->h_wire);
    for (int64_t i = 0; i < c->n_wire_events; i++) cudaEventDestroy(c->ev_wire[i]);
    delete[] c->ev_wire;
    delete c;
}

int psk_craft_host_set_episodes(psk_craft_host_ctx *c, const uint8_t *host_scen_grid,
                                int64_t n_scen, const int32_t *host_scen_idx,
                                const uint8_t *host_init_agent, int64_t n) {
    if (!c || !host_scen_grid || !host_scen_idx || !host_init_agent || n <= 0 || n_scen <= 0 ||
        n > c->max_envs)
        return PSK_ERR_BADARG;
    DeviceScope scope(c->device);
    cudaFree(c->d_scen_grid); cudaFree(c->d_init_agent); cudaFree(c->d_scen_idx);
    c->d_scen_grid = nullptr; c->d_init_agent = nullptr; c->d_scen_idx = nullptr;
    CK(cudaMalloc(&c->d_scen_grid, (size_t)n_scen * c->cell_stride));
    CK(cudaMalloc(&c->d_scen_idx, (size_t)n * sizeof(int32_t)));
    CK(cudaMalloc(&c->d_init_agent, (size_t)n * PSK_AGENT_BYTES));
    CK(cudaMemcpy(c->d_scen_grid, host_scen_grid, (size_t)n_scen * c->cell_stride, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(c->d_scen_idx, host_scen_idx, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(c->d_init_agent, host_init_agent, (size_t)n * PSK_AGENT_BYTES, cudaMemcpyHostToDevice));
    c->n_scen = n_scen;
    c->n_eps = n;
    return PSK_OK;
}

int psk_craft_host_tick(psk_craft_host_ctx *c, uint8_t *host_grid, uint8_t *host_agent,
                        const uint8_t *host_action_in, float *host_features,
                        uint8_t *host_expert, uint8_t *host_done, uint8_t *host_success,
                        int64_t n, unsigned long long *host_stats, int32_t *host_err_flags) {
    if (!c || !host_grid || !host_agent || !host_expert || n < 0 || n > c->n_eps)
        return PSK_ERR_BADARG;
    DeviceScope scope(c->device);
    const int cs = c->cell_stride;
    int k = 0;
    for (int64_t off = 0; off < n; off += c->chunk, k++) {
        const int s = k % PSK_HOST_STREAMS;
        const int64_t m = (n - off) < c->chunk ? (n - off) : c->chunk;
        cudaStream_t st = c->streams[s];
        CK(cudaMemcpyAsync(c->d_grid[s], host_grid + off * cs, (size_t)m * cs, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(c->d_agent[s], host_agent + off * PSK_AGENT_BYTES, (size_t)m * PSK_AGENT_BYTES,
                           cudaMemcpyHostToDevice, st));
        if (host_action_in)
            CK(cudaMemcpyAsync(c->d_action[s], host_action_in + off, (size_t)m, cudaMemcpyHostToDevice, st));
        psk_craft_state state = {c->d_grid[s], c->d_agent[s], m, cs, 0};
        psk_craft_episodes ep = {c->d_scen_grid, c->d_scen_idx + off, c->d_init_agent + off * PSK_AGENT_BYTES};
        int rc = psk_craft_tick(&c->tables, state, ep, host_action_in ? c->d_action[s] : nullptr,
                                host_features ? c->d_feat[s] : nullptr, c->d_expert[s],
                                c->d_done[s], c->d_success[s], c->d_stats, c->d_err, 1, st);
        if (rc) return rc;
        if (host_features)
            CK(cudaMemcpyAsync(host_features + off * c->nf, c->d_feat[s], (size_t)m * c->nf * sizeof(float),
                               cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(host_expert + off, c->d_expert[s], (size_t)m, cudaMemcpyDeviceToHost, st));
        if (host_done) CK(cudaMemcpyAsync(host_done + off, c->d_done[s], (size_t)m, cudaMemcpyDeviceToHost, st));
        if (host_success)
            CK(cudaMemcpyAsync(host_success + off, c->d_success[s], (size_t)m, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(host_grid + off * cs, c->d_grid[s], (size_t)m * cs, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(host_agent + off * PSK_AGENT_BYTES, c->d_agent[s], (size_t)m * PSK_AGENT_BYTES,
                           cudaMemcpyDeviceToHost, st));
    }
    for (int i = 0; i < PSK_HOST_STREAMS; i++) CK(cudaStreamSynchronize(c->streams[i]));
    if (host_stats) CK(cudaMemcpy(host_stats, c->d_stats, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    if (host_err_flags) {
        CK(cudaMemcpy(host_err_flags, c->d_err, sizeof(int32_t), cudaMemcpyDeviceToHost));
        if (*host_err_flags) CK(cudaMemset(c->d_err, 0, sizeof(int32_t)));
    }
    return PSK_OK;
}

// ---------------------------------------------------------------------------------------------
// Resident mode: what crosses PCIe per tick is only what a rollout's caller consumes — the
// actions it chose go up, feature rows / teacher actions / done / success come down; the
// environments stay in HBM (fetch them with psk_craft_host_get_state when .pos / .inventory are
// needed, e.g. for the language teachers' describe()).
static int resident_alloc(psk_craft_host_ctx *c) {
    if (c->resident_ready) return PSK_OK;
    const size_t n = (size_t)c->max_envs;
    CK(cudaMalloc(&c->r_grid, n * c->cell_stride));
    CK(cudaMalloc(&c->r_agent, n * PSK_AGENT_BYTES));
    CK(cudaMalloc(&c->r_action, n));
    CK(cudaMalloc(&c->r_expert, n));
    CK(cudaMalloc(&c->r_done, n));
    CK(cudaMalloc(&c->r_success, n));
    CK(cudaEventCreateWithFlags(&c->ev_in, cudaEventDisableTiming));
    CK(cudaEventCreateWithFlags(&c->ev_end, cudaEventDisableTiming));
    for (int i = 0; i < PSK_HOST_STREAMS; i++)
        CK(cudaEventCreateWithFlags(&c->ev_chunk[i], cudaEventDisableTiming));
    c->resident_ready = true;
    return PSK_OK;
}

int psk_craft_host_reset(psk_craft_host_ctx *c, int64_t n) {
    if (!c || n < 0 || n > c->n_eps) return PSK_ERR_BADARG;
    DeviceScope scope(c->device);
    int rc = resident_alloc(c);
    if (rc) return rc;
    psk_craft_state state = {c->r_grid, c->r_agent, n, c->cell_stride, 0};
    psk_craft_episodes ep = {c->d_scen_grid, c->d_scen_idx, c->d_init_agent};
    rc = psk_craft_reset(state, ep, nullptr, c->streams[0]);
    if (rc) return rc;
    CK(cudaStreamSynchronize(c->streams[0]));
    return PSK_OK;
}

int psk_craft_host_put_state(psk_craft_host_ctx *c, const uint8_t *host_grid,
                             const uint8_t *host_agent, int64_t n) {
    if (!c || !host_grid || !host_agent || n < 0 || n > c->max_envs) return PSK_ERR_BADARG;
    DeviceScope scope(c->device);
    const int rc = resident_alloc(c);
    if (rc) return rc;
    CK(cudaMemcpyAsync(c->r_grid, host_grid, (size_t)n * c->cell_stride, cudaMemcpyHostToDevice, c->streams[0]));
    CK(cudaMemcpyAsync(c->r_agent, host_agent, (size_t)n * PSK_AGENT_BYTES, cudaMemcpyHostToDevice, c->streams[0]));
    CK(cudaStreamSynchronize(c->streams[0]));
    return PSK_OK;
}

int psk_craft_host_get_state(psk_craft_host_ctx *c, uint8_t *host_grid, uint8_t *host_agent, int64_t n) {
    if (!c || !c->resident_ready || n < 0 || n > c->max_envs) return PSK_ERR_BADARG;
    DeviceScope scope(c->device);
    if (host_grid)
        CK(cudaMemcpyAsync(host_grid, c->r_grid, (size_t)n * c->cell_stride, cudaMemcpyDeviceToHost, c->streams[0]));
    if (host_agent)
        CK(cudaMemcpyAsync(host_agent, c->r_agent, (size_t)n * PSK_AGENT_BYTES, cudaMemcpyDeviceToHost, c->streams[0]));
    CK(cudaStreamSynchronize(c->streams[0]));
    return PSK_OK;
}

static int wire_alloc(psk_craft_host_ctx *c) {
    const int64_t chunks = (c->max_envs + c->chunk - 1) / c->chunk;
    const size_t frame = (size_t)c->max_envs * c->nf;
    if (!c->h_wire) CK(cudaHostAlloc(reinterpret_cast<void **>(&c->h_wire), frame, cudaHostAllocDefault));
    if (!c->ev_wire) {
        c->ev_wire = new (std::nothrow) cudaEvent_t[chunks];
        if (!c->ev_wire) return PSK_ERR_BADARG;
    }
    for (; c->n_wire_events < chunks; c->n_wire_events++)
        CK(cudaEventCreateWithFlags(&c->ev_wire[c->n_wire_events], cudaEventDisableTiming));
    if (!c->pool) {
        const int th = c->host_threads > 0 ? c->host_threads - 1 : PskWidenPool::default_threads();
        c->pool = new (std::nothrow) PskWidenPool(th, frame / PSK_WIDEN_BLOCK + (size_t)chunks + 8);
    }
    return c->pool ? PSK_OK : PSK_ERR_BADARG;
}

// How many trailing chunks of this call go down as f32 (split frame, see the context struct).
static int wire_direct_chunks(psk_craft_host_ctx *c, const void *host_features, int chunks) {
    int d = c->wire_direct_fixed >= 0 ? c->wire_direct_fixed : c->wire_direct;
    if (d > chunks) d = chunks;
    if (d < 0) d = 0;
    if (d > 0) {        // an f32 chunk is copied by the DMA engine: only into pinned / registered memory
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, host_features) != cudaSuccess || at.type != cudaMemoryTypeHost) {
            cudaGetLastError();
            d = 0;
        }
    }
    return d;
}

// After a call with `d` of `chunks` chunks sent as f32: PCIe finished `t_pcie` us and the widening
// `t_widen` us after the call started; the rule itself is psk_wire_split_next (psk_hostcpu.cpp).
static void wire_direct_update(psk_craft_host_ctx *c, int chunks, int d, double t_pcie, double t_widen) {
    if (c->wire_direct_fixed >= 0 || chunks < 2 || d >= chunks) return;     // nothing to balance
    c->wire_direct = psk_wire_split_next(chunks, d, t_pcie, t_widen, &c->wire_pcie_us, &c->wire_widen_us);
}

// The running statistics and the error flags (d_stats: u64[4] | i32) into the pinned mailbox, as a
// kernel behind the tick on the same stream: a 40-byte cudaMemcpyAsync costs 10 us of copy-engine
// latency at this size (17 -> 27 us per call), five 8-byte stores over PCIe cost 3.
__global__ void mail_publish_kernel(const unsigned long long *__restrict__ d_stats,
                                    unsigned long long *__restrict__ mail) {
    if (threadIdx.x < 5) mail[threadIdx.x] = d_stats[threadIdx.x];
}

// Device alias of a pinned host pointer, NULL when the memory is pageable.  Looked up on every call
// (well under a microsecond): an address can change hands between calls.
static void *zc_alias(const void *host) {
    if (!host) return nullptr;
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, host) == cudaSuccess && at.type == cudaMemoryTypeHost)
        return at.devicePointer;
    cudaGetLastError();
    return nullptr;
}

// One launch for the whole call.  Returns PSK_ERR_UNSUPPORTED when a buffer is not pinned (the caller
// of this helper then takes the copy-engine route).
static int tick_resident_zerocopy(psk_craft_host_ctx *c, const uint8_t *host_action_in, void *host_features,
                                  int32_t feature_format, int32_t advance_first, uint8_t *host_expert,
                                  uint8_t *host_done, uint8_t *host_success, int64_t n,
                                  unsigned long long *host_stats, int32_t *host_err_flags) {
    const uint8_t *act = static_cast<const uint8_t *>(zc_alias(host_action_in));
    void *feat = zc_alias(host_features);
    uint8_t *expert = static_cast<uint8_t *>(zc_alias(host_expert));
    uint8_t *done = static_cast<uint8_t *>(zc_alias(host_done));
    uint8_t *success = static_cast<uint8_t *>(zc_alias(host_success));
    if ((host_action_in && !act) || (host_features && !feat) || !expert || (host_done && !done) ||
        (host_success && !success))
        return PSK_ERR_UNSUPPORTED;
    if (feature_format == PSK_FEATURES_NONE) feat = nullptr;
    cudaStream_t s0 = c->streams[0];
    psk_craft_state state = {c->r_grid, c->r_agent, n, c->cell_stride, 0};
    psk_craft_episodes ep = {c->d_scen_grid, c->d_scen_idx, c->d_init_agent};
    const int mode = advance_first ? PSK_TICK_ADVANCE_FIRST : PSK_TICK_FUSED;
    int rc;
    if (feature_format == PSK_FEATURES_U8)
        rc = psk_craft_tick_u8(&c->tables, state, ep, act, static_cast<uint8_t *>(feat), expert,
                               done ? done : c->r_done, success ? success : c->r_success, c->d_stats, c->d_err,
                               mode, s0);
    else        // PSK_FEATURES_F32 and PSK_FEATURES_F32_WIRE_U8 promise the same f32 host frame
        rc = psk_craft_tick(&c->tables, state, ep, act, static_cast<float *>(feat), expert,
                            done ? done : c->r_done, success ? success : c->r_success, c->d_stats, c->d_err,
                            mode, s0);
    if (rc) return rc;
    if (host_stats || host_err_flags) {
        void *mail = zc_alias(c->h_mail);
        if (mail) {
            mail_publish_kernel<<<1, 32, 0, s0>>>(c->d_stats, static_cast<unsigned long long *>(mail));
            CK(cudaGetLastError());
        } else {
            CK(cudaMemcpyAsync(c->h_mail, c->d_stats, 40, cudaMemcpyDeviceToHost, s0));
        }
    }
    CK(cudaStreamSynchronize(s0));
    if (host_stats) memcpy(host_stats, c->h_mail, 4 * sizeof(unsigned long long));
    if (host_err_flags) {
        memcpy(host_err_flags, c->h_mail + 4, sizeof(int32_t));
        if (*host_err_flags) CK(cudaMemset(c->d_err, 0, sizeof(int32_t)));
    }
    return PSK_OK;
}

int psk_craft_host_tick_resident(psk_craft_host_ctx *c, const uint8_t *host_action_in,
                                 void *host_features, int32_t feature_format, int32_t advance_first,
                                 uint8_t *host_expert, uint8_t *host_done, uint8_t *host_success,
                                 int64_t n, unsigned long long *host_stats, int32_t *host_err_flags) {
    if (!c || !c->resident_ready || !host_expert || n < 0 || n > c->n_eps) return PSK_ERR_BADARG;
    if (feature_format != PSK_FEATURES_NONE && feature_format != PSK_FEATURES_F32 &&
        feature_format != PSK_FEATURES_U8 && feature_format != PSK_FEATURES_F32_WIRE_U8)
        return PSK_ERR_BADARG;
    if (!host_features) feature_format = PSK_FEATURES_NONE;
    DeviceScope scope(c->device);
    if (n > 0 && n <= c->zerocopy_max && psk::craft_fused_built(&c->tables)) {   // fused kernel only
        const int rc = tick_resident_zerocopy(c, host_action_in, host_features, feature_format, advance_first,
                                              host_expert, host_done, host_success, n, host_stats, host_err_flags);
        if (rc != PSK_ERR_UNSUPPORTED) return rc;
    }
    const bool wire = feature_format == PSK_FEATURES_F32_WIRE_U8;
    const int chunks = static_cast<int>((n + c->chunk - 1) / c->chunk);
    int direct = 0;
    if (wire) {
        const int rc = wire_alloc(c);
        if (rc) return rc;
        direct = wire_direct_chunks(c, host_features, chunks);
    }
    const double t_start = wire ? now_us() : 0.0;
    const int cs = c->cell_stride;
    cudaStream_t s0 = c->streams[0];
    if (host_action_in) {       // one copy for the whole batch, the other streams wait for it
        CK(cudaMemcpyAsync(c->r_action, host_action_in, (size_t)n, cudaMemcpyHostToDevice, s0));
        CK(cudaEventRecord(c->ev_in, s0));
        for (int i = 1; i < PSK_HOST_STREAMS; i++) CK(cudaStreamWaitEvent(c->streams[i], c->ev_in, 0));
    }
    int k = 0;
    for (int64_t off = 0; off < n; off += c->chunk, k++) {
        const int s = k % PSK_HOST_STREAMS;
        const int64_t m = (n - off) < c->chunk ? (n - off) : c->chunk;
        cudaStream_t st = c->streams[s];
        psk_craft_state state = {c->r_grid + off * cs, c->r_agent + off * PSK_AGENT_BYTES, m, cs, 0};
        psk_craft_episodes ep = {c->d_scen_grid, c->d_scen_idx + off, c->d_init_agent + off * PSK_AGENT_BYTES};
        const uint8_t *act = host_action_in ? c->r_action + off : nullptr;
        int rc;
        const int mode = advance_first ? PSK_TICK_ADVANCE_FIRST : PSK_TICK_FUSED;
        // this chunk's frame format on the wire: bytes (compact frame, or to be widened here), or f32
        const bool bytes = feature_format == PSK_FEATURES_U8 || (wire && k < chunks - direct);
        const size_t fsz = bytes ? 1 : 4;
        uint8_t *const landing = (wire && bytes) ? c->h_wire : static_cast<uint8_t *>(host_features);
        if (bytes) {
            // compact frame: the fused kernel writes its u8 tile as it is
            rc = psk_craft_tick_u8(&c->tables, state, ep, act, reinterpret_cast<uint8_t *>(c->d_feat[s]),
                                   c->r_expert + off, c->r_done + off, c->r_success + off, c->d_stats,
                                   c->d_err, mode, st);
        } else {
            rc = psk_craft_tick(&c->tables, state, ep, act,
                                feature_format != PSK_FEATURES_NONE ? c->d_feat[s] : nullptr,
                                c->r_expert + off, c->r_done + off, c->r_success + off, c->d_stats,
                                c->d_err, mode, st);
        }
        if (rc) return rc;
        if (feature_format != PSK_FEATURES_NONE)
            CK(cudaMemcpyAsync(landing + (size_t)off * c->nf * fsz, c->d_feat[s],
                               (size_t)m * c->nf * fsz, cudaMemcpyDeviceToHost, st));
        if (wire && bytes) CK(cudaEventRecord(c->ev_wire[k], st));
    }
    // the per-env byte outputs of the whole batch: one copy each, after every chunk's kernel
    for (int i = 1; i < PSK_HOST_STREAMS; i++) {
        CK(cudaEventRecord(c->ev_chunk[i], c->streams[i]));
        CK(cudaStreamWaitEvent(s0, c->ev_chunk[i], 0));
    }
    CK(cudaMemcpyAsync(host_expert, c->r_expert, (size_t)n, cudaMemcpyDeviceToHost, s0));
    if (host_done) CK(cudaMemcpyAsync(host_done, c->r_done, (size_t)n, cudaMemcpyDeviceToHost, s0));
    if (host_success) CK(cudaMemcpyAsync(host_success, c->r_success, (size_t)n, cudaMemcpyDeviceToHost, s0));
    if (host_stats || host_err_flags)       // one 40-byte copy into pinned memory (pageable targets would stage)
        CK(cudaMemcpyAsync(c->h_mail, c->d_stats, 40, cudaMemcpyDeviceToHost, s0));
    if (wire) {
        CK(cudaEventRecord(c->ev_end, s0));     // s0 waited for every stream: the last byte of the call
        // widen chunk k on the host threads as soon as its bytes have landed, while chunks k+1..
        // are still being computed and copied (the f32 chunks at the end need no host work)
        int done_chunks = 0;
        cudaError_t err = cudaSuccess;
        for (int64_t off = 0; done_chunks < chunks - direct && err == cudaSuccess; off += c->chunk, done_chunks++) {
            const int64_t m = (n - off) < c->chunk ? (n - off) : c->chunk;
            err = cudaEventSynchronize(c->ev_wire[done_chunks]);
            if (err == cudaSuccess)
                c->pool->submit(c->h_wire + (size_t)off * c->nf,
                                static_cast<float *>(host_features) + (size_t)off * c->nf,
                                (size_t)m * c->nf, PSK_WIDEN_BLOCK);
        }
        // help with the widening; note when the wire went quiet and when the widening did
        double t_pcie = 0.0;
        while (!c->pool->idle()) {
            if (t_pcie == 0.0 && cudaEventQuery(c->ev_end) == cudaSuccess) t_pcie = now_us() - t_start;
            c->pool->help();
        }
        const double t_widen = now_us() - t_start;
        cudaGetLastError();                     // cudaErrorNotReady from the queries is not an error
        if (err != cudaSuccess) return PSK_ERR_CUDA;
        for (int i = 0; i < PSK_HOST_STREAMS; i++) CK(cudaStreamSynchronize(c->streams[i]));
        if (t_pcie == 0.0) t_pcie = now_us() - t_start;
        wire_direct_update(c, chunks, direct, t_pcie, t_widen);
    } else {
        for (int i = 0; i < PSK_HOST_STREAMS; i++) CK(cudaStreamSynchronize(c->streams[i]));
    }
    if (host_stats) memcpy(host_stats, c->h_mail, 4 * sizeof(unsigned long long));
    if (host_err_flags) {
        memcpy(host_err_flags, c->h_mail + 4, sizeof(int32_t));
        if (*host_err_flags) CK(cudaMemset(c->d_err, 0, sizeof(int32_t)));
    }
    return PSK_OK;
}

int psk_craft_host_set_zerocopy_max(psk_craft_host_ctx *c, int64_t max_envs) {
    if (!c || max_envs < 0) return PSK_ERR_BADARG;
    c->zerocopy_max = max_envs;
    return PSK_OK;
}

int psk_craft_host_wire_direct(const psk_craft_host_ctx *c) {
    if (!c) return 0;
    return c->wire_direct_fixed >= 0 ? c->wire_direct_fixed : c->wire_direct;
}

int psk_craft_host_set_wire_direct(psk_craft_host_ctx *c, int32_t chunks) {
    if (!c || chunks < -1) return PSK_ERR_BADARG;
    c->wire_direct_fixed = chunks;
    if (chunks < 0) c->wire_direct = 0, c->wire_pcie_us = c->wire_widen_us = 0.0;
    return PSK_OK;
}

int psk_craft_host_threads(const psk_craft_host_ctx *c) {
    return c && c->pool ? c->pool->threads() + 1 : 0;
}

int psk_craft_host_set_threads(psk_craft_host_ctx *c, int32_t threads) {
    if (!c || threads < 1 || threads > 256) return PSK_ERR_BADARG;
    if (c->pool && c->pool->threads() + 1 != threads) {     // between calls: no job is outstanding
        delete c->pool;
        c->pool = nullptr;
    }
    c->host_threads = threads;
    return PSK_OK;
}

}  // extern "C"
