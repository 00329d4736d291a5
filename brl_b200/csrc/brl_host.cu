// brl_host.cu -- host-buffer convenience layer over the stream-first ops: the
// library owns the device-resident packed state, the deal table replica and the
// output staging; callers pass HOST pointers and the copies are part of the call.
// This is what a non-JAX host (or bench.py's `e2e` leg) calls.
#include <cuda.h>

#include <mutex>
#include <new>
#include <unordered_map>

#include "common.h"

struct BrlEnv {
    uint32_t magic;
    int64_t n, env_offset;
    int32_t n_deals, flags;
    uint64_t seed;
    uint32_t step;
    cudaStream_t stream;
    cudaStream_t s_in, s_out;          // copy streams of the pipelined rollout
    cudaEvent_t ev_in[8], ev_k[8];     // per-chunk: uniforms landed / kernel finished
    uint8_t* d_table;
    void* d_state;
    int32_t* d_action;
    uint64_t* d_keys;
    void* d_obs;
    uint8_t* d_mask;
    float* d_rewards;
    uint8_t* d_term;
    int8_t* d_cur;
    size_t obs_row_bytes;
    // rollout trajectory (allocated on first brl_env_rollout_host)
    int32_t traj_k;
    void* t_obs;
    uint8_t* t_mask;
    float* t_rewards;
    uint8_t* t_term;
    int8_t* t_cur;
    int32_t* t_action;
    uint32_t* t_uniforms;
    unsigned long long* d_stats;
    // pipelined rollout (brl_env_rollout_host_async): BRL_ENV_PIPELINE_DEPTH staging slots + events
    int32_t a_k;
    int64_t a_calls;
    float* a_rewards[BRL_ENV_PIPELINE_DEPTH];
    uint8_t* a_term[BRL_ENV_PIPELINE_DEPTH];
    uint32_t* a_uniforms[BRL_ENV_PIPELINE_DEPTH];
    int16_t* a_result[BRL_ENV_PIPELINE_DEPTH];
    unsigned long long* a_stats[BRL_ENV_PIPELINE_DEPTH];
    cudaEvent_t a_in[BRL_ENV_PIPELINE_DEPTH], a_kernel[BRL_ENV_PIPELINE_DEPTH], a_done[BRL_ENV_PIPELINE_DEPTH];
};

namespace {
constexpr uint32_t kMagic = 0x42524C45u;  // "BRLE"

bool ok(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return true;
    brl::fail(BRL_E_LAUNCH, "%s: %s", what, cudaGetErrorString(e));
    return false;
}

BrlParams params_of(const BrlEnv* env, int32_t extra_flags) {
    BrlParams p = {};
    p.n_envs = env->n;
    p.env_offset = env->env_offset;
    p.state_stride = env->n;
    p.seed = env->seed;
    p.n_deals = env->n_deals;
    p.flags = env->flags | extra_flags;
    p.step = env->step;
    p.illegal_penalty = -1.0f;
    p.illegal_bonus = 1.0f;
    return p;
}

int32_t copy_out(BrlEnv* env, void* obs, uint8_t* mask, float* rewards, uint8_t* terminated, int8_t* current_player) {
    cudaStream_t s = env->stream;
    const size_t n = (size_t)env->n;
    if (obs && !ok(cudaMemcpyAsync(obs, env->d_obs, n * env->obs_row_bytes, cudaMemcpyDeviceToHost, s), "D2H obs")) return BRL_E_LAUNCH;
    if (mask && !ok(cudaMemcpyAsync(mask, env->d_mask, n * BRL_NUM_ACTIONS, cudaMemcpyDeviceToHost, s), "D2H mask")) return BRL_E_LAUNCH;
    if (rewards && !ok(cudaMemcpyAsync(rewards, env->d_rewards, n * 16, cudaMemcpyDeviceToHost, s), "D2H rewards")) return BRL_E_LAUNCH;
    if (terminated && !ok(cudaMemcpyAsync(terminated, env->d_term, n, cudaMemcpyDeviceToHost, s), "D2H terminated")) return BRL_E_LAUNCH;
    if (current_player && !ok(cudaMemcpyAsync(current_player, env->d_cur, n, cudaMemcpyDeviceToHost, s), "D2H current_player")) return BRL_E_LAUNCH;
    if (!ok(cudaStreamSynchronize(s), "stream sync")) return BRL_E_LAUNCH;
    return BRL_OK;
}

// ---- compressible trajectory memory (CUDA virtual-memory API) ---------------------------------------------------------------
// The driver's entry points are fetched through the runtime, as encode_fn() does for cuTensorMapEncodeTiled: no -lcuda.
struct Vmm {
    decltype(&::cuDeviceGet) device_get;
    decltype(&::cuDeviceGetAttribute) attribute;
    decltype(&::cuMemGetAllocationGranularity) granularity;
    decltype(&::cuMemAddressReserve) reserve;
    decltype(&::cuMemAddressFree) address_free;
    decltype(&::cuMemCreate) create;
    decltype(&::cuMemGetAllocationPropertiesFromHandle) properties;
    decltype(&::cuMemMap) map;
    decltype(&::cuMemSetAccess) set_access;
    decltype(&::cuMemUnmap) unmap;
    decltype(&::cuMemRelease) release;
    bool loaded;
};

template <class F>
bool entry_point(const char* name, F* fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint(name, &p, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) p = nullptr;
    *fn = reinterpret_cast<F>(p);
    return p != nullptr;
}

const Vmm& vmm() {
    static const Vmm v = [] {
        Vmm t = {};
        t.loaded = entry_point("cuDeviceGet", &t.device_get) && entry_point("cuDeviceGetAttribute", &t.attribute) &&
                   entry_point("cuMemGetAllocationGranularity", &t.granularity) &&
                   entry_point("cuMemAddressReserve", &t.reserve) && entry_point("cuMemAddressFree", &t.address_free) &&
                   entry_point("cuMemCreate", &t.create) &&
                   entry_point("cuMemGetAllocationPropertiesFromHandle", &t.properties) && entry_point("cuMemMap", &t.map) &&
                   entry_point("cuMemSetAccess", &t.set_access) && entry_point("cuMemUnmap", &t.unmap) &&
                   entry_point("cuMemRelease", &t.release);
        return t;
    }();
    return v;
}

struct Mapping {
    size_t bytes;
    int device;
};
std::mutex g_map_mutex;
std::unordered_map<CUdeviceptr, Mapping> g_mappings;  // live brl_alloc_compressible ranges

bool cu_ok(CUresult r, const char* what) {
    if (r == CUDA_SUCCESS) return true;
    brl::fail(BRL_E_LAUNCH, "brl_alloc_compressible: %s failed (CUresult %d)", what, (int)r);
    return false;
}

// device property (compressible where the device supports it) and granularity; the caller holds `device` current
bool vmm_prop(int device, CUmemAllocationProp* prop, size_t* gran) {
    const Vmm& v = vmm();
    if (!v.loaded) {
        brl::fail(BRL_E_LAUNCH, "brl_alloc_compressible: the driver lacks the virtual-memory entry points");
        return false;
    }
    CUdevice dev;
    int compression = 0;
    if (!cu_ok(v.device_get(&dev, device), "cuDeviceGet") ||
        !cu_ok(v.attribute(&compression, CU_DEVICE_ATTRIBUTE_GENERIC_COMPRESSION_SUPPORTED, dev), "cuDeviceGetAttribute"))
        return false;
    *prop = {};
    prop->type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop->location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop->location.id = dev;
    prop->allocFlags.compressionType = compression ? CU_MEM_ALLOCATION_COMP_GENERIC : CU_MEM_ALLOCATION_COMP_NONE;
    return cu_ok(v.granularity(gran, prop, CU_MEM_ALLOC_GRANULARITY_RECOMMENDED), "cuMemGetAllocationGranularity");
}

// runs `fn` with `device` current and restores the caller's device afterwards
template <class F>
bool on_device(int device, F fn) {
    int prev = 0;
    if (!ok(cudaGetDevice(&prev), "cudaGetDevice") || !ok(cudaSetDevice(device), "cudaSetDevice")) return false;
    const bool r = fn();
    cudaSetDevice(prev);
    return r;
}
}  // namespace

extern "C" {

size_t brl_round_up_granularity(size_t bytes, size_t granularity) {
    if (granularity == 0) return bytes;
    return (bytes + granularity - 1) / granularity * granularity;
}

int64_t brl_compressible_granularity(int32_t device) {
    size_t gran = 0;
    CUmemAllocationProp prop;
    if (!on_device(device, [&] { return vmm_prop(device, &prop, &gran); })) return -1;
    return (int64_t)gran;
}

void* brl_alloc_compressible(size_t bytes, int32_t device, int32_t* granted) {
    if (granted) *granted = 0;
    if (bytes == 0) {
        brl::fail(BRL_E_OPAQUE, "brl_alloc_compressible: bytes must be > 0");
        return nullptr;
    }
    CUdeviceptr ptr = 0;
    const bool good = on_device(device, [&] {
        const Vmm& v = vmm();
        CUmemAllocationProp prop;
        size_t gran = 0;
        if (!vmm_prop(device, &prop, &gran)) return false;
        const size_t size = brl_round_up_granularity(bytes, gran);
        if (!cu_ok(v.reserve(&ptr, size, gran, 0, 0), "cuMemAddressReserve")) return false;
        CUmemGenericAllocationHandle h = 0;
        if (!cu_ok(v.create(&h, size, &prop, 0), "cuMemCreate")) {
            v.address_free(ptr, size);
            return false;
        }
        // the driver may hand out a plain allocation for a compressible request: report what was granted
        CUmemAllocationProp got = {};
        const bool mapped = cu_ok(v.properties(&got, h), "cuMemGetAllocationPropertiesFromHandle") &&
                            cu_ok(v.map(ptr, size, 0, h, 0), "cuMemMap");
        v.release(h);  // the mapping keeps the memory alive until cuMemUnmap
        CUmemAccessDesc access = {};
        access.location = prop.location;
        access.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
        if (!mapped || !cu_ok(v.set_access(ptr, size, &access, 1), "cuMemSetAccess")) {
            if (mapped) v.unmap(ptr, size);
            v.address_free(ptr, size);
            return false;
        }
        if (granted) *granted = got.allocFlags.compressionType == CU_MEM_ALLOCATION_COMP_GENERIC ? 1 : 0;
        std::lock_guard<std::mutex> lock(g_map_mutex);
        g_mappings[ptr] = Mapping{size, device};
        return true;
    });
    return good ? reinterpret_cast<void*>(ptr) : nullptr;
}

void brl_free_compressible(void* p) {
    if (p == nullptr) return;
    Mapping m;
    {
        std::lock_guard<std::mutex> lock(g_map_mutex);
        auto it = g_mappings.find(reinterpret_cast<CUdeviceptr>(p));
        if (it == g_mappings.end()) return;
        m = it->second;
        g_mappings.erase(it);
    }
    // unlike cudaFree, unmapping does not wait for the kernels that still write the range
    on_device(m.device, [&] {
        cudaDeviceSynchronize();
        const Vmm& v = vmm();
        v.unmap(reinterpret_cast<CUdeviceptr>(p), m.bytes);
        v.address_free(reinterpret_cast<CUdeviceptr>(p), m.bytes);
        return true;
    });
}

BrlEnv* brl_env_create(int64_t n_envs, int64_t env_offset, const uint8_t* deal_table_host, int32_t n_deals,
                       uint64_t seed, int32_t flags) {
    if (n_envs <= 0 || n_deals <= 0 || deal_table_host == nullptr) {
        brl::fail(BRL_E_OPAQUE, "brl_env_create: n_envs, n_deals must be > 0 and the deal table non-NULL");
        return nullptr;
    }
    BrlEnv* env = new (std::nothrow) BrlEnv();
    if (!env) return nullptr;
    env->magic = kMagic;
    env->n = n_envs;
    env->env_offset = env_offset;
    env->n_deals = n_deals;
    env->flags = flags;
    env->seed = seed;
    env->step = 0;
    env->obs_row_bytes = (flags & BRL_F_OBS_U8) ? BRL_OBS_DIM : ((flags & BRL_F_OBS_BF16) ? BRL_OBS_DIM * 2 : BRL_OBS_DIM * 4);
    const size_t n = (size_t)n_envs;
    bool good = ok(cudaStreamCreateWithFlags(&env->stream, cudaStreamNonBlocking), "stream create") &&
                ok(cudaStreamCreateWithFlags(&env->s_in, cudaStreamNonBlocking), "stream create") &&
                ok(cudaStreamCreateWithFlags(&env->s_out, cudaStreamNonBlocking), "stream create") &&
                ok(cudaMalloc(&env->d_table, (size_t)n_deals * BRL_DEAL_ROW_BYTES), "malloc table") &&
                ok(cudaMalloc(&env->d_state, n * BRL_STATE_BYTES_PER_ENV), "malloc state") &&
                ok(cudaMalloc(&env->d_action, n * 4), "malloc action") &&
                ok(cudaMalloc(&env->d_keys, n * 8), "malloc keys") &&
                ok(cudaMalloc(&env->d_obs, n * env->obs_row_bytes), "malloc obs") &&
                ok(cudaMalloc(&env->d_mask, n * BRL_NUM_ACTIONS), "malloc mask") &&
                ok(cudaMalloc(&env->d_rewards, n * 16), "malloc rewards") &&
                ok(cudaMalloc(&env->d_term, n), "malloc terminated") &&
                ok(cudaMalloc(&env->d_cur, n), "malloc current_player") &&
                ok(cudaMemcpyAsync(env->d_table, deal_table_host, (size_t)n_deals * BRL_DEAL_ROW_BYTES,
                                   cudaMemcpyHostToDevice, env->stream), "H2D table") &&
                ok(cudaStreamSynchronize(env->stream), "sync");
    for (int c = 0; good && c < 8; ++c)
        good = ok(cudaEventCreateWithFlags(&env->ev_in[c], cudaEventDisableTiming), "event create") &&
               ok(cudaEventCreateWithFlags(&env->ev_k[c], cudaEventDisableTiming), "event create");
    if (!good) {
        brl_env_destroy(env);
        return nullptr;
    }
    return env;
}

void brl_env_destroy(BrlEnv* env) {
    if (!env || env->magic != kMagic) return;
    cudaFree(env->d_table); cudaFree(env->d_state); cudaFree(env->d_action); cudaFree(env->d_keys);
    cudaFree(env->d_obs); cudaFree(env->d_mask); cudaFree(env->d_rewards); cudaFree(env->d_term); cudaFree(env->d_cur);
    brl_free_compressible(env->t_obs); brl_free_compressible(env->t_mask);
    cudaFree(env->t_rewards); cudaFree(env->t_term); cudaFree(env->t_cur);
    cudaFree(env->t_action); cudaFree(env->t_uniforms); cudaFree(env->d_stats);
    for (int c = 0; c < 8; ++c) {
        if (env->ev_in[c]) cudaEventDestroy(env->ev_in[c]);
        if (env->ev_k[c]) cudaEventDestroy(env->ev_k[c]);
    }
    for (int c = 0; c < BRL_ENV_PIPELINE_DEPTH; ++c) {
        cudaFree(env->a_rewards[c]); cudaFree(env->a_term[c]); cudaFree(env->a_uniforms[c]); cudaFree(env->a_stats[c]);
        cudaFree(env->a_result[c]);
        if (env->a_in[c]) cudaEventDestroy(env->a_in[c]);
        if (env->a_kernel[c]) cudaEventDestroy(env->a_kernel[c]);
        if (env->a_done[c]) cudaEventDestroy(env->a_done[c]);
    }
    if (env->s_in) cudaStreamDestroy(env->s_in);
    if (env->s_out) cudaStreamDestroy(env->s_out);
    if (env->stream) cudaStreamDestroy(env->stream);
    env->magic = 0;
    delete env;
}

int32_t brl_env_init_host(BrlEnv* env, void* obs, uint8_t* mask, float* rewards, uint8_t* terminated,
                          int8_t* current_player) {
    if (!env || env->magic != kMagic) return brl::fail(BRL_E_HANDLE, "brl_env_init_host: bad handle");
    BrlParams p = params_of(env, 0);
    void* kb[1] = {env->d_keys};
    int32_t rc = brl_make_keys((brl_stream_t)env->stream, kb, &p, sizeof(p));
    if (rc != BRL_OK) return rc;
    void* b[8] = {env->d_keys, env->d_table, env->d_state, env->d_obs, env->d_mask, env->d_rewards, env->d_term, env->d_cur};
    rc = brl_init((brl_stream_t)env->stream, b, &p, sizeof(p));
    if (rc != BRL_OK) return rc;
    env->step = 0;
    return copy_out(env, obs, mask, rewards, terminated, current_player);
}

int32_t brl_env_step_host(BrlEnv* env, const int32_t* action, void* obs, uint8_t* mask, float* rewards,
                          uint8_t* terminated, int8_t* current_player) {
    if (!env || env->magic != kMagic) return brl::fail(BRL_E_HANDLE, "brl_env_step_host: bad handle");
    const bool random = (env->flags & BRL_F_RANDOM_ACTION) != 0;
    if (!random) {
        if (action == nullptr) return brl::fail(BRL_E_BUFFER, "brl_env_step_host: action is NULL");
        if (!ok(cudaMemcpyAsync(env->d_action, action, (size_t)env->n * 4, cudaMemcpyHostToDevice, env->stream), "H2D action"))
            return BRL_E_LAUNCH;
    }
    BrlParams p = params_of(env, 0);
    void* b[10] = {env->d_state, env->d_action, env->d_table, env->d_state, env->d_obs,
                   env->d_mask,  env->d_rewards, env->d_term, env->d_cur, nullptr};
    int32_t rc = brl_step((brl_stream_t)env->stream, b, &p, sizeof(p));
    if (rc != BRL_OK) return rc;
    env->step += 1;
    return copy_out(env, obs, mask, rewards, terminated, current_player);
}

static bool ensure_trajectory(BrlEnv* env, int32_t k) {
    if (env->traj_k >= k) return true;
    brl_free_compressible(env->t_obs); brl_free_compressible(env->t_mask); cudaFree(env->t_rewards); cudaFree(env->t_term); cudaFree(env->t_cur);
    cudaFree(env->t_action); cudaFree(env->t_uniforms);
    env->t_obs = nullptr; env->t_mask = nullptr; env->t_rewards = nullptr; env->t_term = nullptr; env->t_cur = nullptr;
    env->t_action = nullptr; env->t_uniforms = nullptr;
    env->traj_k = 0;
    const size_t rows = (size_t)k * (size_t)env->n;
    // observation and mask rows are mostly zero: compressible memory (where the device has it) shrinks their write-back
    int device = 0;
    bool good = ok(cudaGetDevice(&device), "cudaGetDevice") &&
                (env->t_obs = brl_alloc_compressible(rows * env->obs_row_bytes, device, nullptr)) != nullptr &&
                (env->t_mask = static_cast<uint8_t*>(brl_alloc_compressible(rows * BRL_NUM_ACTIONS, device, nullptr))) != nullptr &&
                ok(cudaMalloc(&env->t_rewards, rows * 16), "malloc traj rewards") &&
                ok(cudaMalloc(&env->t_term, rows), "malloc traj terminated") &&
                ok(cudaMalloc(&env->t_cur, rows), "malloc traj current_player") &&
                ok(cudaMalloc(&env->t_action, rows * 4), "malloc traj action") &&
                ok(cudaMalloc(&env->t_uniforms, rows * 4), "malloc traj uniforms") &&
                (env->d_stats != nullptr || ok(cudaMalloc(&env->d_stats, 32), "malloc stats"));
    if (good) env->traj_k = k;
    return good;
}

int32_t brl_env_rollout_host(BrlEnv* env, int32_t k_steps, const uint32_t* uniforms, float* rewards,
                             uint8_t* terminated, uint64_t* stats) {
    if (!env || env->magic != kMagic) return brl::fail(BRL_E_HANDLE, "brl_env_rollout_host: bad handle");
    if (k_steps <= 0) return brl::fail(BRL_E_OPAQUE, "brl_env_rollout_host: k_steps must be > 0");
    if (!ensure_trajectory(env, k_steps)) return BRL_E_LAUNCH;
    // Zero-copy results: when the caller's result buffers are PINNED host memory (cudaHostAlloc /
    // cudaHostRegister -- torch .pin_memory()), the kernel's writer warps store rewards / terminated
    // straight into them over PCIe (512-byte coalesced bursts per block-step, posted writes that overlap
    // the rest of the step), so there is no device->host copy phase at all: one H2D of the randomness,
    // ONE fused launch, 32 bytes of statistics back.
    {
        auto mapped = [](const void* p, void** dptr) {
            if (p == nullptr) { *dptr = nullptr; return true; }
            cudaPointerAttributes at;
            if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
            if (at.type != cudaMemoryTypeHost || at.devicePointer == nullptr) return false;
            *dptr = at.devicePointer;
            return true;
        };
        void *d_rew = nullptr, *d_term = nullptr;
        if (!(env->flags & BRL_F_HOST_STAGED) && mapped(rewards, &d_rew) && mapped(terminated, &d_term) &&
            (rewards == nullptr || (reinterpret_cast<uintptr_t>(d_rew) & 15u) == 0)) {
            cudaStream_t s = env->stream;
            const size_t rows = (size_t)k_steps * (size_t)env->n;
            if (!ok(cudaMemsetAsync(env->d_stats, 0, 32, s), "memset stats")) return BRL_E_LAUNCH;
            if (uniforms && !ok(cudaMemcpyAsync(env->t_uniforms, uniforms, rows * 4, cudaMemcpyHostToDevice, s), "H2D uniforms"))
                return BRL_E_LAUNCH;
            BrlParams p = params_of(env, 0);
            p.k_steps = k_steps;
            void* b[10] = {env->d_state, env->d_table, env->t_obs, env->t_mask,
                           rewards ? d_rew : (void*)env->t_rewards, terminated ? d_term : (void*)env->t_term,
                           env->t_cur, env->t_action, env->d_stats, uniforms ? (void*)env->t_uniforms : nullptr};
            int32_t rc = brl_rollout_random((brl_stream_t)s, b, &p, sizeof(p));
            if (rc != BRL_OK) return rc;
            env->step += (uint32_t)k_steps;
            if (stats && !ok(cudaMemcpyAsync(stats, env->d_stats, 32, cudaMemcpyDeviceToHost, s), "D2H stats")) return BRL_E_LAUNCH;
            if (!ok(cudaStreamSynchronize(s), "stream sync")) return BRL_E_LAUNCH;
            return BRL_OK;
        }
    }
    // Pageable result buffers: software pipeline over chunks of steps: the H2D copy of chunk c+1's randomness and the
    // D2H copy of chunk c-1's results run on their own streams under chunk c's kernel.
    const int chunks = (k_steps >= 16 && k_steps % 4 == 0 && (env->n * BRL_NUM_ACTIONS * (k_steps / 4)) % 16 == 0) ? 4 : 1;
    const int kc = k_steps / chunks;
    const size_t n = (size_t)env->n, crow = (size_t)kc * n;
    cudaStream_t s = env->stream;
    if (!ok(cudaMemsetAsync(env->d_stats, 0, 32, s), "memset stats")) return BRL_E_LAUNCH;
    if (uniforms)
        for (int c = 0; c < chunks; ++c) {
            if (!ok(cudaMemcpyAsync(env->t_uniforms + c * crow, uniforms + c * crow, crow * 4, cudaMemcpyHostToDevice, env->s_in), "H2D uniforms") ||
                !ok(cudaEventRecord(env->ev_in[c], env->s_in), "event record"))
                return BRL_E_LAUNCH;
        }
    for (int c = 0; c < chunks; ++c) {
        if (uniforms && !ok(cudaStreamWaitEvent(s, env->ev_in[c], 0), "wait event")) return BRL_E_LAUNCH;
        BrlParams p = params_of(env, 0);
        p.k_steps = kc;
        void* b[10] = {env->d_state,
                       env->d_table,
                       static_cast<char*>(env->t_obs) + c * crow * env->obs_row_bytes,
                       env->t_mask + c * crow * BRL_NUM_ACTIONS,
                       env->t_rewards + c * crow * 4,
                       env->t_term + c * crow,
                       env->t_cur + c * crow,
                       env->t_action + c * crow,
                       env->d_stats,
                       uniforms ? (void*)(env->t_uniforms + c * crow) : nullptr};
        int32_t rc = brl_rollout_random((brl_stream_t)s, b, &p, sizeof(p));
        if (rc != BRL_OK) return rc;
        env->step += (uint32_t)kc;
        if (!ok(cudaEventRecord(env->ev_k[c], s), "event record") || !ok(cudaStreamWaitEvent(env->s_out, env->ev_k[c], 0), "wait event"))
            return BRL_E_LAUNCH;
        if (rewards && !ok(cudaMemcpyAsync(rewards + c * crow * 4, env->t_rewards + c * crow * 4, crow * 16, cudaMemcpyDeviceToHost, env->s_out), "D2H rewards"))
            return BRL_E_LAUNCH;
        if (terminated && !ok(cudaMemcpyAsync(terminated + c * crow, env->t_term + c * crow, crow, cudaMemcpyDeviceToHost, env->s_out), "D2H terminated"))
            return BRL_E_LAUNCH;
    }
    if (stats && !ok(cudaMemcpyAsync(stats, env->d_stats, 32, cudaMemcpyDeviceToHost, env->s_out), "D2H stats")) return BRL_E_LAUNCH;
    if (!ok(cudaStreamSynchronize(env->s_out), "stream sync") || !ok(cudaStreamSynchronize(s), "stream sync")) return BRL_E_LAUNCH;
    return BRL_OK;
}

// Shared body of the pipelined calls.  `result16` != NULL selects the compact payload: the kernel writes the f32
// rewards / u8 terminated trajectories into the device-resident trajectory (brl_env_trajectory) and the 2-byte step
// result into the slot's staging buffer, which is all that crosses PCIe; uniforms are u16 or u32 per the env's flags.
static int64_t rollout_async(BrlEnv* env, const char* fn, int32_t k_steps, const void* uniforms, float* rewards,
                             uint8_t* terminated, int16_t* result16, uint64_t* stats) {
    if (!env || env->magic != kMagic) return brl::fail(BRL_E_HANDLE, "%s: bad handle", fn);
    if (k_steps <= 0) return brl::fail(BRL_E_OPAQUE, "%s: k_steps must be > 0", fn);
    if (!ensure_trajectory(env, k_steps)) return BRL_E_LAUNCH;
    const size_t rows = (size_t)k_steps * (size_t)env->n;
    if (env->a_k < k_steps) {
        if (!ok(cudaDeviceSynchronize(), "sync before staging resize")) return BRL_E_LAUNCH;
        for (int c = 0; c < BRL_ENV_PIPELINE_DEPTH; ++c) {
            cudaFree(env->a_rewards[c]); cudaFree(env->a_term[c]); cudaFree(env->a_uniforms[c]); cudaFree(env->a_result[c]);
            env->a_rewards[c] = nullptr; env->a_term[c] = nullptr; env->a_uniforms[c] = nullptr; env->a_result[c] = nullptr;
            bool good = ok(cudaMalloc(&env->a_rewards[c], rows * 16), "malloc staging rewards") &&
                        ok(cudaMalloc(&env->a_term[c], rows), "malloc staging terminated") &&
                        ok(cudaMalloc(&env->a_uniforms[c], rows * 4), "malloc staging uniforms") &&
                        ok(cudaMalloc(&env->a_result[c], rows * 2), "malloc staging result") &&
                        (env->a_stats[c] != nullptr || (ok(cudaMalloc(&env->a_stats[c], 32), "malloc staging stats") &&
                                                        ok(cudaMemset(env->a_stats[c], 0, 32), "memset stats"))) &&
                        (env->a_in[c] != nullptr || ok(cudaEventCreateWithFlags(&env->a_in[c], cudaEventDisableTiming), "event")) &&
                        (env->a_kernel[c] != nullptr || ok(cudaEventCreateWithFlags(&env->a_kernel[c], cudaEventDisableTiming), "event")) &&
                        (env->a_done[c] != nullptr || ok(cudaEventCreateWithFlags(&env->a_done[c], cudaEventDisableTiming), "event"));
            if (!good) return BRL_E_LAUNCH;
        }
        env->a_k = k_steps;
        env->a_calls = 0;
    }
    const int slot = (int)(env->a_calls % BRL_ENV_PIPELINE_DEPTH);
    const bool reuse = env->a_calls >= BRL_ENV_PIPELINE_DEPTH;
    const bool compact = result16 != nullptr;
    const size_t ubytes = (compact && (env->flags & BRL_F_UNIFORM_U16)) ? 2 : 4;
    cudaStream_t s = env->stream;
    if (uniforms) {
        if (reuse && !ok(cudaStreamWaitEvent(env->s_in, env->a_kernel[slot], 0), "wait event")) return BRL_E_LAUNCH;
        if (!ok(cudaMemcpyAsync(env->a_uniforms[slot], uniforms, rows * ubytes, cudaMemcpyHostToDevice, env->s_in), "H2D uniforms") ||
            !ok(cudaEventRecord(env->a_in[slot], env->s_in), "event record") || !ok(cudaStreamWaitEvent(s, env->a_in[slot], 0), "wait event"))
            return BRL_E_LAUNCH;
    }
    // the slot's statistics were re-zeroed on the copy-out stream right after their last D2H (off the kernel stream)
    if (reuse && !ok(cudaStreamWaitEvent(s, env->a_done[slot], 0), "wait event")) return BRL_E_LAUNCH;
    BrlParams p = params_of(env, 0);
    p.k_steps = k_steps;
    p.flags &= ~(BRL_F_UNIFORM_U16 | BRL_F_RESULT_I16);
    if (compact) p.flags |= BRL_F_RESULT_I16 | (ubytes == 2 ? BRL_F_UNIFORM_U16 : 0);
    void* b[11] = {env->d_state, env->d_table, env->t_obs, env->t_mask,
                   compact ? (void*)env->t_rewards : (void*)env->a_rewards[slot],
                   compact ? (void*)env->t_term : (void*)env->a_term[slot],
                   env->t_cur, env->t_action, env->a_stats[slot], uniforms ? (void*)env->a_uniforms[slot] : nullptr,
                   compact ? (void*)env->a_result[slot] : nullptr};
    int32_t rc = brl_rollout_random((brl_stream_t)s, b, &p, sizeof(p));
    if (rc != BRL_OK) return rc;
    env->step += (uint32_t)k_steps;
    if (!ok(cudaEventRecord(env->a_kernel[slot], s), "event record") ||
        !ok(cudaStreamWaitEvent(env->s_out, env->a_kernel[slot], 0), "wait event"))
        return BRL_E_LAUNCH;
    if (compact && !ok(cudaMemcpyAsync(result16, env->a_result[slot], rows * 2, cudaMemcpyDeviceToHost, env->s_out), "D2H result"))
        return BRL_E_LAUNCH;
    if (rewards && !ok(cudaMemcpyAsync(rewards, env->a_rewards[slot], rows * 16, cudaMemcpyDeviceToHost, env->s_out), "D2H rewards"))
        return BRL_E_LAUNCH;
    if (terminated && !ok(cudaMemcpyAsync(terminated, env->a_term[slot], rows, cudaMemcpyDeviceToHost, env->s_out), "D2H terminated"))
        return BRL_E_LAUNCH;
    if (stats && !ok(cudaMemcpyAsync(stats, env->a_stats[slot], 32, cudaMemcpyDeviceToHost, env->s_out), "D2H stats"))
        return BRL_E_LAUNCH;
    if (!ok(cudaMemsetAsync(env->a_stats[slot], 0, 32, env->s_out), "memset stats")) return BRL_E_LAUNCH;
    if (!ok(cudaEventRecord(env->a_done[slot], env->s_out), "event record")) return BRL_E_LAUNCH;
    return ++env->a_calls;
}

// Pipelined form of brl_env_rollout_host: returns as soon as the work is enqueued; call c's H2D runs under
// call c-1's kernel and its D2H under call c+1's kernel (BRL_ENV_PIPELINE_DEPTH staging slots, three streams).
// The host buffers of call c are valid after brl_env_wait(env, ticket_c); at most BRL_ENV_PIPELINE_DEPTH calls
// may be in flight (a deeper submit waits on the device for the slot it reuses).  Three in flight keep the
// GPU fed: with two, the host learns that D2H(c-1) is done only as kernel c ends, too late to enqueue c+1.
int64_t brl_env_rollout_host_async(BrlEnv* env, int32_t k_steps, const uint32_t* uniforms, float* rewards,
                                   uint8_t* terminated, uint64_t* stats) {
    return rollout_async(env, "brl_env_rollout_host_async", k_steps, uniforms, rewards, terminated, nullptr, stats);
}

int64_t brl_env_rollout_host_compact_async(BrlEnv* env, int32_t k_steps, const void* uniforms, int16_t* result,
                                           uint64_t* stats) {
    if (result == nullptr) return brl::fail(BRL_E_BUFFER, "brl_env_rollout_host_compact_async: result is NULL");
    return rollout_async(env, "brl_env_rollout_host_compact_async", k_steps, uniforms, nullptr, nullptr, result, stats);
}

int32_t brl_env_rollout_host_compact(BrlEnv* env, int32_t k_steps, const void* uniforms, int16_t* result, uint64_t* stats) {
    const int64_t t = brl_env_rollout_host_compact_async(env, k_steps, uniforms, result, stats);
    if (t <= 0) return (int32_t)t;
    return brl_env_wait(env, t);
}

// host-side decode of the compact payload into the Env-surface arrays (plain CPU loop over host memory)
void brl_result16_decode(const int16_t* result, int64_t rows, float* rewards, uint8_t* terminated) {
    for (int64_t r = 0; r < rows; ++r) {
        const int32_t w = result[r];
        const float sc = (float)(w >> 1);
        if (rewards) { rewards[4 * r] = sc; rewards[4 * r + 1] = sc; rewards[4 * r + 2] = -sc; rewards[4 * r + 3] = -sc; }
        if (terminated) terminated[r] = (uint8_t)(w & 1);
    }
}

int32_t brl_env_wait(BrlEnv* env, int64_t ticket) {
    if (!env || env->magic != kMagic) return brl::fail(BRL_E_HANDLE, "brl_env_wait: bad handle");
    if (ticket <= 0 || ticket > env->a_calls) return brl::fail(BRL_E_OPAQUE, "brl_env_wait: unknown ticket");
    // if the ticket's slot has been reused since, its event now marks the later call, which queued behind this one on
    // the device: waiting for it is conservative but still correct
    if (!ok(cudaEventSynchronize(env->a_done[(ticket - 1) % BRL_ENV_PIPELINE_DEPTH]), "event sync")) return BRL_E_LAUNCH;
    return BRL_OK;
}

int32_t brl_env_trajectory(BrlEnv* env, void** out) {
    if (!env || env->magic != kMagic) return brl::fail(BRL_E_HANDLE, "brl_env_trajectory: bad handle");
    if (env->traj_k == 0) return brl::fail(BRL_E_HANDLE, "brl_env_trajectory: no rollout has run yet");
    out[0] = env->t_obs; out[1] = env->t_mask; out[2] = env->t_rewards; out[3] = env->t_term; out[4] = env->t_cur;
    out[5] = env->t_action;
    return BRL_OK;
}

}  // extern "C"
