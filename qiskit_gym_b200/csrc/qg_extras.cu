// qg_extras.cu — C-ABI entry points around the fused step: bulk solution read-out, the packed host wire format, NUMA-local pinned
// memory, the cross-GPU end of a sharded search (NCCL, loaded at run time) and the DLPack view of the observation ring.
#include <dlfcn.h>
#include <nccl.h>          // types and prototypes only: the library is dlopen()ed, nothing links against it
#include <sched.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <new>
#include <sstream>

#include "qg_engine_priv.hpp"

using namespace qg;

namespace qg {

// ---- Env::solution for many envs ------------------------------------------------------------------------------------------------
// One thread per env walks its column of the slot-major log sol[slot][env] (consecutive threads read consecutive addresses) and writes its
// env-major row (write_solution, qg_kernels.cuh).
__global__ void k_solutions(const __grid_constant__ DevCfg c, int64_t first, int64_t count, uint32_t* __restrict__ out, int cap, int32_t* __restrict__ len) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const int64_t env = first + i;
    const int n = (int)(c.rec[(size_t)HD_FLAGS * c.Bpad + env] >> FL_LEN_SHIFT);
    if (n > cap) { len[i] = -n; return; }
    len[i] = n;
    write_solution(c, env, n, out + (size_t)i * cap);
}

// ---- per-target winners of a multi-target search --------------------------------------------------------------------------------------
// One warp per group g of `group` consecutive envs: the lanes stride over the group's rollouts, a shuffle reduction finds the largest
// rollout_key (keys are unique, so the result does not depend on the order), and lane 0 writes the key and, if the winner succeeded, its
// Env::solution (len = 0: no success; len = -(length): longer than cap, nothing written).
constexpr int kGroupWarps = 8;
__global__ void __launch_bounds__(kGroupWarps * 32) k_best_grouped(const __grid_constant__ DevCfg c, int64_t group, int64_t num_groups,
                                                                    int64_t* __restrict__ keys, uint32_t* __restrict__ actions, int cap,
                                                                    int32_t* __restrict__ len) {
    const int64_t g = (int64_t)blockIdx.x * kGroupWarps + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (g >= num_groups) return;
    const int64_t e0 = g * group;
    unsigned long long key = 0;
    for (int64_t j = lane; j < group; j += 32) {
        const int64_t env = e0 + j;
        const unsigned long long k = rollout_key((c.rec[(size_t)HD_FLAGS * c.Bpad + env] & FL_SUCCESS) != 0, c.ret[env], c.first_id + env);
        key = k > key ? k : key;
    }
    for (int o = 16; o > 0; o >>= 1) { const unsigned long long other = __shfl_xor_sync(0xFFFFFFFFu, key, o); key = other > key ? other : key; }
    if (lane != 0) return;
    keys[g] = (int64_t)key;
    if (!((key >> 62) & 1ull)) { len[g] = 0; return; }
    const int64_t env = (0x3FFFFFFFll - (int64_t)(key & 0x3FFFFFFFull)) - c.first_id;
    const int n = (int)(c.rec[(size_t)HD_FLAGS * c.Bpad + env] >> FL_LEN_SHIFT);
    if (n > cap) { len[g] = -n; return; }
    len[g] = n;
    write_solution(c, env, n, actions + (size_t)g * cap);
}

// ---- end of a sharded search -------------------------------------------------------------------------------------------------------
// row layout (uint32): [0] key lo, [1] key hi, [2] solution length (0 if the winner did not succeed or does not fit), [3] rank, [4..] actions
constexpr int kFinHdr = 4;
__global__ void k_pack_winner(const __grid_constant__ DevCfg c, const unsigned long long* __restrict__ best, uint32_t* __restrict__ row, int cap, int rank) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const unsigned long long key = *best;
    row[0] = (uint32_t)key; row[1] = (uint32_t)(key >> 32); row[2] = 0; row[3] = (uint32_t)rank;
    if (key == 0 || !((key >> 62) & 1ull)) return;
    const int64_t env = (0x3FFFFFFFll - (int64_t)(key & 0x3FFFFFFFull)) - c.first_id;
    if (env < 0 || env >= c.B) return;
    const int n = (int)(c.rec[(size_t)HD_FLAGS * c.Bpad + env] >> FL_LEN_SHIFT);
    if (n > cap) return;
    write_solution(c, env, n, row + kFinHdr);
    row[2] = (uint32_t)n;
}
// rows [world][row_words] -> the row with the largest key into out (keys are unique: they embed the global rollout id)
__global__ void k_pick_winner(const uint32_t* __restrict__ rows, int world, int row_words, uint32_t* __restrict__ out) {
    __shared__ int win;
    if (threadIdx.x == 0) {
        unsigned long long bk = 0; int b = 0;
        for (int r = 0; r < world; ++r) {
            const unsigned long long k = (unsigned long long)rows[(size_t)r * row_words] | ((unsigned long long)rows[(size_t)r * row_words + 1] << 32);
            if (k > bk) { bk = k; b = r; }
        }
        win = b;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < row_words; i += blockDim.x) out[i] = rows[(size_t)win * row_words + i];
}
__global__ void k_best_key(const __grid_constant__ DevCfg c, unsigned long long* best);     // (defined below; same key as qg_search_best)

}  // namespace qg

// ---- NCCL, resolved at run time --------------------------------------------------------------------------------------------------------
namespace {
struct NcclApi {
    void* handle = nullptr; bool tried = false;
    decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
    decltype(&ncclCommInitRank) CommInitRank = nullptr;
    decltype(&ncclCommDestroy) CommDestroy = nullptr;
    decltype(&ncclCommCount) CommCount = nullptr;
    decltype(&ncclCommUserRank) CommUserRank = nullptr;
    decltype(&ncclAllGather) AllGather = nullptr;
    decltype(&ncclGetErrorString) GetErrorString = nullptr;
};
NcclApi g_nccl;
bool nccl_load() {
    if (g_nccl.tried) return g_nccl.handle != nullptr;
    g_nccl.tried = true;
    // the copy this process already uses (torch bundles one) if any, else the system library
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) { set_error(std::string("NCCL library not found: ") + (dlerror() ? dlerror() : "")); return false; }
    auto sym = [&](const char* n) { return dlsym(h, n); };
    g_nccl.GetUniqueId = (decltype(g_nccl.GetUniqueId))sym("ncclGetUniqueId");
    g_nccl.CommInitRank = (decltype(g_nccl.CommInitRank))sym("ncclCommInitRank");
    g_nccl.CommDestroy = (decltype(g_nccl.CommDestroy))sym("ncclCommDestroy");
    g_nccl.CommCount = (decltype(g_nccl.CommCount))sym("ncclCommCount");
    g_nccl.CommUserRank = (decltype(g_nccl.CommUserRank))sym("ncclCommUserRank");
    g_nccl.AllGather = (decltype(g_nccl.AllGather))sym("ncclAllGather");
    g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))sym("ncclGetErrorString");
    if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.CommDestroy || !g_nccl.CommCount || !g_nccl.CommUserRank || !g_nccl.AllGather) {
        set_error("NCCL library lacks a required symbol"); return false;
    }
    g_nccl.handle = h;
    return true;
}
#define NCCL_OK(expr)                                                                                                  \
    do {                                                                                                               \
        ncclResult_t _r = (expr);                                                                                      \
        if (_r != ncclSuccess) {                                                                                       \
            set_error(std::string(#expr) + ": " + (g_nccl.GetErrorString ? g_nccl.GetErrorString(_r) : "NCCL error")); \
            return QG_ERR_CUDA;                                                                                        \
        }                                                                                                              \
    } while (0)

// ---- NUMA helpers (sysfs + raw syscalls: no libnuma in the image) -------------------------------------------------------------------------
int device_numa_node(int device) {
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof(bus), device) != cudaSuccess) { cudaGetLastError(); return -1; }
    for (char* p = bus; *p; ++p) *p = (char)std::tolower((unsigned char)*p);
    std::ifstream f(std::string("/sys/bus/pci/devices/") + bus + "/numa_node");
    int node = -1;
    if (!(f >> node)) return -1;
    return node;
}
bool node_cpus(int node, cpu_set_t* set) {      // parses /sys/devices/system/node/nodeN/cpulist ("0-31,64-95")
    std::ifstream f("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist");
    std::string s;
    if (!std::getline(f, s)) return false;
    CPU_ZERO(set);
    std::stringstream ss(s);
    std::string part; int n = 0;
    while (std::getline(ss, part, ',')) {
        int a = 0, b = 0;
        if (std::sscanf(part.c_str(), "%d-%d", &a, &b) == 2) { for (int c = a; c <= b && c < CPU_SETSIZE; ++c) { CPU_SET(c, set); ++n; } }
        else if (std::sscanf(part.c_str(), "%d", &a) == 1 && a < CPU_SETSIZE) { CPU_SET(a, set); ++n; }
    }
    return n > 0;
}
}  // namespace

void qg::extras_release(qg_engine* e) {
    if (e->fin_send) cudaFree(e->fin_send);
    if (e->fin_recv) cudaFree(e->fin_recv);
    if (e->h_fin) cudaFreeHost(e->h_fin);
    if (e->bulk_sol) cudaFree(e->bulk_sol);
    if (e->bulk_len) cudaFree(e->bulk_len);
    if (e->dl_obs) cudaFree(e->dl_obs);
    for (int s2 = 0; s2 < 2; ++s2) {
        if (e->hp_act[s2]) cudaFree(e->hp_act[s2]);
        if (e->hp_coin[s2]) cudaFree(e->hp_coin[s2]);
        if (e->hp_ev_done[s2]) cudaEventDestroy(e->hp_ev_done[s2]);
        if (e->hp_ev_zero[s2]) cudaEventDestroy(e->hp_ev_zero[s2]);
        e->hp_act[s2] = e->hp_coin[s2] = nullptr; e->hp_ev_done[s2] = e->hp_ev_zero[s2] = nullptr;
    }
    if (e->hp_flags) cudaFree(e->hp_flags);
    if (e->hp_ones) cudaFreeHost(e->hp_ones);
    if (e->hp_stream) cudaStreamDestroy(e->hp_stream);
    e->hp_flags = e->hp_ones = nullptr; e->hp_stream = nullptr; e->hp_cap = 0;
    e->fin_send = e->fin_recv = e->h_fin = e->bulk_sol = nullptr; e->bulk_len = nullptr; e->dl_obs = nullptr;
}

// ---- DLPack v0.8 ABI (dlpack.h's plain structs; restated here because the header is not part of the CUDA toolkit) ------------------------
namespace {
struct QgDLDevice { int32_t device_type; int32_t device_id; };
struct QgDLDataType { uint8_t code; uint8_t bits; uint16_t lanes; };
struct QgDLTensor { void* data; QgDLDevice device; int32_t ndim; QgDLDataType dtype; int64_t* shape; int64_t* strides; uint64_t byte_offset; };
struct QgDLManagedTensor { QgDLTensor dl_tensor; void* manager_ctx; void (*deleter)(QgDLManagedTensor*); };
void dl_deleter(QgDLManagedTensor* m) {
    if (!m) return;
    delete[] m->dl_tensor.shape;
    delete m;
}
}  // namespace

extern "C" {

int qg_solutions(qg_engine* e, int64_t first, int64_t count, uint32_t* out_dev, int32_t cap, int32_t* len_dev, qg_stream stream) {
    if (!e || !out_dev || !len_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (first < 0 || count < 0 || first + count > e->B || cap < 1) { set_error("qg_solutions: env range outside the batch or cap < 1"); return QG_ERR_INVALID; }
    if (count == 0) return QG_OK;
    CUDA_OK(cudaSetDevice(e->device));
    k_solutions<<<(unsigned)((count + 127) / 128), 128, 0, (cudaStream_t)stream>>>(e->dc, first, count, out_dev, cap, len_dev);
    CUDA_OK(cudaGetLastError());
    return QG_OK;
}

int qg_solutions_host(qg_engine* e, int64_t first, int64_t count, uint32_t* out_host, int32_t cap, int32_t* len_host, qg_stream stream) {
    if (!e || !out_host || !len_host) { set_error("null argument"); return QG_ERR_INVALID; }
    if (first < 0 || count < 0 || first + count > e->B || cap < 1) { set_error("qg_solutions_host: env range outside the batch or cap < 1"); return QG_ERR_INVALID; }
    if (count == 0) return QG_OK;
    CUDA_OK(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    if (count > e->bulk_count || cap > e->bulk_cap) {
        CUDA_OK(cudaStreamSynchronize(st));
        if (e->bulk_sol) cudaFree(e->bulk_sol);
        if (e->bulk_len) cudaFree(e->bulk_len);
        e->bulk_sol = nullptr; e->bulk_len = nullptr; e->bulk_count = 0; e->bulk_cap = 0;
        const int64_t nc = std::max(count, e->bulk_count); const int ncap = std::max(cap, e->bulk_cap);
        CUDA_OK(cudaMalloc(&e->bulk_sol, (size_t)nc * ncap * 4));
        CUDA_OK(cudaMalloc(&e->bulk_len, (size_t)nc * 4));
        e->bulk_count = nc; e->bulk_cap = ncap;
    }
    k_solutions<<<(unsigned)((count + 127) / 128), 128, 0, st>>>(e->dc, first, count, e->bulk_sol, cap, e->bulk_len);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaMemcpyAsync(len_host, e->bulk_len, (size_t)count * 4, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaMemcpyAsync(out_host, e->bulk_sol, (size_t)count * cap * 4, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    return QG_OK;
}

int qg_search_best_grouped(qg_engine* e, int64_t group, int64_t num_groups, int64_t* keys_dev, uint32_t* actions_dev, int32_t cap, int32_t* len_dev,
                           qg_stream stream) {
    if (!e) { set_error("null engine"); return QG_ERR_INVALID; }
    if (group <= 0 || num_groups < 0 || num_groups > e->B / group || cap < 1) {
        set_error("qg_search_best_grouped: group must be >= 1, num_groups * group within the batch and cap >= 1"); return QG_ERR_INVALID;
    }
    if (num_groups == 0) return QG_OK;
    if (!keys_dev || !actions_dev || !len_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    CUDA_OK(cudaSetDevice(e->device));
    k_best_grouped<<<(unsigned)((num_groups + kGroupWarps - 1) / kGroupWarps), kGroupWarps * 32, 0, (cudaStream_t)stream>>>(e->dc, group, num_groups, keys_dev,
                                                                                                                          actions_dev, cap, len_dev);
    CUDA_OK(cudaGetLastError());
    return QG_OK;
}

int qg_replay_packed(qg_engine* e, int32_t num_steps, const uint8_t* actions8_dev, const uint8_t* coins_dev, float* obs_dev, uint8_t* mask_dev,
                     int32_t ring, float* reward_dev, uint32_t* done_bits_dev, uint32_t* success_bits_dev, qg_stream stream) {
    if (!e || !actions8_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (num_steps < 0 || ring < 1) { set_error("qg_replay_packed: num_steps must be >= 0 and ring >= 1"); return QG_ERR_INVALID; }
    if (e->L.A > 256) { set_error("the packed wire format needs num_actions <= 256"); return QG_ERR_UNSUPPORTED; }
    if (success_bits_dev && !done_bits_dev) { set_error("qg_replay_packed: success bits need done bits"); return QG_ERR_INVALID; }
    if (num_steps == 0) return QG_OK;
    StepArgs a{}; a.actions8 = actions8_dev; a.coins = coins_dev; a.obs = obs_dev; a.mask = mask_dev; a.reward = reward_dev;
    a.done_bits = done_bits_dev; a.success_bits = success_bits_dev; a.bits_stride = num_steps; a.bits_t0 = 0;
    a.nsteps = num_steps; a.ring = ring; a.in_stride = e->B; a.out_stride = e->B;
    return launch_step(e, MODE_STEP, a, (cudaStream_t)stream);
}

static int replay_host_packed_impl(qg_engine* e, int32_t num_steps, const uint8_t* actions8_host, const uint8_t* coins_host, float* obs_dev, uint8_t* mask_dev,
                                   int32_t ring, float* reward_host, float* reward_dev, uint32_t* done_bits_host, uint32_t* success_bits_host, qg_stream stream,
                                   bool synchronise) {
    if (!e || !actions8_host) { set_error("null argument"); return QG_ERR_INVALID; }
    if (num_steps < 0 || ring < 1) { set_error("qg_replay_host_packed: num_steps must be >= 0 and ring >= 1"); return QG_ERR_INVALID; }
    if (e->L.A > 256) { set_error("the packed wire format needs num_actions <= 256"); return QG_ERR_UNSUPPORTED; }
    if (reward_host && reward_dev) { set_error("qg_replay_host_packed: give reward_host or reward_dev, not both"); return QG_ERR_INVALID; }
    if (success_bits_host && !done_bits_host) { set_error("qg_replay_host_packed: success bits need done bits"); return QG_ERR_INVALID; }
    if (num_steps == 0 || e->B == 0) return QG_OK;
    CUDA_OK(cudaSetDevice(e->device));
    void* const m_act = mapped_host(actions8_host); void* const m_coin = mapped_host(coins_host); void* const m_rew = mapped_host(reward_host);
    void* const m_done = mapped_host(done_bits_host); void* const m_suc = mapped_host(success_bits_host);
    if (!m_act || (coins_host && !m_coin) || (reward_host && !m_rew) || (done_bits_host && !m_done) || (success_bits_host && !m_suc)) {
        set_error("qg_replay_host_packed needs pinned (page-locked) host buffers: qg_host_alloc / cudaHostAlloc / cudaHostRegister");
        return QG_ERR_INVALID;
    }
    StepArgs a{}; a.actions8 = (const uint8_t*)m_act; a.coins = (const uint8_t*)m_coin; a.obs = obs_dev; a.mask = mask_dev;
    cudaStream_t st = (cudaStream_t)stream;
    // Inputs: read by the kernel straight from host memory, a launch makes one 32-byte PCIe read per tile and step (262 144 of them for
    // 65 536 envs x 128 steps) and is throttled by their rate (profiles/r2_v25_e2e_probe.json).  Instead the copy engine streams the rows into
    // a device staging buffer in three chunks of growing size (4, 28 steps, the rest) on a second stream, each followed by a 4-byte copy that
    // raises the chunk's flag; the kernel starts with the first chunk and polls a flag only when it crosses a chunk border
    // (wait_input_chunk) — by then the engine, which moves a step's row in ~1 us against ~10 us per step of the kernel, is far ahead.
    // Two staging slots alternate, so the inputs of an episode queued behind a running one (qg_replay_host_packed_async) arrive while
    // that one still plays.  Everything is queued BEFORE the launch: a tool that serialises launches (ncu, compute-sanitizer) cannot
    // dead-lock it; flags are cleared by a copy too (a memset kernel would wait for an SM slot).
    const size_t row = (size_t)e->B, total = row * (size_t)num_steps;
    int slot = -1;
    if (num_steps >= 16 && total >= (size_t)1 << 20) {
        if (!e->hp_stream) {
            CUDA_OK(cudaStreamCreateWithFlags(&e->hp_stream, cudaStreamNonBlocking));
            for (int s2 = 0; s2 < 2; ++s2) {
                CUDA_OK(cudaEventCreateWithFlags(&e->hp_ev_done[s2], cudaEventDisableTiming));
                CUDA_OK(cudaEventCreateWithFlags(&e->hp_ev_zero[s2], cudaEventDisableTiming));
            }
            CUDA_OK(cudaMalloc(&e->hp_flags, 2 * 4 * sizeof(uint32_t)));
            CUDA_OK(cudaMemset(e->hp_flags, 0, 2 * 4 * sizeof(uint32_t)));
            CUDA_OK(cudaHostAlloc(&e->hp_ones, 8 * sizeof(uint32_t), cudaHostAllocDefault));
            for (int i = 0; i < 4; ++i) { e->hp_ones[i] = 1u; e->hp_ones[4 + i] = 0u; }
        }
        if (total > e->hp_cap) {
            CUDA_OK(cudaStreamSynchronize(st));
            CUDA_OK(cudaStreamSynchronize(e->hp_stream));
            for (int s2 = 0; s2 < 2; ++s2) {
                if (e->hp_act[s2]) cudaFree(e->hp_act[s2]);
                if (e->hp_coin[s2]) cudaFree(e->hp_coin[s2]);
                e->hp_act[s2] = nullptr; e->hp_coin[s2] = nullptr;
            }
            e->hp_cap = 0;
            for (int s2 = 0; s2 < 2; ++s2) { CUDA_OK(cudaMalloc(&e->hp_act[s2], total)); CUDA_OK(cudaMalloc(&e->hp_coin[s2], total)); }
            e->hp_cap = total; e->hp_used[0] = e->hp_used[1] = false;
        }
        slot = e->hp_next; e->hp_next ^= 1;
        uint32_t* const flags = e->hp_flags + 4 * slot;
        if (e->hp_used[slot]) CUDA_OK(cudaStreamWaitEvent(e->hp_stream, e->hp_ev_done[slot], 0));     // the launch that last read this slot is over
        CUDA_OK(cudaMemcpyAsync(flags, e->hp_ones + 4, 4 * sizeof(uint32_t), cudaMemcpyHostToDevice, e->hp_stream));
        CUDA_OK(cudaEventRecord(e->hp_ev_zero[slot], e->hp_stream));
        const int begin[4] = {0, 4, 32, num_steps};
        for (int k = 0; k < 4; ++k) a.in_chunk[k] = -1;
        for (int k = 0; k < 3; ++k) {
            if (begin[k] >= num_steps) continue;
            const size_t o = (size_t)begin[k] * row, n = (size_t)(std::min(begin[k + 1], (int)num_steps) - begin[k]) * row;
            CUDA_OK(cudaMemcpyAsync(e->hp_act[slot] + o, actions8_host + o, n, cudaMemcpyHostToDevice, e->hp_stream));
            if (coins_host) CUDA_OK(cudaMemcpyAsync(e->hp_coin[slot] + o, coins_host + o, n, cudaMemcpyHostToDevice, e->hp_stream));
            CUDA_OK(cudaMemcpyAsync(flags + k, e->hp_ones + k, sizeof(uint32_t), cudaMemcpyHostToDevice, e->hp_stream));
            a.in_chunk[k] = begin[k];
        }
        CUDA_OK(cudaStreamWaitEvent(st, e->hp_ev_zero[slot], 0));                                        // the launch must not see the previous episode's flags
        a.actions8 = e->hp_act[slot]; a.coins = coins_host ? e->hp_coin[slot] : nullptr; a.in_flags = flags;
    }
    a.reward = reward_host ? (float*)m_rew : reward_dev;
    a.done_bits = (uint32_t*)m_done; a.success_bits = (uint32_t*)m_suc; a.bits_stride = num_steps; a.bits_t0 = 0;
    a.nsteps = num_steps; a.ring = ring; a.in_stride = e->B; a.out_stride = e->B;
    const int rc = launch_step(e, MODE_STEP, a, st);
    if (rc != QG_OK) { if (slot >= 0) cudaStreamSynchronize(e->hp_stream); return rc; }
    if (slot >= 0) { CUDA_OK(cudaEventRecord(e->hp_ev_done[slot], st)); e->hp_used[slot] = true; }
    if (synchronise) CUDA_OK(cudaStreamSynchronize(st));
    return QG_OK;
}

int qg_replay_host_packed(qg_engine* e, int32_t num_steps, const uint8_t* actions8_host, const uint8_t* coins_host, float* obs_dev, uint8_t* mask_dev,
                          int32_t ring, float* reward_host, float* reward_dev, uint32_t* done_bits_host, uint32_t* success_bits_host, qg_stream stream) {
    return replay_host_packed_impl(e, num_steps, actions8_host, coins_host, obs_dev, mask_dev, ring, reward_host, reward_dev, done_bits_host, success_bits_host, stream, true);
}

int qg_replay_host_packed_async(qg_engine* e, int32_t num_steps, const uint8_t* actions8_host, const uint8_t* coins_host, float* obs_dev, uint8_t* mask_dev,
                                int32_t ring, float* reward_host, float* reward_dev, uint32_t* done_bits_host, uint32_t* success_bits_host, qg_stream stream) {
    return replay_host_packed_impl(e, num_steps, actions8_host, coins_host, obs_dev, mask_dev, ring, reward_host, reward_dev, done_bits_host, success_bits_host, stream, false);
}

int qg_bind_thread_to_device(int32_t device) {
    const int node = device_numa_node(device);
    if (node < 0) return -1;
    cpu_set_t set;
    if (!node_cpus(node, &set)) return -1;
    if (sched_setaffinity(0, sizeof(set), &set) != 0) return -1;
    return node;
}

int qg_host_alloc(int32_t device, size_t bytes, void** out_host, int32_t* numa_node_out) {
    if (!out_host) { set_error("null argument"); return QG_ERR_INVALID; }
    *out_host = nullptr;
    if (numa_node_out) *numa_node_out = -1;
    int ndev = 0;
    CUDA_OK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) { set_error("no such CUDA device"); return QG_ERR_CUDA; }
    CUDA_OK(cudaSetDevice(device));
    const int node = device_numa_node(device);
    cpu_set_t old_set, node_set;
    bool bound = false, policy = false;
    if (node >= 0 && node < 1024 && sched_getaffinity(0, sizeof(old_set), &old_set) == 0 && node_cpus(node, &node_set)) {
        bound = sched_setaffinity(0, sizeof(node_set), &node_set) == 0;
        unsigned long mask[16] = {0};
        mask[node / (8 * sizeof(unsigned long))] |= 1ul << (node % (8 * sizeof(unsigned long)));
        policy = syscall(SYS_set_mempolicy, 1 /*MPOL_PREFERRED*/, mask, (unsigned long)(sizeof(mask) * 8)) == 0;
    }
    void* p = nullptr;
    cudaError_t ce = cudaHostAlloc(&p, std::max<size_t>(bytes, 1), cudaHostAllocPortable | cudaHostAllocMapped);
    if (ce == cudaSuccess) std::memset(p, 0, bytes);                 // first touch while the policy is in force
    if (policy) syscall(SYS_set_mempolicy, 0 /*MPOL_DEFAULT*/, nullptr, 0ul);
    if (bound) sched_setaffinity(0, sizeof(old_set), &old_set);
    if (ce != cudaSuccess) { set_error(std::string("cudaHostAlloc: ") + cudaGetErrorString(ce)); return QG_ERR_CUDA; }
    *out_host = p;
    if (numa_node_out) *numa_node_out = (bound || policy) ? node : -1;
    return QG_OK;
}

int qg_host_free(void* host) {
    if (!host) return QG_OK;
    CUDA_OK(cudaFreeHost(host));
    return QG_OK;
}

int qg_dlpack_obs(qg_engine* e, int32_t ring, void** managed_tensor_out, float** obs_dev_out) {
    if (!e || !managed_tensor_out) { set_error("null argument"); return QG_ERR_INVALID; }
    if (ring < 1) { set_error("qg_dlpack_obs: ring must be >= 1"); return QG_ERR_INVALID; }
    if (e->dl_obs && e->dl_ring != ring) { set_error("qg_dlpack_obs: the engine already owns an observation ring of another size"); return QG_ERR_INVALID; }
    CUDA_OK(cudaSetDevice(e->device));
    if (!e->dl_obs) {
        const size_t bytes = std::max<size_t>((size_t)ring * (size_t)e->B * (size_t)e->L.obs_size * 4, 16);
        CUDA_OK(cudaMalloc(&e->dl_obs, bytes));
        CUDA_OK(cudaMemset(e->dl_obs, 0, bytes));
        e->dl_ring = ring;
    }
    QgDLManagedTensor* m = new (std::nothrow) QgDLManagedTensor();
    if (!m) { set_error("out of memory"); return QG_ERR_INVALID; }
    const bool with_ring = ring > 1;
    const int nd = with_ring ? 4 : 3;
    int64_t* shape = new (std::nothrow) int64_t[4];
    if (!shape) { delete m; set_error("out of memory"); return QG_ERR_INVALID; }
    int k = 0;
    if (with_ring) shape[k++] = ring;
    shape[k++] = e->B; shape[k++] = e->L.obs_rows; shape[k++] = e->L.obs_cols;
    m->dl_tensor.data = e->dl_obs;
    m->dl_tensor.device = QgDLDevice{2 /*kDLCUDA*/, e->device};
    m->dl_tensor.ndim = nd;
    m->dl_tensor.dtype = QgDLDataType{2 /*kDLFloat*/, 32, 1};
    m->dl_tensor.shape = shape;
    m->dl_tensor.strides = nullptr;          // compact row-major
    m->dl_tensor.byte_offset = 0;
    m->manager_ctx = nullptr;
    m->deleter = dl_deleter;
    *managed_tensor_out = m;
    if (obs_dev_out) *obs_dev_out = e->dl_obs;
    return QG_OK;
}

int qg_nccl_unique_id(uint8_t id_out[128]) {
    if (!id_out) { set_error("null argument"); return QG_ERR_INVALID; }
    if (!nccl_load()) return QG_ERR_UNSUPPORTED;
    static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
    ncclUniqueId id;
    NCCL_OK(g_nccl.GetUniqueId(&id));
    std::memcpy(id_out, &id, 128);
    return QG_OK;
}

int qg_nccl_comm_create(const uint8_t id[128], int32_t rank, int32_t world, int32_t device, qg_nccl_comm* out) {
    if (!id || !out) { set_error("null argument"); return QG_ERR_INVALID; }
    if (world < 1 || rank < 0 || rank >= world) { set_error("qg_nccl_comm_create: bad rank / world"); return QG_ERR_INVALID; }
    if (!nccl_load()) return QG_ERR_UNSUPPORTED;
    CUDA_OK(cudaSetDevice(device));
    ncclUniqueId uid;
    std::memcpy(&uid, id, 128);
    ncclComm_t c = nullptr;
    NCCL_OK(g_nccl.CommInitRank(&c, world, uid, rank));
    *out = (qg_nccl_comm)c;
    return QG_OK;
}

int qg_nccl_comm_destroy(qg_nccl_comm comm) {
    if (!comm) return QG_OK;
    if (!nccl_load()) return QG_ERR_UNSUPPORTED;
    NCCL_OK(g_nccl.CommDestroy((ncclComm_t)comm));
    return QG_OK;
}

int qg_search_finish(qg_engine* e, qg_nccl_comm comm, int64_t* best_key_host, int32_t* success_host, int64_t* rollout_id_host, int32_t* owner_rank_host,
                     uint32_t* actions_host, int32_t cap, int32_t* len_host, qg_stream stream) {
    if (!e || !best_key_host || !len_host) { set_error("null argument"); return QG_ERR_INVALID; }
    if (cap < 0 || (cap > 0 && !actions_host)) { set_error("qg_search_finish: bad action buffer"); return QG_ERR_INVALID; }
    CUDA_OK(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    int world = 1, rank = 0;
    if (comm) {
        if (!nccl_load()) return QG_ERR_UNSUPPORTED;
        NCCL_OK(g_nccl.CommCount((ncclComm_t)comm, &world));
        NCCL_OK(g_nccl.CommUserRank((ncclComm_t)comm, &rank));
    }
    const int row_words = kFinHdr + std::max(cap, 1);
    if (!e->fin_send || e->fin_cap < cap || e->fin_world < world) {
        CUDA_OK(cudaStreamSynchronize(st));
        if (e->fin_send) cudaFree(e->fin_send);
        if (e->fin_recv) cudaFree(e->fin_recv);
        if (e->h_fin) cudaFreeHost(e->h_fin);
        e->fin_send = e->fin_recv = e->h_fin = nullptr;
        CUDA_OK(cudaMalloc(&e->fin_send, (size_t)row_words * 4));
        CUDA_OK(cudaMalloc(&e->fin_recv, (size_t)(world + 1) * row_words * 4));
        CUDA_OK(cudaMallocHost(&e->h_fin, (size_t)row_words * 4));
        e->fin_cap = cap; e->fin_world = world;
    }
    const int rw = kFinHdr + std::max(e->fin_cap, 1);          // (buffers may be larger than this call needs: rows keep the allocated stride)
    CUDA_OK(cudaMemsetAsync(e->best, 0, 8, st));
    if (e->B > 0) k_best_key<<<(unsigned)((e->B + 255) / 256), 256, 0, st>>>(e->dc, e->best);
    k_pack_winner<<<1, 32, 0, st>>>(e->dc, e->best, e->fin_send, e->fin_cap, rank);
    CUDA_OK(cudaGetLastError());
    const uint32_t* winner = e->fin_send;
    if (comm && world > 1) {
        NCCL_OK(g_nccl.AllGather(e->fin_send, e->fin_recv, (size_t)rw, ncclUint32, (ncclComm_t)comm, st));
        uint32_t* out = e->fin_recv + (size_t)world * rw;
        k_pick_winner<<<1, 128, 0, st>>>(e->fin_recv, world, rw, out);
        CUDA_OK(cudaGetLastError());
        winner = out;
    }
    CUDA_OK(cudaMemcpyAsync(e->h_fin, winner, (size_t)rw * 4, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    const unsigned long long key = (unsigned long long)e->h_fin[0] | ((unsigned long long)e->h_fin[1] << 32);
    *best_key_host = (int64_t)key;
    const bool ok = key != 0 && ((key >> 62) & 1ull);
    if (success_host) *success_host = ok ? 1 : 0;
    if (rollout_id_host) *rollout_id_host = key ? (0x3FFFFFFFll - (int64_t)(key & 0x3FFFFFFFull)) : -1;
    if (owner_rank_host) *owner_rank_host = key ? (int32_t)e->h_fin[3] : -1;
    const int n = ok ? (int)e->h_fin[2] : 0;
    *len_host = std::min(n, (int)cap);
    for (int i = 0; i < *len_host; ++i) actions_host[i] = e->h_fin[kFinHdr + i];
    return QG_OK;
}

}  // extern "C"

namespace qg {
__global__ void k_best_key(const __grid_constant__ DevCfg c, unsigned long long* best) {
    const int64_t env = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long key = 0;
    if (env < c.B) key = rollout_key((c.rec[(size_t)HD_FLAGS * c.Bpad + env] & FL_SUCCESS) != 0, c.ret[env], c.first_id + env);
    for (int o = 16; o > 0; o >>= 1) { const unsigned long long other = __shfl_xor_sync(0xFFFFFFFFu, key, o); key = other > key ? other : key; }
    if ((threadIdx.x & 31) == 0 && key) atomicMax(best, key);
}
}  // namespace qg
