// qg_engine.cu — implementation of the C ABI declared in include/qg_engine.h.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "qg_engine_priv.hpp"
#include "qg_aux_kernels.cuh"
#include "qg_policy_host.hpp"

using namespace qg;

namespace {

inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }
inline uint64_t magic40(uint32_t d) { return ((1ull << 40) + d - 1) / d; }

struct WsPlan {
    int64_t rec, snap, sol, ret, gates, ident, qperms, aperms, pgen, staged, io_actions, io_coins, io_reward, io_done, io_success, best, total;
};
WsPlan plan_ws(const Layout& L, int64_t B, int64_t nperms, int64_t pgen_words) {
    const int64_t Bpad = align_up(std::max<int64_t>(B, 1), 32);
    WsPlan p{}; int64_t o = 0;
    auto take = [&](int64_t bytes) { const int64_t at = o; o = align_up(o + bytes, 256); return at; };
    p.rec = take((int64_t)L.W * Bpad * 4);
    p.snap = take((int64_t)L.W * Bpad * 4);
    p.sol = take((int64_t)L.sol_cap * Bpad * 4);
    p.ret = take(Bpad * 4);
    p.gates = take((int64_t)L.A * 4);
    p.ident = take((int64_t)L.SW * 4);
    p.qperms = take(std::max<int64_t>(nperms * L.n, 1));
    p.aperms = take(std::max<int64_t>(nperms * L.A * 2, 1));
    p.pgen = take(std::max<int64_t>(pgen_words * 4, 4));
    p.staged = take((int64_t)L.PW * Bpad * 4);
    p.io_actions = take(Bpad * 4); p.io_coins = take(Bpad); p.io_reward = take(Bpad * 4); p.io_done = take(Bpad); p.io_success = take(Bpad);
    p.best = take(64);
    p.total = o;
    return p;
}

int pauli_perms(const qg_config* cfg, Twists& tw) {
    if (cfg->env_kind != QG_ENV_PAULI_NETWORK || !cfg->add_perms) { tw = Twists(); return QG_OK; }
    return compute_twists(cfg, true, tw);
}

// shared memory of an SM that CTAs can share (228 KB, 1 KB of it reserved per CTA) and the largest request the replay cap makes (2 CTAs per SM)
constexpr size_t kSmSharedBytes = 228 * 1024, kReplaySmemCapMax = kSmSharedBytes / 2 - 1024;

int prepare_kernels(qg_engine* e) {   // kernel attributes (shared-memory carve-out, > 48 KB opt-in) once, outside any stream capture
    // (replay launches may ask for more shared memory than their layout needs, to bound the CTAs an SM holds: launch_step)
    const size_t attr_bytes = std::max(e->smem_bytes, (size_t)kReplaySmemCapMax);
    switch (e->L.kind) {
        case QG_ENV_PERMUTATION: CUDA_OK(prepare_step_kind<QG_ENV_PERMUTATION>(attr_bytes)); break;
        case QG_ENV_LINEAR_FUNCTION: CUDA_OK(prepare_step_kind<QG_ENV_LINEAR_FUNCTION>(attr_bytes)); break;
        case QG_ENV_CLIFFORD: CUDA_OK(prepare_step_kind<QG_ENV_CLIFFORD>(attr_bytes)); break;
        default: CUDA_OK(prepare_step_kind<QG_ENV_PAULI_NETWORK>(attr_bytes)); break;
    }
    return QG_OK;
}
}  // namespace

// The device-side address of a pinned (page-locked) host buffer — under unified addressing such memory is mapped into the device's address
// space, so a kernel can read / write it over PCIe — or nullptr for pageable memory.
void* qg::mapped_host(const void* h) {
    if (!h) return nullptr;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, h) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return at.type == cudaMemoryTypeHost ? at.devicePointer : nullptr;
}

int qg::launch_step(qg_engine* e, int mode, StepArgs a, cudaStream_t st, int64_t logical_batch) {
    // logical_batch >= 0: the launch covers that many logical envs addressed through a.src_slot / a.dst_slot (qg_step_slots)
    const int64_t LB = logical_batch >= 0 ? logical_batch : e->B;
    if (LB == 0) return QG_OK;
    int cur = -1;
    CUDA_OK(cudaGetDevice(&cur));
    if (cur != e->device) CUDA_OK(cudaSetDevice(e->device));
    if (a.nsteps <= 0) a.nsteps = 1;
    if (a.ring <= 0) a.ring = 1;
    a.pdl_mode = e->pdl_mode; a.num_sms = e->num_sms;
    a.stagger_ns = (mode == MODE_STEP && a.nsteps >= 8) ? e->stagger_ns : 0;
    // tile size.  Measured at 65 536 envs (profiles/r2_v2_tile_sweep.txt): 16-env tiles (twice the warps, lanes 16..31 idle in the step logic)
    // lose 2-14 % in replay launches for every config and in single-step launches of the small observations (C1 / C2 / C3), but a single-step
    // launch of a large observation gains (C4 0.53 -> 0.58, C5 0.68 -> 0.82 of the roofline): its warps each store 60-90 KB per step, and half-size
    // tiles let the first stores start after half the step logic.  Host-packed launches keep 32 (16-env tiles halve the PCIe transaction sizes).
    const int64_t tiles32 = (LB + 31) / 32;
    int epw = (mode != MODE_OBSERVE && a.nsteps <= 1 && e->L.obs_size >= 384 && !a.done_bits && tiles32 <= (int64_t)e->num_sms * 20) ? 16 : 32;
    if (e->cfg.tile_envs == 16 || e->cfg.tile_envs == 32) epw = e->cfg.tile_envs;
    if (e->epw_forced == 16 || e->epw_forced == 32) epw = e->epw_forced;
    if (mode == MODE_OBSERVE) epw = 32;
    const int stride = epw + 1;
    const int lay_words = e->L.W + e->L.SCR + e->L.OW;
    const int cat_w = e->cat_words ? (e->cat_words * epw + 31) / 32 : 0;
    a.sm_scr = e->L.W * stride; a.sm_obs = (e->L.W + e->L.SCR) * stride;
    // Permutation builds the concatenated stream straight from the state: it takes the place of the per-environment stream O (which such a
    // launch does not build unless packed observations are requested as well); the other kinds gather it from O into a region of its own
    const bool cat_in_O = e->L.kind == QG_ENV_PERMUTATION && !a.obs_bits && cat_w <= e->L.OW * stride;
    a.sm_cat = (cat_w && a.obs && mode != MODE_SEARCH && !a.skip_negative) ? (cat_in_O ? a.sm_obs : lay_words * stride) : -1;
    a.sm_warp_words = lay_words * stride + ((a.sm_cat >= 0 && !cat_in_O) ? cat_w : 0);
    a.sm_wts = -1;
    if (mode == MODE_SEARCH && a.weights && (int64_t)(e->L.A | 1) * epw * 4 <= 16 * 1024) {        // staged action weights (step_tile)
        a.sm_wts = a.sm_warp_words; a.sm_warp_words += (e->L.A | 1) * epw;
    }
    // replay launches that write dense observations: a warp PAIR per tile (step warp + store warp, step_tile roles 1 / 2) when the tile's
    // observation bits can be handed over as one buffer — LinearFunction / Clifford (the state words), or the concatenated-stream kinds — and a
    // bound on the CTAs (= tiles) an SM holds at a time.  Measured at 65 536 envs with one observation slab per step
    // (profiles/r2_v27_resident_sweep.txt, fractions of the copy bandwidth): what decides is how many tiles write at once — with all 2 048
    // tiles resident a launch reaches 0.89 (C3) whether tiles are pairs or not; with 3-5 pair CTAs per SM 0.98-0.99 (C3), 1.00-1.01 (C5); the
    // kinds whose step logic dominates need more tiles in flight to cover it: 8 per SM gives C2 0.80 (all resident: 0.74), C4 0.945 (0.89),
    // C1 0.80 (0.79), while 4 per SM loses a third.  Pairs because a bounded SM needs the step logic of step t+1 overlapped with the stores of
    // step t on the SAME tile (single-warp tiles at the best bound: C3 0.94, and 0.75 one notch off it).
    a.pair = 0; a.sm_pair = 0; a.pair_words = 0;
    int resident = 0;                // CTAs per SM of this launch (0 = whatever fits)
    if (mode == MODE_STEP && a.nsteps >= 8 && a.obs && !a.obs_bits && !a.skip_negative && epw == 32 && e->pair_forced >= 0) {
        const int k = e->L.kind;
        int pw = 0;
        if (k == QG_ENV_LINEAR_FUNCTION || k == QG_ENV_CLIFFORD) pw = e->L.SW * stride;
        else if (a.sm_cat >= 0) pw = (k == QG_ENV_PERMUTATION) ? cat_w : e->L.OW * stride;
        if (pw > 0 && (k != QG_ENV_LINEAR_FUNCTION && k != QG_ENV_CLIFFORD ? true : (cat_w == 0 || a.sm_cat >= 0))) {
            a.pair = 1; a.pair_words = pw; a.sm_pair = a.sm_warp_words;
            a.sm_pair_bar = (a.sm_pair + 2 * pw + 2 + 1) & ~1;          // after the two ballot words, 8-byte aligned (the region starts 16-byte aligned)
            a.sm_warp_words = a.sm_pair_bar + 8;
            // CTAs per SM (profiles/r2_v27_resident_sweep.txt, r2_v28_resident_sweep2.txt; 2 048 tiles on 148 SMs).  Where the stores dominate a
            // step (LinearFunction / Clifford / Permutation with >= 160 entries) 3-5 are equally good (C3 0.98-0.99, C5 1.00-1.01) and the tail
            // of a partly filled last wave costs nothing (its tiles get the bandwidth of the missing ones).  Where the step logic dominates,
            // a tile runs at its own pace however few are left: the last wave has to be full — 7 per SM is 1.98 waves (C1 0.82, C2 0.84), 6 is
            // 2.31 (0.64, 0.67), 8 is 1.73 (0.80, 0.79): the bound with the best-filled last wave among 7..10.  PauliNetwork, both at once: 8.
            const int64_t t32 = (LB + 31) / 32;
            if (k != QG_ENV_PAULI_NETWORK && e->L.obs_size >= 160) resident = 5;
            else if (k == QG_ENV_PAULI_NETWORK) resident = 8;
            else {
                double best = -1.0;
                for (int r = 7; r <= 10; ++r) {
                    const int64_t slots = (int64_t)e->num_sms * r, waves = (t32 + slots - 1) / slots;
                    const double fill = (double)t32 / (double)(waves * slots);
                    if (fill > best + 1e-9) { best = fill; resident = r; }
                }
            }
        }
    }
    if (e->replay_ctas) resident = e->replay_ctas > 0 ? e->replay_ctas : 0;
    a.magic_obs = e->magic_obs; a.magic_A = e->magic_A;
    a.magic_vpe = e->magic_vpe; a.magic_a4 = e->magic_a4;
    { const uint32_t vpe = (uint32_t)e->L.obs_size / 4; a.exp_q = vpe ? 32u / vpe : 0u; a.exp_r = vpe ? 32u - a.exp_q * vpe : 0u; }
    a.symplectic = e->all_symplectic ? 1 : 0;
    a.magic_ow = magic40(((uint32_t)e->L.obs_size + 31u) / 32u);
    if (a.obs_bits && e->L.kind == QG_ENV_PERMUTATION && e->L.OW == 0) { set_error("packed observations need num_qubits <= 64 for Permutation"); return QG_ERR_UNSUPPORTED; }
    if (a.obs && (reinterpret_cast<uintptr_t>(a.obs) & 15)) { set_error("obs_dev must be 16-byte aligned"); return QG_ERR_INVALID; }
    if (a.mask && (reinterpret_cast<uintptr_t>(a.mask) & 15)) { set_error("mask_dev must be 16-byte aligned"); return QG_ERR_INVALID; }
    const int64_t tiles = (LB + epw - 1) / epw;
    DevCfg dc = e->dc;
    dc.B = LB;
    LaunchGeom g{(unsigned)((tiles + kWarpsPerCta - 1) / kWarpsPerCta), ((size_t)kLutWords + (size_t)a.sm_warp_words * kWarpsPerCta) * 4, a.pdl_mode ? 1 : 0, epw};
    if (a.pair) { g.grid = (unsigned)tiles; g.smem_bytes = ((size_t)kLutWords + (size_t)a.sm_warp_words) * 4; }
    // the bound: the request is padded to 1 / resident of the SM's shared memory
    int resident_step = 0;           // (tools builds: QG_STEP_CTAS bounds single-step launches the same way)
#ifdef QG_TOOLS_KNOBS
    if (mode == MODE_STEP && a.nsteps < 8 && a.obs) resident_step = e->step_ctas;
#endif
    if (resident_step >= 2) resident = resident_step;
    if (mode == MODE_STEP && (a.nsteps >= 8 || resident_step >= 2) && a.obs && resident >= 2) {
        const size_t cap = (kSmSharedBytes / (size_t)resident - 1024) & ~(size_t)127;
        if (cap > g.smem_bytes) g.smem_bytes = cap;
    }
    if (e->l2_persist_bytes > 0 && mode == MODE_STEP && a.nsteps > 1 && a.actions) {
        // replay: keep the resident action stream in L2 (persisting window) so that the launch's DRAM traffic is writes only
        g.l2_base = a.actions; g.l2_bytes = std::min<size_t>((size_t)a.nsteps * (size_t)a.in_stride * 4, e->l2_persist_bytes);
    }
    // register bucket of the add_inverts inverse (qg_gf2.cuh); 0 = generic shared-memory path (dimension > 32, or no inverts)
    int inv = 0;
    if (e->dc.add_inverts && e->inv_bucket_enabled && (e->L.kind == QG_ENV_LINEAR_FUNCTION || e->L.kind == QG_ENV_CLIFFORD))
        inv = e->L.D <= 8 ? 8 : e->L.D <= 16 ? 16 : e->L.D <= 32 ? 32 : 0;
    switch (e->L.kind) {
        case QG_ENV_PERMUTATION: CUDA_OK(launch_step_kind<QG_ENV_PERMUTATION>(mode, inv, dc, a, g, st)); break;
        case QG_ENV_LINEAR_FUNCTION: CUDA_OK(launch_step_kind<QG_ENV_LINEAR_FUNCTION>(mode, inv, dc, a, g, st)); break;
        case QG_ENV_CLIFFORD: CUDA_OK(launch_step_kind<QG_ENV_CLIFFORD>(mode, inv, dc, a, g, st)); break;
        default: CUDA_OK(launch_step_kind<QG_ENV_PAULI_NETWORK>(mode, inv, dc, a, g, st)); break;
    }
    return QG_OK;
}

namespace {

int launch_load(qg_engine* e, int64_t first, int64_t count, int64_t group, uint32_t depth_init, cudaStream_t st) {
    if (count <= 0) return QG_OK;
    const unsigned grid = (unsigned)((count + 255) / 256);
    switch (e->L.kind) {
        case QG_ENV_PERMUTATION: k_load<QG_ENV_PERMUTATION><<<grid, 256, 0, st>>>(e->dc, e->staged, e->L.PW, first, count, group, depth_init); break;
        case QG_ENV_LINEAR_FUNCTION: k_load<QG_ENV_LINEAR_FUNCTION><<<grid, 256, 0, st>>>(e->dc, e->staged, e->L.PW, first, count, group, depth_init); break;
        case QG_ENV_CLIFFORD: k_load<QG_ENV_CLIFFORD><<<grid, 256, 0, st>>>(e->dc, e->staged, e->L.PW, first, count, group, depth_init); break;
        default: k_load<QG_ENV_PAULI_NETWORK><<<grid, 256, 0, st>>>(e->dc, e->staged, e->L.PW, first, count, group, depth_init); break;
    }
    CUDA_OK(cudaGetLastError());
    return QG_OK;
}

int ensure_host_staging(qg_engine* e, int64_t words) {
    if (e->h_staged_words >= words) return QG_OK;
    if (e->h_staged) cudaFreeHost(e->h_staged);
    e->h_staged = nullptr; e->h_staged_words = 0;
    CUDA_OK(cudaMallocHost(&e->h_staged, (size_t)words * 4));
    e->h_staged_words = words;
    return QG_OK;
}

}  // namespace

extern "C" {

const char* qg_version(void) { return "qiskit_gym_b200 0.1.0 (sm_100a)"; }
const char* qg_last_error(void) { return get_error(); }

void qg_config_default(qg_config* cfg, int32_t env_kind) {
    if (!cfg) return;
    std::memset(cfg, 0, sizeof(*cfg));
    cfg->env_kind = env_kind; cfg->difficulty = 1; cfg->depth_slope = 2; cfg->max_depth = 128;
    cfg->w_n_cnots = 0.01f; cfg->w_n_layers_cnots = 0.0f; cfg->w_n_layers = 0.0f; cfg->w_n_gates = 0.0001f;   // metrics.rs:158-166
    cfg->add_inverts = env_kind == QG_ENV_PAULI_NETWORK ? 0 : 1; cfg->add_perms = 1; cfg->track_solution = 1;
    cfg->max_rotations = 5; cfg->pauli_diff_scale = 8; cfg->num_qubits_decay = 0.5f; cfg->final_pauli_layers = -1; cfg->pauli_layer_reward = 0.01f;
}

int qg_gate_kind_from_name(const char* name, int32_t num_indices) {   // common.rs:61-99
    if (!name) return QG_ERR_INVALID;
    std::string s(name);
    const size_t a = s.find_first_not_of(" \t\r\n\f\v"), b = s.find_last_not_of(" \t\r\n\f\v");
    s = (a == std::string::npos) ? std::string() : s.substr(a, b - a + 1);
    for (char& ch : s) if (ch >= 'A' && ch <= 'Z') ch = (char)(ch - 'A' + 'a');
    static const struct { const char* nm; int kind; int arity; } table[] = {
        {"h", QG_H, 1}, {"s", QG_S, 1}, {"sdg", QG_SDG, 1}, {"sx", QG_SX, 1}, {"sxdg", QG_SXDG, 1}, {"cx", QG_CX, 2}, {"cz", QG_CZ, 2}, {"swap", QG_SWAP, 2}};
    for (const auto& t : table)
        if (s == t.nm) return num_indices == t.arity ? t.kind : QG_ERR_STATE;
    return QG_ERR_INVALID;
}

int qg_config_validate(const qg_config* cfg) { return validate_config(cfg); }

int qg_config_obs_shape(const qg_config* cfg, int32_t out_shape[2]) {
    Layout L; const int rc = make_layout(cfg, L);
    if (rc != QG_OK) return rc;
    out_shape[0] = L.obs_rows; out_shape[1] = L.obs_cols;
    return QG_OK;
}
int64_t qg_config_state_len(const qg_config* cfg) {
    Layout L; const int rc = make_layout(cfg, L);
    return rc != QG_OK ? rc : L.state_len;
}

int qg_twists_create(const qg_config* cfg, qg_twists** out) {
    if (!out) { set_error("null out"); return QG_ERR_INVALID; }
    qg_twists* t = new (std::nothrow) qg_twists();
    if (!t) { set_error("out of memory"); return QG_ERR_INVALID; }
    const int rc = compute_twists(cfg, false, t->t);
    if (rc != QG_OK) { delete t; return rc; }
    *out = t; return QG_OK;
}
void qg_twists_destroy(qg_twists* t) { delete t; }
int64_t qg_twists_count(const qg_twists* t) { return t ? (int64_t)t->t.obs_perms.size() : 0; }
int64_t qg_twists_obs_len(const qg_twists* t) { return (t && !t->t.obs_perms.empty()) ? (int64_t)t->t.obs_perms[0].size() : 0; }
int64_t qg_twists_act_len(const qg_twists* t) { return (t && !t->t.act_perms.empty()) ? (int64_t)t->t.act_perms[0].size() : 0; }
int qg_twists_copy(const qg_twists* t, int64_t* obs, int64_t* act) {
    if (!t) { set_error("null twists"); return QG_ERR_INVALID; }
    for (const auto& p : t->t.obs_perms) { if (obs) { std::copy(p.begin(), p.end(), obs); obs += p.size(); } }
    for (const auto& p : t->t.act_perms) { if (act) { std::copy(p.begin(), p.end(), act); act += p.size(); } }
    return QG_OK;
}

int64_t qg_workspace_bytes(const qg_config* cfg, int64_t batch) {
    Layout L; int rc = make_layout(cfg, L);
    if (rc != QG_OK) return rc;
    if (batch < 0) { set_error("batch must be >= 0"); return QG_ERR_INVALID; }
    Twists tw; rc = pauli_perms(cfg, tw);
    if (rc != QG_OK) return rc;
    std::vector<uint32_t> pg;
    if (cfg->env_kind == QG_ENV_PAULI_NETWORK) pauli_gen_tables(cfg, pg);
    return plan_ws(L, batch, (int64_t)tw.act_perms.size(), (int64_t)pg.size()).total;
}

int qg_create(const qg_config* cfg, int32_t device, int64_t batch, void* workspace_dev, qg_engine** out) {
    if (!out) { set_error("null out"); return QG_ERR_INVALID; }
    *out = nullptr;
    Layout L; int rc = make_layout(cfg, L);
    if (rc != QG_OK) return rc;
    if (batch < 0) { set_error("batch must be >= 0"); return QG_ERR_INVALID; }
    int ndev = 0;
    CUDA_OK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) { set_error("no such CUDA device (the engine has no CPU fallback)"); return QG_ERR_CUDA; }
    CUDA_OK(cudaSetDevice(device));
    Twists tw; rc = pauli_perms(cfg, tw);
    if (rc != QG_OK) return rc;
    if (tw.act_perms.size() > 65535) { set_error("PauliNetwork: more than 65535 qubit permutations are not supported"); return QG_ERR_UNSUPPORTED; }

    qg_engine* e = new (std::nothrow) qg_engine();
    if (!e) { set_error("out of memory"); return QG_ERR_INVALID; }
    e->cfg = *cfg; e->gates.assign(cfg->gateset, cfg->gateset + cfg->num_gates); e->cfg.gateset = e->gates.data();
    e->L = L; e->device = device; e->B = batch; e->Bpad = align_up(std::max<int64_t>(batch, 1), 32);
    e->nperms = (int)tw.act_perms.size();
#ifdef QG_TOOLS_KNOBS      // A/B switches for tools/ builds (make EXTRA=-DQG_TOOLS_KNOBS); the product library reads no environment variables
    if (const char* v = std::getenv("QG_PDL")) e->pdl_mode = std::atoi(v);
    if (const char* v = std::getenv("QG_L2_PERSIST_MB")) {                 // A/B runs: persisting-L2 window over the replay's action stream
        int mx = 0, win = 0;
        cudaDeviceGetAttribute(&mx, cudaDevAttrMaxPersistingL2CacheSize, device);
        cudaDeviceGetAttribute(&win, cudaDevAttrMaxAccessPolicyWindowSize, device);
        const size_t want = (size_t)std::atoi(v) << 20;
        e->l2_persist_bytes = std::min({want, (size_t)mx, (size_t)win});
        if (e->l2_persist_bytes > 0) cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, e->l2_persist_bytes);
    }
    if (const char* v = std::getenv("QG_INV_REG")) e->inv_bucket_enabled = std::atoi(v) != 0;
    if (const char* v = std::getenv("QG_INV_SYMPLECTIC")) e->all_symplectic = std::atoi(v) != 0;   // 0: never use the transpose shortcut
    if (const char* v = std::getenv("QG_STAGGER_NS")) e->stagger_ns = std::atoi(v);
    if (const char* v = std::getenv("QG_EPW")) e->epw_forced = std::atoi(v);
    if (const char* v = std::getenv("QG_REPLAY_CTAS")) e->replay_ctas = std::atoi(v);
    if (const char* v = std::getenv("QG_STEP_CTAS")) e->step_ctas = std::atoi(v);
    if (const char* v = std::getenv("QG_PAIR")) e->pair_forced = std::atoi(v) > 0 ? 1 : -1;      // 0: single-warp tiles in replay launches too
#endif
    { int v = 0; if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && v > 0) e->num_sms = v; }
    // replay stagger (warp k of an SM starting k slab-times late so that the warps do not alternate between the step logic and the
    // expansion in lock-step): measured on the final kernel, 1.600 ms with it and 1.594 ms without (65 536 envs): off unless asked for
    std::vector<uint32_t> pg;
    if (cfg->env_kind == QG_ENV_PAULI_NETWORK) pauli_gen_tables(cfg, pg);
    const WsPlan p = plan_ws(L, batch, e->nperms, (int64_t)pg.size());
    auto fail = [&](int code) { qg_destroy(e); return code; };
    if (workspace_dev) {
        if (reinterpret_cast<uintptr_t>(workspace_dev) & 255) { set_error("workspace must be 256-byte aligned"); return fail(QG_ERR_INVALID); }
        e->ws = (uint8_t*)workspace_dev;
    } else {
        cudaError_t ce = cudaMalloc(&e->ws, (size_t)p.total);
        if (ce != cudaSuccess) { set_error(std::string("cudaMalloc workspace: ") + cudaGetErrorString(ce)); e->ws = nullptr; return fail(QG_ERR_CUDA); }
        e->owns_ws = true;
    }
    // shared-memory plan: each warp owns [W | SCR | OW] words x kStride for its 32 envs
    const int words = L.W + L.SCR + L.OW;
    e->sm_warp_words = words * kStride; e->sm_scr = L.W * kStride; e->sm_obs = (L.W + L.SCR) * kStride;
    // observations that are not whole words per environment are expanded from the tile's concatenated bit stream (expand_cat): obs words per
    // 32-env tile; a Permutation too wide for a bit stream (OW == 0) keeps the direct byte test
    e->cat_words = ((L.obs_size & 31) != 0 && !(L.kind == QG_ENV_PERMUTATION && L.OW == 0)) ? L.obs_size : 0;
    const int wts_words = ((int64_t)(L.A | 1) * 32 * 4 <= 16 * 1024) ? (L.A | 1) * 32 : 0;
    {
        const int region = e->sm_warp_words + std::max(e->cat_words, wts_words);
        const int pair_w = 2 * std::max({L.SW * kStride, L.OW * kStride, e->cat_words}) + 12;
        e->smem_bytes = ((size_t)kLutWords + (size_t)std::max(region * kWarpsPerCta, region + pair_w)) * 4;   // the largest layout a launch may ask for
    }
    if (e->smem_bytes > 200 * 1024) { set_error("configuration needs more shared memory than one SM has"); return fail(QG_ERR_UNSUPPORTED); }
    e->magic_obs = magic40((uint32_t)L.obs_size); e->magic_A = magic40((uint32_t)L.A);
    auto magic32 = [](uint32_t d) { return d <= 1 ? 0u : (uint32_t)(((1ull << 32) + d - 1) / d); };
    e->magic_vpe = magic32((uint32_t)L.obs_size / 4); e->magic_a4 = magic32((uint32_t)L.A / 4);
    rc = prepare_kernels(e);
    if (rc != QG_OK) return fail(rc);

    DevCfg& d = e->dc;
    d.kind = L.kind; d.n = L.n; d.D = L.D; d.A = L.A; d.obs_size = L.obs_size; d.obs_cols = L.obs_cols;
    d.SW = L.SW; d.MW = L.MW; d.W = L.W; d.off_lastg = L.off_lastg; d.off_lastcx = L.off_lastcx; d.off_state = L.off_state; d.off_extra = L.off_extra; d.OW = L.OW;
    d.max_depth = cfg->max_depth; d.depth_slope = cfg->depth_slope; d.difficulty = cfg->difficulty;
    d.add_inverts = (L.kind != QG_ENV_PAULI_NETWORK && cfg->add_inverts) ? 1 : 0; d.track = cfg->track_solution ? 1 : 0; d.sol_cap = cfg->track_solution ? L.sol_cap : 0;
    d.max_rot = L.max_rot; d.Rtot = L.Rtot; d.CW = L.CW; d.nperms = e->nperms;
    d.w0 = cfg->w_n_cnots; d.w1 = cfg->w_n_layers_cnots; d.w2 = cfg->w_n_layers; d.w3 = cfg->w_n_gates; d.plr = cfg->pauli_layer_reward;
    d.B = batch; d.Bpad = e->Bpad;
    d.rec = (uint32_t*)(e->ws + p.rec); d.sol = (uint32_t*)(e->ws + p.sol); d.ret = (float*)(e->ws + p.ret);
    d.gates = (const uint32_t*)(e->ws + p.gates); d.ident = (const uint32_t*)(e->ws + p.ident);
    d.qperms = (const uint8_t*)(e->ws + p.qperms); d.aperms = (const uint16_t*)(e->ws + p.aperms); d.pgen = (const uint32_t*)(e->ws + p.pgen);
    d.seed = 0; d.first_id = 0;
    d.magic_n = (uint32_t)(((1ull << 32) + (uint32_t)L.n - 1) / (uint32_t)L.n);
    d.row_shift = -1;
    if ((L.kind == QG_ENV_LINEAR_FUNCTION || L.kind == QG_ENV_CLIFFORD) && L.D >= 1 && L.D <= 32 && (L.D & (L.D - 1)) == 0) {
        int sh = 0; while ((1 << sh) < L.D) ++sh;
        d.row_shift = sh;
    }
#ifdef QG_TOOLS_KNOBS
    if (const char* v = std::getenv("QG_ROW_POW2")) { if (std::atoi(v) == 0) d.row_shift = -1; }      // A/B runs
#endif
    e->staged = (uint32_t*)(e->ws + p.staged);
    e->snap = (uint32_t*)(e->ws + p.snap);
    e->io_actions = (int32_t*)(e->ws + p.io_actions); e->io_coins = e->ws + p.io_coins; e->io_reward = (float*)(e->ws + p.io_reward);
    e->io_done = e->ws + p.io_done; e->io_success = e->ws + p.io_success; e->best = (unsigned long long*)(e->ws + p.best);

    // constant tables
    std::vector<uint32_t> gt((size_t)L.A);
    for (int i = 0; i < L.A; ++i) gt[i] = (uint32_t)e->gates[i].kind | ((uint32_t)e->gates[i].q0 << 8) | ((uint32_t)(e->gates[i].kind >= QG_CX ? e->gates[i].q1 : 0) << 16);
    std::vector<uint32_t> ident((size_t)L.PW, 0); pack_identity(L, ident.data());
    cudaError_t ce = cudaMemcpy((void*)d.gates, gt.data(), gt.size() * 4, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess) ce = cudaMemcpy((void*)d.ident, ident.data(), (size_t)L.SW * 4, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess && e->nperms > 0) {
        std::vector<uint8_t> qp((size_t)e->nperms * L.n); std::vector<uint16_t> ap((size_t)e->nperms * L.A);
        for (int k = 0; k < e->nperms; ++k) {
            for (int q = 0; q < L.n; ++q) qp[(size_t)k * L.n + q] = (uint8_t)tw.obs_perms[k][q];
            for (int g = 0; g < L.A; ++g) ap[(size_t)k * L.A + g] = (uint16_t)tw.act_perms[k][g];
        }
        ce = cudaMemcpy((void*)d.qperms, qp.data(), qp.size(), cudaMemcpyHostToDevice);
        if (ce == cudaSuccess) ce = cudaMemcpy((void*)d.aperms, ap.data(), ap.size() * 2, cudaMemcpyHostToDevice);
    }
    if (ce == cudaSuccess && !pg.empty()) ce = cudaMemcpy((void*)d.pgen, pg.data(), pg.size() * 4, cudaMemcpyHostToDevice);
    if (ce == cudaSuccess) ce = cudaMallocHost(&e->h_best, 64);
    if (ce != cudaSuccess) { set_error(std::string("engine table upload: ") + cudaGetErrorString(ce)); return fail(QG_ERR_CUDA); }
    // constructor state: identity, depth 1, success, reward 1.0 (permutation.rs:75-98, clifford.rs:205-236, pauli.rs:354-409)
    ce = cudaMemcpy(e->staged, ident.data(), (size_t)L.PW * 4, cudaMemcpyHostToDevice);
    if (ce != cudaSuccess) { set_error(std::string("engine init: ") + cudaGetErrorString(ce)); return fail(QG_ERR_CUDA); }
    rc = launch_load(e, 0, batch, batch, 1u, 0);
    if (rc != QG_OK) return fail(rc);
    ce = cudaStreamSynchronize(0);
    if (ce != cudaSuccess) { set_error(std::string("engine init: ") + cudaGetErrorString(ce)); return fail(QG_ERR_CUDA); }
    *out = e;
    return QG_OK;
}

void qg_destroy(qg_engine* e) {
    if (!e) return;
    if (e->h_staged) cudaFreeHost(e->h_staged);
    if (e->h_best) cudaFreeHost(e->h_best);
    for (int b = 0; b < 2; ++b) {
        if (e->rp_actions[b]) cudaFree(e->rp_actions[b]);
        if (e->rp_coins[b]) cudaFree(e->rp_coins[b]);
        if (e->rp_reward[b]) cudaFree(e->rp_reward[b]);
        if (e->rp_done[b]) cudaFree(e->rp_done[b]);
        if (e->rp_success[b]) cudaFree(e->rp_success[b]);
        if (e->rp_ev_in[b]) cudaEventDestroy(e->rp_ev_in[b]);
        if (e->rp_ev_run[b]) cudaEventDestroy(e->rp_ev_run[b]);
        if (e->rp_ev_out[b]) cudaEventDestroy(e->rp_ev_out[b]);
    }
    if (e->rp_ev_start) cudaEventDestroy(e->rp_ev_start);
    if (e->rp_in) cudaStreamDestroy(e->rp_in);
    if (e->rp_out) cudaStreamDestroy(e->rp_out);
    extras_release(e);
    if (e->owns_ws && e->ws) cudaFree(e->ws);
    delete e;
}

int64_t qg_batch(const qg_engine* e) { return e ? e->B : 0; }
int32_t qg_num_actions(const qg_engine* e) { return e ? e->L.A : 0; }
int32_t qg_obs_size(const qg_engine* e) { return e ? e->L.obs_size : 0; }
int qg_obs_shape(const qg_engine* e, int32_t out_shape[2]) {
    if (!e) { set_error("null engine"); return QG_ERR_INVALID; }
    out_shape[0] = e->L.obs_rows; out_shape[1] = e->L.obs_cols; return QG_OK;
}
int qg_set_difficulty(qg_engine* e, int32_t difficulty) {
    if (!e || difficulty < 0) { set_error("bad difficulty"); return QG_ERR_INVALID; }
    e->cfg.difficulty = difficulty; e->dc.difficulty = difficulty; return QG_OK;
}
int32_t qg_get_difficulty(const qg_engine* e) { return e ? e->cfg.difficulty : 0; }

namespace {
// `payloads` payloads packed once each, env first + i loads payload i / group
int set_state_impl(qg_engine* e, const int64_t* states_host, int64_t stride, int64_t first, int64_t count, int64_t payloads, int64_t group, qg_stream stream) {
    if (count == 0) return QG_OK;
    CUDA_OK(cudaSetDevice(e->device));
    int rc = ensure_host_staging(e, payloads * e->L.PW);
    if (rc != QG_OK) return rc;
    for (int64_t i = 0; i < payloads; ++i) {
        int64_t used = 0;
        rc = pack_state(&e->cfg, e->L, states_host + i * stride, stride, e->h_staged + i * e->L.PW, &used);
        if (rc != QG_OK) return rc;
        if (e->L.kind == QG_ENV_CLIFFORD && e->all_symplectic && !is_symplectic(e->L, e->h_staged + i * e->L.PW)) e->all_symplectic = false;
    }
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_OK(cudaMemcpyAsync(e->staged, e->h_staged, (size_t)payloads * e->L.PW * 4, cudaMemcpyHostToDevice, st));
    rc = launch_load(e, first, count, group, (uint32_t)e->cfg.max_depth, st);
    if (rc != QG_OK) return rc;
    CUDA_OK(cudaStreamSynchronize(st));   // the pinned staging buffer is reused by the next call
    return QG_OK;
}
}  // namespace

int qg_set_state(qg_engine* e, const int64_t* states_host, int64_t stride, int64_t first, int64_t count, int32_t broadcast, qg_stream stream) {
    if (!e || !states_host) { set_error("null argument"); return QG_ERR_INVALID; }
    if (first < 0 || count < 0 || first + count > e->B) { set_error("set_state: env range outside the batch"); return QG_ERR_INVALID; }
    // broadcast: one payload read by all `count` envs; otherwise one payload per env
    return set_state_impl(e, states_host, stride, first, count, broadcast ? 1 : count, broadcast ? count : 1, stream);
}

int qg_set_state_grouped(qg_engine* e, const int64_t* states_host, int64_t stride, int64_t num_states, int64_t group, qg_stream stream) {
    if (!e || !states_host) { set_error("null argument"); return QG_ERR_INVALID; }
    if (group <= 0 || num_states < 0 || num_states > e->B / group) {
        set_error("set_state_grouped: group must be >= 1 and num_states * group within the batch"); return QG_ERR_INVALID;
    }
    return set_state_impl(e, states_host, stride, 0, num_states * group, num_states, group, stream);
}

namespace {
int launch_reset(qg_engine* e, uint64_t seed, int64_t first_env_id, int which, const uint8_t* select_dev, cudaStream_t st, const uint64_t* seed_dev = nullptr) {
    CUDA_OK(cudaSetDevice(e->device));
    if (!seed_dev) e->dc.seed = seed;
    e->dc.first_id = first_env_id; e->dc.seed_dev = seed_dev;
    if (e->B == 0) return QG_OK;
    if (e->L.kind == QG_ENV_PAULI_NETWORK) {
        const int words = e->L.SW + e->L.XW + 3 * e->L.Rtot;
        const int fl = e->cfg.final_pauli_layers >= 0 ? e->cfg.final_pauli_layers : e->cfg.max_rotations + 2;
        k_reset_pauli<32><<<(unsigned)((e->B + 31) / 32), 32, (size_t)words * 32 * 4, st>>>(e->dc, std::max(e->cfg.pauli_diff_scale, 1), e->cfg.num_qubits_decay, fl,
                                                                                              which, select_dev);
        CUDA_OK(cudaGetLastError());
        return QG_OK;
    }
    const unsigned grid = (unsigned)((e->B + 63) / 64);
    const size_t sm = (size_t)e->L.SW * 64 * 4;
    switch (e->L.kind) {
        case QG_ENV_PERMUTATION: k_reset<QG_ENV_PERMUTATION, 64><<<grid, 64, sm, st>>>(e->dc, which, select_dev); break;
        case QG_ENV_LINEAR_FUNCTION: k_reset<QG_ENV_LINEAR_FUNCTION, 64><<<grid, 64, sm, st>>>(e->dc, which, select_dev); break;
        default: k_reset<QG_ENV_CLIFFORD, 64><<<grid, 64, sm, st>>>(e->dc, which, select_dev); break;
    }
    CUDA_OK(cudaGetLastError());
    return QG_OK;
}
}  // namespace

int qg_reset(qg_engine* e, uint64_t seed, int64_t first_env_id, qg_stream stream) {
    if (!e) { set_error("null engine"); return QG_ERR_INVALID; }
    return launch_reset(e, seed, first_env_id, RESET_ALL, nullptr, (cudaStream_t)stream);
}

int qg_reset_select(qg_engine* e, uint64_t seed, int64_t first_env_id, const uint8_t* select_dev, qg_stream stream) {
    if (!e) { set_error("null engine"); return QG_ERR_INVALID; }
    return launch_reset(e, seed, first_env_id, select_dev ? RESET_SELECT : RESET_FINAL, select_dev, (cudaStream_t)stream);
}

int qg_reset_select_dev(qg_engine* e, const uint64_t* seed_dev, int64_t first_env_id, const uint8_t* select_dev, qg_stream stream) {
    if (!e || !seed_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    const int rc = launch_reset(e, 0, first_env_id, select_dev ? RESET_SELECT : RESET_FINAL, select_dev, (cudaStream_t)stream, seed_dev);
    e->dc.seed_dev = nullptr;
    return rc;
}

int qg_snapshot(qg_engine* e, qg_stream stream) {
    if (!e) { set_error("null engine"); return QG_ERR_INVALID; }
    CUDA_OK(cudaMemcpyAsync(e->snap, e->dc.rec, (size_t)e->L.W * e->Bpad * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    e->has_snap = true;
    return QG_OK;
}
int qg_restore(qg_engine* e, qg_stream stream) {
    if (!e) { set_error("null engine"); return QG_ERR_INVALID; }
    if (!e->has_snap) { set_error("qg_restore without a snapshot"); return QG_ERR_INVALID; }
    CUDA_OK(cudaMemcpyAsync(e->dc.rec, e->snap, (size_t)e->L.W * e->Bpad * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
    return QG_OK;
}

int qg_step(qg_engine* e, const int32_t* actions_dev, const uint8_t* coins_dev, const uint32_t* perm_raw_dev, float* obs_dev, uint8_t* mask_dev,
            float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, qg_stream stream) {
    if (!e || !actions_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    StepArgs a{}; a.actions = actions_dev; a.coins = coins_dev; a.perm_raw = perm_raw_dev; a.obs = obs_dev; a.mask = mask_dev;
    a.reward = reward_dev; a.done = done_dev; a.success = success_dev;
    return launch_step(e, MODE_STEP, a, (cudaStream_t)stream);
}

int qg_replay(qg_engine* e, int32_t num_steps, const int32_t* actions_dev, const uint8_t* coins_dev, const uint32_t* perm_raw_dev,
              float* obs_dev, uint8_t* mask_dev, int32_t ring, float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, qg_stream stream) {
    if (!e || !actions_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (num_steps < 0 || ring < 1) { set_error("qg_replay: num_steps must be >= 0 and ring >= 1"); return QG_ERR_INVALID; }
    if (num_steps == 0) return QG_OK;
    StepArgs a{}; a.actions = actions_dev; a.coins = coins_dev; a.perm_raw = perm_raw_dev; a.obs = obs_dev; a.mask = mask_dev;
    a.reward = reward_dev; a.done = done_dev; a.success = success_dev;
    a.nsteps = num_steps; a.ring = ring; a.in_stride = e->B; a.out_stride = e->B;
    return launch_step(e, MODE_STEP, a, (cudaStream_t)stream);
}

// Episode replay with HOST buffers.  Pinned buffers: one launch, the kernel accesses them itself.  Pageable buffers: pipelined in chunks
// of steps over three streams: the copy-in stream uploads the actions of chunk c+1 while the caller's stream replays chunk c (one
// fused launch per chunk) and the copy-out stream downloads the rewards / flags of chunk c-1.
int qg_replay_host(qg_engine* e, int32_t num_steps, const int32_t* actions_host, const uint8_t* coins_host, float* obs_dev, uint8_t* mask_dev,
                   int32_t ring, float* reward_host, uint8_t* done_host, uint8_t* success_host, qg_stream stream) {
    if (!e || !actions_host) { set_error("null argument"); return QG_ERR_INVALID; }
    if (num_steps < 0 || ring < 1) { set_error("qg_replay_host: num_steps must be >= 0 and ring >= 1"); return QG_ERR_INVALID; }
    if (num_steps == 0 || e->B == 0) return QG_OK;
    CUDA_OK(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t B = (size_t)e->B;
    bool zero_copy = true;
#ifdef QG_TOOLS_KNOBS
    if (const char* zc = std::getenv("QG_REPLAY_ZEROCOPY")) zero_copy = std::atoi(zc) != 0;      // A/B runs: 0 = always stage through device buffers
#endif
    if (zero_copy) {
        // pinned host buffers: ONE launch for the whole episode, the kernel reading the actions (one step ahead) and writing reward /
        // done / success over PCIe itself (see qg_step_host); no staging copies, no chunk boundaries.  Measured at 65 536 envs:
        // 5.20 x 10^9 env-steps/s against 4.49 x 10^9 for the chunked copy pipeline below (and 5.09 x 10^9 device resident: the three
        // small output streams leave over PCIe instead of taking HBM bandwidth)
        void* const m_act = mapped_host(actions_host); void* const m_coin = mapped_host(coins_host);
        void* const m_rew = mapped_host(reward_host); void* const m_done = mapped_host(done_host); void* const m_suc = mapped_host(success_host);
        if (m_act && (!coins_host || m_coin) && (!reward_host || m_rew) && (!done_host || m_done) && (!success_host || m_suc)) {
            StepArgs a{}; a.actions = (const int32_t*)m_act; a.coins = (const uint8_t*)m_coin; a.obs = obs_dev; a.mask = mask_dev;
            a.reward = (float*)m_rew; a.done = (uint8_t*)m_done; a.success = (uint8_t*)m_suc;
            a.nsteps = num_steps; a.ring = ring; a.slot0 = 0; a.in_stride = e->B; a.out_stride = e->B;
            const int rc = launch_step(e, MODE_STEP, a, st);
            if (rc != QG_OK) return rc;
            CUDA_OK(cudaStreamSynchronize(st));
            return QG_OK;
        }
    }
    if (!e->rp_in) {
        // chunk: about 1 MB of actions per upload, at least 1 and at most 32 steps (the first upload and the last download are not
        // overlapped with compute; measured at 65 536 envs: chunks of 16 / 8 / 4 / 2 steps -> 4.35 / 4.45 / 4.51 / 3.67 x 10^9 env-steps/s)
        e->rp_chunk = (int)std::min<int64_t>(32, std::max<int64_t>(1, (int64_t)(1 << 20) / std::max<int64_t>((int64_t)B * 4, 1)));
#ifdef QG_TOOLS_KNOBS
        if (const char* v = std::getenv("QG_REPLAY_CHUNK")) e->rp_chunk = std::max(1, std::atoi(v));      // A/B runs
#endif
        CUDA_OK(cudaStreamCreateWithFlags(&e->rp_in, cudaStreamNonBlocking));
        CUDA_OK(cudaStreamCreateWithFlags(&e->rp_out, cudaStreamNonBlocking));
        CUDA_OK(cudaEventCreateWithFlags(&e->rp_ev_start, cudaEventDisableTiming));
        for (int b = 0; b < 2; ++b) {
            const size_t n = (size_t)e->rp_chunk * B;
            CUDA_OK(cudaMalloc(&e->rp_actions[b], n * 4)); CUDA_OK(cudaMalloc(&e->rp_coins[b], n));
            CUDA_OK(cudaMalloc(&e->rp_reward[b], n * 4)); CUDA_OK(cudaMalloc(&e->rp_done[b], n)); CUDA_OK(cudaMalloc(&e->rp_success[b], n));
            CUDA_OK(cudaEventCreateWithFlags(&e->rp_ev_in[b], cudaEventDisableTiming));
            CUDA_OK(cudaEventCreateWithFlags(&e->rp_ev_run[b], cudaEventDisableTiming));
            CUDA_OK(cudaEventCreateWithFlags(&e->rp_ev_out[b], cudaEventDisableTiming));
        }
    }
    const int chunk = e->rp_chunk, nchunks = (num_steps + chunk - 1) / chunk;
    CUDA_OK(cudaEventRecord(e->rp_ev_start, st));
    CUDA_OK(cudaStreamWaitEvent(e->rp_in, e->rp_ev_start, 0));
    for (int c = 0; c < nchunks; ++c) {
        const int b = c & 1, t0 = c * chunk, ns = std::min(chunk, num_steps - t0);
        const size_t n = (size_t)ns * B, o = (size_t)t0 * B;
        if (c >= 2) CUDA_OK(cudaStreamWaitEvent(e->rp_in, e->rp_ev_run[b], 0));          // chunk c-2 has consumed this buffer
        CUDA_OK(cudaMemcpyAsync(e->rp_actions[b], actions_host + o, n * 4, cudaMemcpyHostToDevice, e->rp_in));
        if (coins_host) CUDA_OK(cudaMemcpyAsync(e->rp_coins[b], coins_host + o, n, cudaMemcpyHostToDevice, e->rp_in));
        CUDA_OK(cudaEventRecord(e->rp_ev_in[b], e->rp_in));
        CUDA_OK(cudaStreamWaitEvent(st, e->rp_ev_in[b], 0));
        if (c >= 2) CUDA_OK(cudaStreamWaitEvent(st, e->rp_ev_out[b], 0));                // chunk c-2's results have left this buffer
        StepArgs a{}; a.actions = e->rp_actions[b]; a.coins = coins_host ? e->rp_coins[b] : nullptr; a.obs = obs_dev; a.mask = mask_dev;
        a.reward = reward_host ? e->rp_reward[b] : nullptr; a.done = done_host ? e->rp_done[b] : nullptr; a.success = success_host ? e->rp_success[b] : nullptr;
        a.nsteps = ns; a.ring = ring; a.slot0 = t0 % ring; a.in_stride = e->B; a.out_stride = e->B;
        const int rc = launch_step(e, MODE_STEP, a, st);
        if (rc != QG_OK) return rc;
        CUDA_OK(cudaEventRecord(e->rp_ev_run[b], st));
        CUDA_OK(cudaStreamWaitEvent(e->rp_out, e->rp_ev_run[b], 0));
        if (reward_host) CUDA_OK(cudaMemcpyAsync(reward_host + o, e->rp_reward[b], n * 4, cudaMemcpyDeviceToHost, e->rp_out));
        if (done_host) CUDA_OK(cudaMemcpyAsync(done_host + o, e->rp_done[b], n, cudaMemcpyDeviceToHost, e->rp_out));
        if (success_host) CUDA_OK(cudaMemcpyAsync(success_host + o, e->rp_success[b], n, cudaMemcpyDeviceToHost, e->rp_out));
        CUDA_OK(cudaEventRecord(e->rp_ev_out[b], e->rp_out));
    }
    for (int b = 0; b < std::min(2, nchunks); ++b) CUDA_OK(cudaStreamWaitEvent(st, e->rp_ev_out[b], 0));
    CUDA_OK(cudaStreamSynchronize(st));
    return QG_OK;
}

int qg_step_host(qg_engine* e, const int32_t* actions_host, const uint8_t* coins_host, float* obs_dev, uint8_t* mask_dev,
                 float* reward_host, uint8_t* done_host, uint8_t* success_host, qg_stream stream) {
    if (!e || !actions_host) { set_error("null argument"); return QG_ERR_INVALID; }
    CUDA_OK(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t B = (size_t)e->B;
    // Pinned host buffers are mapped into the device's address space (unified addressing): the kernel then reads the actions and writes
    // reward / done / success over PCIe itself, and the call is one launch + one synchronisation instead of up to five copies around it.
    void* const m_act = mapped_host(actions_host); void* const m_coin = mapped_host(coins_host);
    void* const m_rew = mapped_host(reward_host); void* const m_done = mapped_host(done_host); void* const m_suc = mapped_host(success_host);
    if (m_act && (!coins_host || m_coin) && (!reward_host || m_rew) && (!done_host || m_done) && (!success_host || m_suc)) {
        StepArgs a{}; a.actions = (const int32_t*)m_act; a.coins = (const uint8_t*)m_coin; a.obs = obs_dev; a.mask = mask_dev;
        a.reward = (float*)m_rew; a.done = (uint8_t*)m_done; a.success = (uint8_t*)m_suc;
        const int rc = launch_step(e, MODE_STEP, a, st);
        if (rc != QG_OK) return rc;
        CUDA_OK(cudaStreamSynchronize(st));
        return QG_OK;
    }
    CUDA_OK(cudaMemcpyAsync(e->io_actions, actions_host, B * 4, cudaMemcpyHostToDevice, st));
    if (coins_host) CUDA_OK(cudaMemcpyAsync(e->io_coins, coins_host, B, cudaMemcpyHostToDevice, st));
    StepArgs a{}; a.actions = e->io_actions; a.coins = coins_host ? e->io_coins : nullptr; a.obs = obs_dev; a.mask = mask_dev;
    a.reward = e->io_reward; a.done = e->io_done; a.success = e->io_success;
    const int rc = launch_step(e, MODE_STEP, a, st);
    if (rc != QG_OK) return rc;
    if (reward_host) CUDA_OK(cudaMemcpyAsync(reward_host, e->io_reward, B * 4, cudaMemcpyDeviceToHost, st));
    if (done_host) CUDA_OK(cudaMemcpyAsync(done_host, e->io_done, B, cudaMemcpyDeviceToHost, st));
    if (success_host) CUDA_OK(cudaMemcpyAsync(success_host, e->io_success, B, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    return QG_OK;
}

int qg_observe(qg_engine* e, const uint32_t* perm_raw_dev, float* obs_dev, qg_stream stream) {
    if (!e || !obs_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    StepArgs a{}; a.perm_raw = perm_raw_dev; a.obs = obs_dev;
    return launch_step(e, MODE_OBSERVE, a, (cudaStream_t)stream);
}
int qg_masks(qg_engine* e, uint8_t* mask_dev, qg_stream stream) {
    if (!e || !mask_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    StepArgs a{}; a.mask = mask_dev;
    return launch_step(e, MODE_OBSERVE, a, (cudaStream_t)stream);
}
int qg_read_status(qg_engine* e, float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, int32_t* depth_dev, qg_stream stream) {
    if (!e) { set_error("null engine"); return QG_ERR_INVALID; }
    if (e->B == 0) return QG_OK;
    k_read_status<<<(unsigned)((e->B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(e->dc, reward_dev, done_dev, success_dev, depth_dev);
    CUDA_OK(cudaGetLastError());
    return QG_OK;
}
int qg_read_metrics(qg_engine* e, uint32_t* counts_dev, qg_stream stream) {
    if (!e || !counts_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (e->B == 0) return QG_OK;
    k_read_metrics<<<(unsigned)((e->B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(e->dc, counts_dev);
    CUDA_OK(cudaGetLastError());
    return QG_OK;
}
int qg_read_errors(qg_engine* e, uint32_t* flags_dev, qg_stream stream) {
    if (!e || !flags_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (e->B == 0) return QG_OK;
    k_read_errors<<<(unsigned)((e->B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(e->dc, flags_dev);
    CUDA_OK(cudaGetLastError());
    return QG_OK;
}

int qg_get_state_host(qg_engine* e, int64_t env, uint8_t* out_host, int64_t cap, int64_t* len, qg_stream stream) {
    if (!e || !out_host || !len) { set_error("null argument"); return QG_ERR_INVALID; }
    if (env < 0 || env >= e->B) { set_error("env index outside the batch"); return QG_ERR_INVALID; }
    CUDA_OK(cudaSetDevice(e->device));
    std::vector<uint32_t> col((size_t)e->L.W);
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_OK(cudaMemcpy2DAsync(col.data(), 4, e->dc.rec + env, (size_t)e->Bpad * 4, 4, (size_t)e->L.W, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    return unpack_state(e->L, col.data(), out_host, cap, len);
}

int qg_solution_host(qg_engine* e, int64_t env, uint32_t* out_host, int32_t cap, int32_t* len, qg_stream stream) {
    if (!e || !len) { set_error("null argument"); return QG_ERR_INVALID; }
    if (env < 0 || env >= e->B) { set_error("env index outside the batch"); return QG_ERR_INVALID; }
    CUDA_OK(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    uint32_t flags = 0;
    CUDA_OK(cudaMemcpyAsync(&flags, e->dc.rec + (size_t)HD_FLAGS * e->Bpad + env, 4, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    const int n = (int)(flags >> FL_LEN_SHIFT);
    *len = n;
    if (n == 0 || !out_host) return QG_OK;
    if (cap < n) { set_error("solution buffer too small"); return QG_ERR_INVALID; }
    std::vector<uint32_t> col((size_t)n);
    CUDA_OK(cudaMemcpy2DAsync(col.data(), 4, e->dc.sol + env, (size_t)e->Bpad * 4, 4, (size_t)n, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    if (e->L.kind == QG_ENV_PAULI_NETWORK) { std::copy(col.begin(), col.end(), out_host); return QG_OK; }
    // solution ++ reverse(solution_inv) (clifford.rs:376-381); bit 31 marks entries logged while inverted
    int k = 0;
    for (int i = 0; i < n; ++i) if (!(col[i] & 0x80000000u)) out_host[k++] = col[i];
    for (int i = n - 1; i >= 0; --i) if (col[i] & 0x80000000u) out_host[k++] = col[i] & 0x7FFFFFFFu;
    return QG_OK;
}

int qg_search_begin(qg_engine* e, uint64_t seed, int64_t first_rollout_id, qg_stream stream) {
    if (!e) { set_error("null engine"); return QG_ERR_INVALID; }
    if (first_rollout_id < 0 || first_rollout_id + e->B > 0x3FFFFFFFll) { set_error("rollout ids must stay below 2^30"); return QG_ERR_INVALID; }
    e->dc.seed = seed; e->dc.first_id = first_rollout_id;
    if (e->B == 0) return QG_OK;
    k_fill_f32<<<(unsigned)((e->B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(e->dc.ret, e->B, 0.0f);
    CUDA_OK(cudaGetLastError());
    return QG_OK;
}

int qg_search_step(qg_engine* e, const float* weights_dev, int32_t deterministic, float* obs_dev, uint8_t* mask_dev, int32_t* chosen_dev,
                   int32_t* num_active_dev, qg_stream stream) {
    if (!e || !weights_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    if (num_active_dev) CUDA_OK(cudaMemsetAsync(num_active_dev, 0, 4, st));
    StepArgs a{}; a.weights = weights_dev; a.deterministic = deterministic; a.obs = obs_dev; a.mask = mask_dev; a.chosen = chosen_dev; a.num_active = num_active_dev;
    return launch_step(e, MODE_SEARCH, a, st);
}

int qg_collect_step(qg_engine* e, uint64_t seed, const float* weights_dev, int32_t deterministic, float* obs_dev, uint8_t* mask_dev, int32_t* chosen_dev,
                    float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, qg_stream stream) {
    if (!e || !weights_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    e->dc.seed = seed;
    StepArgs a{}; a.weights = weights_dev; a.deterministic = deterministic; a.obs = obs_dev; a.mask = mask_dev; a.chosen = chosen_dev;
    a.reward = reward_dev; a.done = done_dev; a.success = success_dev;
    return launch_step(e, MODE_SEARCH, a, (cudaStream_t)stream);
}

int qg_collect_step_dev(qg_engine* e, const uint64_t* seed_dev, const float* weights_dev, int32_t deterministic, float* obs_dev, uint8_t* mask_dev,
                        int32_t* chosen_dev, float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, qg_stream stream) {
    if (!e || !weights_dev || !seed_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    e->dc.seed_dev = seed_dev;
    StepArgs a{}; a.weights = weights_dev; a.deterministic = deterministic; a.obs = obs_dev; a.mask = mask_dev; a.chosen = chosen_dev;
    a.reward = reward_dev; a.done = done_dev; a.success = success_dev;
    const int rc = launch_step(e, MODE_SEARCH, a, (cudaStream_t)stream);
    e->dc.seed_dev = nullptr;
    return rc;
}

int qg_collect_step_twisted_dev(qg_engine* e, const uint64_t* seed_dev, const float* weights_dev, const int32_t* act_perm_dev, const int32_t* twist_dev,
                                int32_t deterministic, int32_t* chosen_dev, int32_t* policy_chosen_dev, float* reward_dev, uint8_t* done_dev,
                                uint8_t* success_dev, qg_stream stream) {
    if (!e || !weights_dev || !seed_dev || !act_perm_dev || !twist_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    e->dc.seed_dev = seed_dev;
    StepArgs a{}; a.weights = weights_dev; a.deterministic = deterministic; a.chosen = chosen_dev;
    a.act_perm = act_perm_dev; a.twist = twist_dev; a.policy_chosen = policy_chosen_dev;
    a.reward = reward_dev; a.done = done_dev; a.success = success_dev;
    const int rc = launch_step(e, MODE_SEARCH, a, (cudaStream_t)stream);
    e->dc.seed_dev = nullptr;
    return rc;
}

int qg_gae(const float* reward_dev, const float* value_dev, const uint8_t* done_dev, const uint8_t* valid_dev, int32_t num_steps, int64_t batch,
           float gamma, float lambda, float* adv_dev, float* ret_dev, qg_stream stream) {
    if (!reward_dev || !value_dev || !done_dev || !adv_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (num_steps < 0 || batch < 0) { set_error("qg_gae: negative size"); return QG_ERR_INVALID; }
    if (num_steps == 0 || batch == 0) return QG_OK;
    k_gae<<<(unsigned)((batch + 127) / 128), 128, 0, (cudaStream_t)stream>>>(reward_dev, value_dev, done_dev, valid_dev, num_steps, batch, gamma, lambda, adv_dev, ret_dev);
    CUDA_OK(cudaGetLastError());
    return QG_OK;
}

int qg_twist_gather(const float* in_dev, float* out_dev, const int32_t* table_dev, const int32_t* index_dev, int64_t batch, int32_t len, qg_stream stream) {
    if (!in_dev || !out_dev || !table_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (batch < 0 || len <= 0) { set_error("qg_twist_gather: bad size"); return QG_ERR_INVALID; }
    if (in_dev == out_dev) { set_error("qg_twist_gather cannot run in place"); return QG_ERR_INVALID; }
    if (batch == 0) return QG_OK;
    const uint64_t magic = len == 1 ? 0ull : (~0ull / (uint64_t)len) + 1ull;   // ceil(2^64 / len) for len that is not a power of two, exact enough: see k_twist_gather
    const int64_t total = batch * (int64_t)len;
    const unsigned grid = (unsigned)std::min<int64_t>((total + 255) / 256, 148 * 16);
    k_twist_gather<<<grid, 256, 0, (cudaStream_t)stream>>>(in_dev, out_dev, table_dev, index_dev, batch, len, magic);
    CUDA_OK(cudaGetLastError());
    return QG_OK;
}

int qg_twist_bits(const uint32_t* in_bits_dev, uint32_t* out_bits_dev, int64_t batch, int32_t obs_size, int32_t num_qubits, int32_t dim,
                  const uint8_t* qperm_inv_dev, int32_t num_twists, const int32_t* index_dev, const uint64_t* seed_dev, int64_t first_env_id,
                  int32_t draw, int32_t* index_out_dev, qg_stream stream) {
    if (!in_bits_dev || !out_bits_dev || !qperm_inv_dev || (!index_dev && !seed_dev)) { set_error("null argument"); return QG_ERR_INVALID; }
    if (in_bits_dev == out_bits_dev) { set_error("qg_twist_bits cannot run in place"); return QG_ERR_INVALID; }
    if (batch < 0 || num_qubits < 1 || num_twists < 1 || draw < 0 || (dim != num_qubits && dim != 2 * num_qubits) || obs_size != dim * dim) {
        set_error("qg_twist_bits: bad size (obs_size must be dim * dim with dim = num_qubits or 2 * num_qubits)");
        return QG_ERR_INVALID;
    }
    if (batch == 0) return QG_OK;
    const int ow = (obs_size + 31) / 32;
    const int64_t total = batch * (int64_t)ow;
    const unsigned grid = (unsigned)std::min<int64_t>((total + 255) / 256, 148 * 16);
    k_twist_bits<<<grid, 256, 0, (cudaStream_t)stream>>>(in_bits_dev, out_bits_dev, ow, obs_size, num_qubits, dim, qperm_inv_dev, (uint32_t)num_twists,
                                                         index_dev, seed_dev, first_env_id, (uint32_t)draw, index_out_dev, batch);
    CUDA_OK(cudaGetLastError());
    return QG_OK;
}

// ---- packed-bit observation variants (SURVEY.md §8f row 3) ------------------------------------------------------------
int32_t qg_obs_words(const qg_engine* e) { return e ? (e->L.obs_size + 31) / 32 : 0; }

int qg_step_bits(qg_engine* e, const int32_t* actions_dev, const uint8_t* coins_dev, const uint32_t* perm_raw_dev, uint32_t* obs_bits_dev, uint8_t* mask_dev,
                 float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, qg_stream stream) {
    if (!e || !actions_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    StepArgs a{}; a.actions = actions_dev; a.coins = coins_dev; a.perm_raw = perm_raw_dev; a.obs_bits = obs_bits_dev; a.mask = mask_dev;
    a.reward = reward_dev; a.done = done_dev; a.success = success_dev;
    return launch_step(e, MODE_STEP, a, (cudaStream_t)stream);
}

int qg_replay_bits(qg_engine* e, int32_t num_steps, const int32_t* actions_dev, const uint8_t* coins_dev, const uint32_t* perm_raw_dev,
                   uint32_t* obs_bits_dev, uint8_t* mask_dev, int32_t ring, float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, qg_stream stream) {
    if (!e || !actions_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (num_steps < 0 || ring < 1) { set_error("qg_replay_bits: num_steps must be >= 0 and ring >= 1"); return QG_ERR_INVALID; }
    if (num_steps == 0) return QG_OK;
    StepArgs a{}; a.actions = actions_dev; a.coins = coins_dev; a.perm_raw = perm_raw_dev; a.obs_bits = obs_bits_dev; a.mask = mask_dev;
    a.reward = reward_dev; a.done = done_dev; a.success = success_dev;
    a.nsteps = num_steps; a.ring = ring; a.in_stride = e->B; a.out_stride = e->B;
    return launch_step(e, MODE_STEP, a, (cudaStream_t)stream);
}

int qg_observe_bits(qg_engine* e, const uint32_t* perm_raw_dev, uint32_t* obs_bits_dev, qg_stream stream) {
    if (!e || !obs_bits_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    StepArgs a{}; a.perm_raw = perm_raw_dev; a.obs_bits = obs_bits_dev;
    return launch_step(e, MODE_OBSERVE, a, (cudaStream_t)stream);
}

int qg_search_step_bits(qg_engine* e, const float* weights_dev, int32_t deterministic, uint32_t* obs_bits_dev, int32_t* chosen_dev,
                        int32_t* num_active_dev, qg_stream stream) {
    if (!e || !weights_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    if (num_active_dev) CUDA_OK(cudaMemsetAsync(num_active_dev, 0, 4, st));
    StepArgs a{}; a.weights = weights_dev; a.deterministic = deterministic; a.obs_bits = obs_bits_dev; a.chosen = chosen_dev; a.num_active = num_active_dev;
    return launch_step(e, MODE_SEARCH, a, st);
}

// ---- tree-search support: clone + step through record slots, cross-engine record copies -----------------------------------
namespace qg {
__global__ void k_copy_records(DevCfg dst, const int32_t* __restrict__ dst_slot, const uint32_t* __restrict__ src_rec, int64_t src_bpad, int W, int64_t count) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    const int64_t slot = dst_slot ? (int64_t)dst_slot[i] : i;
    for (int w = 0; w < W; ++w) {
        uint32_t v = src_rec[(size_t)w * src_bpad + i];
        if (w == HD_FLAGS) v &= (1u << FL_LEN_SHIFT) - 1u;       // the copy restarts its solution log
        dst.rec[(size_t)w * dst.Bpad + slot] = v;
    }
}
}  // namespace qg

int qg_step_slots(qg_engine* e, int64_t count, const int32_t* src_slot_dev, const int32_t* dst_slot_dev, const int32_t* actions_dev, float* obs_dev,
                  uint32_t* obs_bits_dev, uint8_t* mask_dev, float* reward_dev, uint8_t* done_dev, uint8_t* success_dev, qg_stream stream) {
    if (!e || !src_slot_dev || !dst_slot_dev || !actions_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (count < 0 || count > e->B) { set_error("qg_step_slots: count must be within the slot pool"); return QG_ERR_INVALID; }
    StepArgs a{}; a.actions = actions_dev; a.src_slot = src_slot_dev; a.dst_slot = dst_slot_dev; a.skip_negative = 1;
    a.obs = obs_dev; a.obs_bits = obs_bits_dev; a.mask = mask_dev; a.reward = reward_dev; a.done = done_dev; a.success = success_dev;
    return launch_step(e, MODE_STEP, a, (cudaStream_t)stream, count);
}

int qg_copy_records(qg_engine* dst, const int32_t* dst_slot_dev, qg_engine* src, int64_t count, qg_stream stream) {
    if (!dst || !src) { set_error("null engine"); return QG_ERR_INVALID; }
    if (dst->L.kind != src->L.kind || dst->L.n != src->L.n || dst->L.W != src->L.W || dst->L.A != src->L.A || dst->device != src->device) {
        set_error("qg_copy_records: the engines must share env kind, qubits, gateset size and device"); return QG_ERR_INVALID;
    }
    if (count < 0 || count > src->B || (!dst_slot_dev && count > dst->B)) { set_error("qg_copy_records: count outside the batch"); return QG_ERR_INVALID; }
    if (count == 0) return QG_OK;
    CUDA_OK(cudaSetDevice(dst->device));
    k_copy_records<<<(unsigned)((count + 255) / 256), 256, 0, (cudaStream_t)stream>>>(dst->dc, dst_slot_dev, src->dc.rec, src->Bpad, dst->L.W, count);
    CUDA_OK(cudaGetLastError());
    if (dst->L.kind == QG_ENV_CLIFFORD && !src->all_symplectic) dst->all_symplectic = false;
    return QG_OK;
}

}  // extern "C"

namespace {

// qg_search_run and qg_search_run_twisted (tw: the twisted search's tables, a.act_perm = act_perm_dev; null: untwisted)
int search_run(qg_engine* e, qg_policy* pol, int32_t deterministic, int32_t max_decisions, uint32_t* obs_bits_dev, float* weights_dev,
               int32_t* decisions_dev, const SearchTwist* tw, const int32_t* act_perm_dev, qg_stream stream) {
    if (!e || !pol || !obs_bits_dev || !weights_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (pol->device != e->device) { set_error("qg_search_run: policy and engine live on different devices"); return QG_ERR_INVALID; }
    if (pol->d.obs_size != e->L.obs_size || pol->d.num_actions != e->L.A) { set_error("qg_search_run: the policy's observation size / action count do not match the env"); return QG_ERR_INVALID; }
    if (e->L.kind == QG_ENV_PERMUTATION && e->L.OW == 0) { set_error("packed observations need num_qubits <= 64 for Permutation"); return QG_ERR_UNSUPPORTED; }
    if (max_decisions < 0) { set_error("qg_search_run: negative decision budget"); return QG_ERR_INVALID; }
    CUDA_OK(cudaSetDevice(e->device));
    StepArgs a{}; a.weights = weights_dev; a.deterministic = deterministic;      // (no packed-observation output: the kernel keeps the bit stream on chip)
    if (tw) { a.act_perm = act_perm_dev; a.twist = tw->twist; }
    a.nsteps = 1; a.ring = 1; a.pdl_mode = 0; a.num_sms = e->num_sms;
    a.sm_warp_words = e->sm_warp_words; a.sm_scr = e->sm_scr; a.sm_obs = e->sm_obs; a.sm_cat = -1; a.sm_wts = -1; a.magic_obs = e->magic_obs; a.magic_A = e->magic_A;
    a.magic_vpe = e->magic_vpe; a.magic_a4 = e->magic_a4; a.symplectic = e->all_symplectic ? 1 : 0;
    a.magic_ow = magic40(((uint32_t)e->L.obs_size + 31u) / 32u);
    const size_t step_smem = (size_t)e->sm_warp_words * 4 + 16;
    {   // the bytes launch_search_fused will request (policy + step region + the CTA's action weights + static) against the device's limit
        size_t dyn = 0, stat = 0, limit = 0;
        switch (e->L.kind) {
            case QG_ENV_PERMUTATION: CUDA_OK((tw ? search_fused_smem<QG_ENV_PERMUTATION, true>(pol->d, step_smem, e->device, &dyn, &stat, &limit)
                                                        : search_fused_smem<QG_ENV_PERMUTATION, false>(pol->d, step_smem, e->device, &dyn, &stat, &limit))); break;
            case QG_ENV_LINEAR_FUNCTION: CUDA_OK((tw ? search_fused_smem<QG_ENV_LINEAR_FUNCTION, true>(pol->d, step_smem, e->device, &dyn, &stat, &limit)
                                                        : search_fused_smem<QG_ENV_LINEAR_FUNCTION, false>(pol->d, step_smem, e->device, &dyn, &stat, &limit))); break;
            case QG_ENV_CLIFFORD: CUDA_OK((tw ? search_fused_smem<QG_ENV_CLIFFORD, true>(pol->d, step_smem, e->device, &dyn, &stat, &limit)
                                                        : search_fused_smem<QG_ENV_CLIFFORD, false>(pol->d, step_smem, e->device, &dyn, &stat, &limit))); break;
            default: CUDA_OK((tw ? search_fused_smem<QG_ENV_PAULI_NETWORK, true>(pol->d, step_smem, e->device, &dyn, &stat, &limit)
                                                        : search_fused_smem<QG_ENV_PAULI_NETWORK, false>(pol->d, step_smem, e->device, &dyn, &stat, &limit))); break;
        }
        if (dyn + stat > limit) {
            set_error("qg_search_run: policy + env + action weights need " + std::to_string(dyn + stat) + " bytes of shared memory (" + std::to_string(dyn) +
                      " dynamic + " + std::to_string(stat) + " static), one block may have " + std::to_string(limit));
            return QG_ERR_UNSUPPORTED;
        }
    }
    if (e->B == 0 || max_decisions == 0) return QG_OK;          // (after every support check: a zero-decision call is the caller's probe)
    cudaStream_t st = (cudaStream_t)stream;
    // the policy's first-layer accumulators, one set per CTA of 8 rollouts (grown on first use; a launch in flight on another stream
    // with the same policy handle must not overlap a growing call: one host thread per handle, like the engine)
    const size_t ctas = (size_t)((e->B + kPolRows - 1) / kPolRows);
    if (ctas > pol->acc0_ctas) {
        if (pol->acc0) { CUDA_OK(cudaDeviceSynchronize()); CUDA_OK(cudaFree(pol->acc0)); pol->acc0 = nullptr; pol->acc0_ctas = 0; }
        CUDA_OK(cudaMalloc(&pol->acc0, ctas * kPolRows * (size_t)pol->d.width[0] * sizeof(long long)));
        pol->acc0_ctas = ctas;
    }
    switch (e->L.kind) {
        case QG_ENV_PERMUTATION: CUDA_OK(launch_search_fused<QG_ENV_PERMUTATION>(e->dc, a, pol->d, max_decisions, decisions_dev, step_smem, pol->acc0, obs_bits_dev, tw, st)); break;
        case QG_ENV_LINEAR_FUNCTION: CUDA_OK(launch_search_fused<QG_ENV_LINEAR_FUNCTION>(e->dc, a, pol->d, max_decisions, decisions_dev, step_smem, pol->acc0, obs_bits_dev, tw, st)); break;
        case QG_ENV_CLIFFORD: CUDA_OK(launch_search_fused<QG_ENV_CLIFFORD>(e->dc, a, pol->d, max_decisions, decisions_dev, step_smem, pol->acc0, obs_bits_dev, tw, st)); break;
        default: CUDA_OK(launch_search_fused<QG_ENV_PAULI_NETWORK>(e->dc, a, pol->d, max_decisions, decisions_dev, step_smem, pol->acc0, obs_bits_dev, tw, st)); break;
    }
    return QG_OK;
}

// Arguments of the twisted search's entry points: the tables are given, K >= 1; PauliNetwork (its symmetry is applied inside the env by
// add_perms) and a Permutation without packed observations (> 64 qubits) have no twisted search.
int check_twisted(const qg_engine* e, const uint8_t* qperm_inv_dev, const int32_t* act_perm_dev, bool need_act, int32_t num_twists, const int32_t* twist_dev) {
    if (!e || !qperm_inv_dev || (need_act && !act_perm_dev) || !twist_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (num_twists < 1) { set_error("the twisted search needs num_twists >= 1"); return QG_ERR_INVALID; }
    if (e->L.kind == QG_ENV_PAULI_NETWORK) { set_error("PauliNetwork has no twisted search: its qubit symmetry is applied inside the env (add_perms)"); return QG_ERR_UNSUPPORTED; }
    if (e->L.kind == QG_ENV_PERMUTATION && e->L.OW == 0) { set_error("packed observations need num_qubits <= 64 for Permutation"); return QG_ERR_UNSUPPORTED; }
    return QG_OK;
}

int launch_observe_twisted(qg_engine* e, uint32_t* obs_bits_dev, const uint8_t* qperm_inv_dev, int32_t num_twists, int32_t* twist_dev, cudaStream_t st) {
    if (e->B == 0) return QG_OK;
    const int ow = (e->L.obs_size + 31) / 32, d = e->L.kind == QG_ENV_CLIFFORD ? 2 * e->L.n : e->L.n;
    const int64_t total = e->B * (int64_t)ow;
    const unsigned grid = (unsigned)std::min<int64_t>((total + 255) / 256, 148 * 16);
    switch (e->L.kind) {
        case QG_ENV_PERMUTATION: k_observe_twisted<QG_ENV_PERMUTATION><<<grid, 256, 0, st>>>(e->dc, obs_bits_dev, ow, qperm_inv_dev, (uint32_t)num_twists, d, twist_dev); break;
        case QG_ENV_LINEAR_FUNCTION: k_observe_twisted<QG_ENV_LINEAR_FUNCTION><<<grid, 256, 0, st>>>(e->dc, obs_bits_dev, ow, qperm_inv_dev, (uint32_t)num_twists, d, twist_dev); break;
        default: k_observe_twisted<QG_ENV_CLIFFORD><<<grid, 256, 0, st>>>(e->dc, obs_bits_dev, ow, qperm_inv_dev, (uint32_t)num_twists, d, twist_dev); break;
    }
    CUDA_OK(cudaGetLastError());
    return QG_OK;
}

}  // namespace

extern "C" {

int qg_search_run(qg_engine* e, qg_policy* pol, int32_t deterministic, int32_t max_decisions, uint32_t* obs_bits_dev, float* weights_dev,
                  int32_t* decisions_dev, qg_stream stream) {
    return search_run(e, pol, deterministic, max_decisions, obs_bits_dev, weights_dev, decisions_dev, nullptr, nullptr, stream);
}

int qg_search_observe_twisted(qg_engine* e, uint32_t* obs_bits_dev, const uint8_t* qperm_inv_dev, int32_t num_twists, int32_t* twist_dev, qg_stream stream) {
    const int rc = check_twisted(e, qperm_inv_dev, nullptr, false, num_twists, twist_dev);
    if (rc != QG_OK) return rc;
    if (!obs_bits_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    CUDA_OK(cudaSetDevice(e->device));
    return launch_observe_twisted(e, obs_bits_dev, qperm_inv_dev, num_twists, twist_dev, (cudaStream_t)stream);
}

int qg_search_step_twisted(qg_engine* e, const float* weights_dev, int32_t deterministic, uint32_t* obs_bits_dev, const uint8_t* qperm_inv_dev,
                           const int32_t* act_perm_dev, int32_t num_twists, int32_t* twist_dev, int32_t* chosen_dev, int32_t* num_active_dev, qg_stream stream) {
    const int rc = check_twisted(e, qperm_inv_dev, act_perm_dev, true, num_twists, twist_dev);
    if (rc != QG_OK) return rc;
    if (!weights_dev || !obs_bits_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    if (num_active_dev) CUDA_OK(cudaMemsetAsync(num_active_dev, 0, 4, st));
    // the existing twisted step (the sampler reads weights[act_perm[twist[i]][a]], qg_collect_step_twisted_dev's path), then the next
    // observation in the frame drawn from the post-step tick
    StepArgs a{}; a.weights = weights_dev; a.deterministic = deterministic; a.chosen = chosen_dev; a.num_active = num_active_dev;
    a.act_perm = act_perm_dev; a.twist = twist_dev;
    const int src = launch_step(e, MODE_SEARCH, a, st);
    if (src != QG_OK) return src;
    return launch_observe_twisted(e, obs_bits_dev, qperm_inv_dev, num_twists, twist_dev, st);
}

int qg_search_run_twisted(qg_engine* e, qg_policy* pol, int32_t deterministic, int32_t max_decisions, uint32_t* obs_bits_dev, float* weights_dev,
                          int32_t* decisions_dev, const uint8_t* qperm_inv_dev, const int32_t* act_perm_dev, int32_t num_twists, int32_t* twist_dev,
                          qg_stream stream) {
    const int rc = check_twisted(e, qperm_inv_dev, act_perm_dev, true, num_twists, twist_dev);
    if (rc != QG_OK) return rc;
    const SearchTwist tw{qperm_inv_dev, twist_dev, (uint32_t)num_twists, e->L.kind == QG_ENV_CLIFFORD ? 2 * e->L.n : e->L.n};
    return search_run(e, pol, deterministic, max_decisions, obs_bits_dev, weights_dev, decisions_dev, &tw, act_perm_dev, stream);
}

int qg_search_best(qg_engine* e, int64_t* best_key_host, int64_t* best_env_host, qg_stream stream) {
    if (!e || !best_key_host || !best_env_host) { set_error("null argument"); return QG_ERR_INVALID; }
    CUDA_OK(cudaSetDevice(e->device));
    *best_key_host = 0; *best_env_host = -1;
    if (e->B == 0) return QG_OK;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_OK(cudaMemsetAsync(e->best, 0, 8, st));
    k_best<<<(unsigned)((e->B + 255) / 256), 256, 0, st>>>(e->dc, e->best);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaMemcpyAsync(e->h_best, e->best, 8, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    const unsigned long long key = *e->h_best;
    *best_key_host = (int64_t)key;
    *best_env_host = (0x3FFFFFFFll - (int64_t)(key & 0x3FFFFFFFull)) - e->dc.first_id;
    return QG_OK;
}

int qg_read_returns(qg_engine* e, float* returns_dev, qg_stream stream) {
    if (!e || !returns_dev) { set_error("null argument"); return QG_ERR_INVALID; }
    if (e->B == 0) return QG_OK;
    k_copy_f32<<<(unsigned)((e->B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(e->dc.ret, returns_dev, e->B);
    CUDA_OK(cudaGetLastError());
    return QG_OK;
}

}  // extern "C"
