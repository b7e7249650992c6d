/*
 * bgw.cu -- host side of libbgw.so: the C-ABI declared in include/bgw.h.
 *
 * Plain C entry points over raw device pointers; kernels (bgw_dev.cuh) are enqueued on the caller's stream.
 * The library owns the opaque handle and the compiled spec tables only; there is no CPU fallback and no
 * dependency on the test oracle.
 */
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#define BGW_SMALL_KERNELS
#include "bgw_dev.cuh"
#include "bgw_fast.cuh"
#include "bgw_maze.cuh"
#include "bgw_jit.h"

namespace {

thread_local char g_err[2048] = "";   /* room for an NVRTC diagnostic (bgw_set_program) */

int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CUDA_OK(call)                                                                                  \
    do {                                                                                               \
        cudaError_t err__ = (call);                                                                    \
        if (err__ != cudaSuccess) return fail(2, "%s failed: %s", #call, cudaGetErrorString(err__));   \
    } while (0)

struct DeviceGuard {
    int prev = -1;
    explicit DeviceGuard(int dev) { if (cudaGetDevice(&prev) == cudaSuccess && prev != dev) cudaSetDevice(dev); else prev = -1; }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

int align16(int x) { return (x + 15) & ~15; }
int pow2ceil(int x) { int p = 1; while (p < x) p <<= 1; return p; }

}  // namespace

static const void *observe_fast_fn(int R)
{
    switch (R) {
    case 1: return (const void *)bgw_observe_fast_kernel<1>;
    case 2: return (const void *)bgw_observe_fast_kernel<2>;
    case 3: return (const void *)bgw_observe_fast_kernel<3>;
    case 4: return (const void *)bgw_observe_fast_kernel<4>;
    case 5: return (const void *)bgw_observe_fast_kernel<5>;
    }
    return nullptr;
}

struct BgwEngine {
    int device = 0;
    GeneralStepFn step_fn = nullptr;   /* the bgw_step_kernel instantiation of this sim's program */
    bgwjit::Kernel jit;                /* bgw_specialize / bgw_set_program: the same body compiled at run time for this spec alone (launched instead of step_fn) */
    bgwjit::Kernel fast_jit;           /* bgw_specialize: the specialised kernel's body with this spec's shape as its compile-time shape */
    bool fast_jit_on = false;          /* launch fast_jit instead of fast_fn (off again when the caller binds its own layouts) */
    const void *fast_fn = nullptr;     /* the bgw_step_fast_kernel instantiation of this sim's shape */
    MazeParams maze{};            /* device-side MazePlacementState (bgw_maze.cuh); device pointers */
    bool maze_ok = false, maze_small = false;
    DevSpec ds{}, dsf{};          /* general kernels / fast kernel (own slot table size) */
    FastSpec fs{};
    int threads_fast = 0;
    bool pdl = true;              /* launch the fast step kernel with programmatic stream serialization */
    bool poisoned = false;        /* a step launch was rejected: the ticket counters are out of step */
    bool chain_ok = false;        /* consecutive launches of bgw_rollout_sampled may be chained per env (bgw_fast.cuh) */
    bool rollout_fused = true;    /* bgw_rollout_sampled runs a rollout of the specialised kernel in one launch (BGW_ROLLOUT_FUSED=0: one launch per step) */
    bool randomize_action_input = false;   /* AllStepManager(randomize_action_input): steps without a caller-given order use the keyed one */
    int16_t *order_buf = nullptr;     /* [E][L] device: the keyed order of the step (bgw_order_kernel) */
    bool use_device_layouts = true;   /* bgw_use_device_layouts(): the caller supplies its own layouts when false */
    uint32_t seq = 0;             /* sequence number of the last fast step launch */
    uint32_t *ticket_ring = nullptr;                /* [BGW_TICKET_RING] device: env ticket counters, one per launch in flight */
    std::vector<uint32_t> ticket_next;              /* value each counter will have when the launches that used it are done (a launch
                                                       draws exactly n_tickets + grid tickets) */
    int fast_shape = 0;           /* compile-time shape instantiation of the fast kernel: 0 run-time shapes, 1 FastStaticC5, 2 FastStaticC2 */
    const void *observe_fn = nullptr;   /* bgw_observe_fast_kernel<view range> when the sim qualifies, else the general observe kernel runs */
    int observe_grid = 0, observe_smem = 0;
    BgwDims dims{};
    BgwState st{};
    bool bound = false;
    int threads = 0;
    uint64_t launches = 0;
    std::vector<void *> allocs;
};

namespace {

template <typename T>
int upload(BgwEngine *h, const T *src, size_t n, const T **dst)
{
    void *p = nullptr;
    CUDA_OK(cudaMalloc(&p, std::max<size_t>(n, 1) * sizeof(T)));
    h->allocs.push_back(p);
    if (n) CUDA_OK(cudaMemcpy(p, src, n * sizeof(T), cudaMemcpyHostToDevice));
    *dst = (const T *)p;
    return 0;
}

/* host restatement of the LOS rays for bgw_los_mask (utils.py:45-115); same arithmetic as los_apply_dev:
 * (a/b)*t in IEEE float64 (this file is compiled with -ffp-contract=off), strict comparisons. */
void los_apply_host(uint8_t *mask, int R, int rd, int cd)
{
    const int n = 2 * R + 1;
    if (rd == 0 && cd == 0) return;
    if (cd != 0) {
        double du, dl;
        if (rd == 0) { du = dl = (cd > 0) ? (double)cd - 0.5 : (double)cd + 0.5; }
        else if ((rd > 0) == (cd > 0)) { du = (double)cd - 0.5; dl = (double)cd + 0.5; }
        else { du = (double)cd + 0.5; dl = (double)cd - 0.5; }
        volatile double ku = ((double)rd + 0.5) / du, kl = ((double)rd - 0.5) / dl;
        const int c0 = cd > 0 ? cd : -R, c1 = cd > 0 ? R : cd;
        const int r0 = rd > 0 ? rd : -R, r1 = rd < 0 ? rd : R;
        for (int c = c0; c <= c1; ++c) {
            volatile double up = ku * (double)c, lo = kl * (double)c;
            for (int r = r0; r <= r1; ++r) {
                if (c == cd && r == rd) continue;
                if (lo < (double)r && (double)r < up) mask[(r + R) * n + (c + R)] = 0;
            }
        }
    } else {
        const double d = rd > 0 ? (double)rd - 0.5 : (double)rd + 0.5;
        volatile double kl = ((double)cd - 0.5) / d, kr = ((double)cd + 0.5) / d;
        const int r0 = rd > 0 ? rd : -R, r1 = rd > 0 ? R : rd;
        for (int r = r0; r <= r1; ++r) {
            volatile double le = kl * (double)r, ri = kr * (double)r;
            for (int c = -R; c <= R; ++c) {
                if (c == cd && r == rd) continue;
                if (le < (double)c && (double)c < ri) mask[(r + R) * n + (c + R)] = 0;
            }
        }
    }
}

/* CTAs of one working thread walk the envs (the algorithm is a serial chain of keyed draws, about a millisecond per
 * maze; what matters is how many run at once).  The scratch sits in shared memory: as a local array its 15 KB would make
 * the driver reserve 4 GB (measured) for all the threads the device can hold, and in global memory every store-then-load
 * of the set table would go to L2 (measured 3x slower). */
template <typename Scratch>
__global__ void bgw_layout_kernel(const MazeParams p, const BgwState st, int E, int env_offset, const uint8_t *env_mask, int only_done)
{
    __shared__ Scratch w;
    if (threadIdx.x != 0) return;
    for (int e = blockIdx.x; e < E; e += gridDim.x) {              /* the grid is what fits the device at once */
        if (only_done ? !(st.env_flags[e] & BGW_ENV_ALL_DONE) : (env_mask && !env_mask[e])) continue;
        const int err = maze_layout(p, (uint32_t)(env_offset + e), st.episode[e] + 1u, w, st.layout + (size_t)e * p.A);
        if (err) st.error[e] = (uint32_t)err;
    }
}

int first_role(const BgwSpec *sp, int role)
{
    for (int a = 0; a < sp->n_agents; ++a) if (sp->role[a] == role) return a;
    return -1;
}

}  // namespace

extern "C" {

const char *bgw_last_error(void) { return g_err; }
int bgw_abi_version(void) { return BGW_ABI_VERSION; }

int bgw_create(const BgwSpec *sp, int device, bgw_handle *out)
{
    if (!sp || !out) return fail(1, "bgw_create: null argument");
    *out = nullptr;
    if (sp->abi_version != BGW_ABI_VERSION) return fail(1, "bgw_create: ABI version %d, library has %d", sp->abi_version, BGW_ABI_VERSION);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(2, "bgw_create: no CUDA device (this engine has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(1, "bgw_create: device %d out of range (%d devices)", device, ndev);
    const int A = sp->n_agents, H = sp->rows, W = sp->cols, HW = H * W;
    if (A < 1 || A > BGW_MAX_AGENTS) return fail(1, "bgw_create: n_agents %d not in 1..%d", A, BGW_MAX_AGENTS);
    if (H < 1 || W < 1 || HW > BGW_MAX_CELLS) return fail(1, "bgw_create: grid %dx%d not supported (at most %d cells)", H, W, BGW_MAX_CELLS);
    if (sp->n_envs < 1) return fail(1, "bgw_create: n_envs must be positive");

    BgwEngine *h = new BgwEngine();
    h->device = device;
    DeviceGuard guard(device);
    DevSpec &d = h->ds;
    auto bail = [&](int rc) { bgw_destroy(h); return rc; };

    d.H = H; d.W = W; d.HW = HW; d.A = A; d.E = sp->n_envs; d.env_offset = sp->env_offset;
    d.program = sp->program; d.move_actor = sp->move_actor; d.attack_actor = sp->attack_actor;
    d.observer = sp->observer; d.observe_self = sp->observe_self; d.done_mask = sp->done_mask;
    d.manager = sp->manager; d.ravel = sp->ravel_actions; d.no_overlap = sp->no_overlap_at_reset;
    d.stacked = sp->stacked_attacks; d.horizon = sp->horizon; d.auto_reset = sp->auto_reset;
    d.randomize_placement_order = sp->randomize_placement_order;
    d.seed = sp->seed;
    memcpy(d.reward, sp->reward, sizeof(d.reward));

    /* ---- per-entity tables ------------------------------------------------------------------ */
    std::vector<int16_t> learner_of(A, -1), agent_of;
    std::vector<uint16_t> blk, blk_static, var, init_cell(A, BGW_NONE);
    int max_enc = 0, rmax_obs = 0, rmax_att = 0, n_ammo = 0, att_payload = 1;
    for (int a = 0; a < A; ++a) if (sp->encoding[a] > max_enc) max_enc = std::min((int)sp->encoding[a], BGW_MAX_ENCODING);
    if (sp->attack_actor < BGW_ATTACK_NONE || sp->attack_actor > BGW_ATTACK_SELECTIVE) return bail(fail(1, "bgw_create: unknown attack actor %d", sp->attack_actor));
    for (int a = 0; a < A; ++a) {
        const int e = sp->encoding[a];
        if (e < 1 || e > BGW_MAX_ENCODING) return bail(fail(1, "bgw_create: entity %d has encoding %d, must be 1..%d", a, e, BGW_MAX_ENCODING));
        if (sp->target && (sp->target[a] < -1 || sp->target[a] >= A)) return bail(fail(1, "bgw_create: entity %d names target %d, must be -1 or an entity index below %d", a, (int)sp->target[a], A));
        if (sp->klass[a] & BGW_AG_LEARNER) { learner_of[a] = (int16_t)agent_of.size(); agent_of.push_back((int16_t)a); }
        if (sp->klass[a] & BGW_AG_BLOCKING) {
            /* static = never moves, never dies, fixed start cell (walls); dynamic blockers are listed first */
            const bool is_static = !(sp->klass[a] & (BGW_AG_MOVING | BGW_AG_HEALTH)) && sp->init_row[a] >= 0;
            (is_static ? blk_static : blk).push_back((uint16_t)a);
        }
        if (sp->init_row[a] < 0) var.push_back((uint16_t)a);
        else {
            if (sp->init_row[a] >= H || sp->init_col[a] < 0 || sp->init_col[a] >= W)
                return bail(fail(1, "bgw_create: entity %d initial position off the grid", a));
            init_cell[a] = (uint16_t)(sp->init_row[a] * W + sp->init_col[a]);
        }
        if ((sp->klass[a] & BGW_AG_LEARNER) && (sp->klass[a] & BGW_AG_OBSERVING)) {
            int R = sp->view_range[a];
            if (R < 0) return bail(fail(1, "bgw_create: negative view range"));
            rmax_obs = std::max(rmax_obs, R);
        }
        if (sp->klass[a] & BGW_AG_AMMO) {
            ++n_ammo;
            if (!sp->initial_ammo || sp->initial_ammo[a] < 0) return bail(fail(1, "bgw_create: entity %d is an AmmoAgent without a non-negative initial_ammo", a));
        }
        if ((sp->klass[a] & BGW_AG_ATTACKING) && sp->attack_actor != BGW_ATTACK_NONE) {
            const int R = sp->attack_range[a], n = 2 * R + 1, sim = sp->simultaneous_attacks[a];
            rmax_att = std::max(rmax_att, R);
            if (R < 0) return bail(fail(1, "bgw_create: negative attack range"));
            /* Binary / EncodingBased hand TeamBattleSim.step an ndarray: `not attacked_agents` raises for more than
             * one element (team_battle_example.py:41); the two selective actors return lists */
            if ((sp->program == BGW_PROG_TEAM_BATTLE || sp->program == BGW_PROG_REACH_TARGET) && sp->attack_actor == BGW_ATTACK_BINARY && sim > 1)
                return bail(fail(1, "bgw_create: TeamBattleSim.step with the BinaryAttackActor is only defined for simultaneous_attacks == 1 (team_battle_example.py:41)"));
            if (sim > BGW_MAX_SIMATT) return bail(fail(1, "bgw_create: simultaneous_attacks %d exceeds %d", sim, BGW_MAX_SIMATT));
            /* attack bytes of the action row and the most agents one attack can name */
            int w = 1, groups = 1;
            if (sp->attack_actor == BGW_ATTACK_ENCODING) { w = max_enc; groups = 0; for (int e = 1; e <= max_enc; ++e) groups += (int)((sp->attack_map[sp->encoding[a]] >> e) & 1); }
            else if (sp->attack_actor == BGW_ATTACK_RESTRICTED) { w = sim; groups = 1; }
            else if (sp->attack_actor == BGW_ATTACK_SELECTIVE) { w = n * n; groups = n * n; }
            if (n * n > 256 && sp->attack_actor >= BGW_ATTACK_RESTRICTED) return bail(fail(1, "bgw_create: attack range %d: a ravelled window cell must fit one byte (range <= 7)", R));
            if (groups * std::max(sim, 1) > BGW_MAX_VICTIMS)
                return bail(fail(1, "bgw_create: entity %d could attack %d agents in one step, the limit is %d", a, groups * sim, BGW_MAX_VICTIMS));
            att_payload = std::max(att_payload, w);
        }
    }
    const int L = (int)agent_of.size();
    if (L < 1) return bail(fail(1, "bgw_create: the simulation has no learning agent"));
    d.n_dyn_blk = (int)blk.size();
    blk.insert(blk.end(), blk_static.begin(), blk_static.end());
    d.L = L; d.max_enc = max_enc; d.n_blk = (int)blk.size(); d.n_var = (int)var.size();
    if (sp->attack_actor != BGW_ATTACK_NONE && d.n_blk > 0 && (2 * rmax_att + 1) * (2 * rmax_att + 1) > 32 * BGW_ATT_MASK_WORDS)
        return bail(fail(1, "bgw_create: attack_range %d with view-blocking entities exceeds the attacker's LOS mask (range <= 7)", rmax_att));
    if (sp->observer == BGW_OBS_STACKED && A > 127) return bail(fail(1, "bgw_create: stacked observer counts are int8 (at most 127 entities)"));
    if (sp->ravel_actions && sp->move_actor != BGW_MOVE_BOX) return bail(fail(1, "bgw_create: ravel_actions needs MoveActor"));

    d.a_nav = first_role(sp, BGW_ROLE_NAVIGATOR); d.a_target = first_role(sp, BGW_ROLE_TARGET);
    d.a_pacman = first_role(sp, BGW_ROLE_PACMAN); d.has_food = first_role(sp, BGW_ROLE_FOOD) >= 0;
    if (sp->program == BGW_PROG_MAZE && (d.a_nav < 0 || d.a_target < 0 || learner_of[d.a_nav] < 0))
        return bail(fail(1, "bgw_create: MazeNavigationSim needs a learning navigator and a target"));
    if (sp->program == BGW_PROG_MULTI_MAZE && d.a_target < 0) return bail(fail(1, "bgw_create: MultiMazeNavigationSim needs a target"));
    for (int k = 0; k < 10; ++k) d.a_script[k] = first_role(sp, BGW_ROLE_SCRIPTED_BADDIE + k);
    if ((sp->program == BGW_PROG_PACMAN || sp->program == BGW_PROG_PACMAN_SIMPLE) && (d.a_pacman < 0 || learner_of[d.a_pacman] < 0 || H <= 9 || W <= 20))
        return bail(fail(1, "bgw_create: PacmanSim needs a learning pacman and the (9,0)<->(9,20) tunnel (pacman.py:87-92)"));
    if (sp->program == BGW_PROG_REACH_TARGET && (d.a_target < 0 || learner_of[d.a_target] < 0))
        return bail(fail(1, "bgw_create: ReachTheTargetSim needs a learning target agent"));
    if (sp->program < BGW_PROG_TEAM_BATTLE || sp->program > BGW_PROG_USER) return bail(fail(1, "bgw_create: unknown program %d", sp->program));
    if (sp->program == BGW_PROG_USER && sp->manager == BGW_MANAGER_DYNAMIC_ORDER)
        return bail(fail(1, "bgw_create: a user step program cannot run under BGW_MANAGER_DYNAMIC_ORDER (its next_agent rule is built in)"));

    /* ---- observation geometry (same rule as the oracle's bgwo_dims) ------------------------------ */
    BgwDims &dm = h->dims;
    dm.n_envs = d.E; dm.n_agents = A; dm.n_learners = L;
    dm.obs_c = 1;
    if (sp->observer == BGW_OBS_ABSOLUTE) { dm.obs_h = H; dm.obs_w = W; }          /* observer.py:74 */
    else dm.obs_h = dm.obs_w = 2 * rmax_obs + 1;                                    /* observer.py:170,266 */
    if (sp->observer == BGW_OBS_STACKED) dm.obs_c = max_enc;                        /* observer.py:264 */
    const long long ncell = (long long)dm.obs_h * dm.obs_w * dm.obs_c;
    if (ncell > (1 << 24)) return bail(fail(1, "bgw_create: observation of %lld cells is too large", ncell));
    dm.ammo_offset = -1;
    long long obs_bytes = ncell;
    if (sp->ammo_observer) { dm.ammo_offset = (int)((ncell + 3) / 4 * 4); obs_bytes = dm.ammo_offset + 4; }   /* observer.py:376-413 */
    dm.position_offset = -1;
    if (sp->position_observer) { dm.position_offset = (int)((obs_bytes + 3) / 4 * 4); obs_bytes = dm.position_offset + 4; }   /* observer.py:337-373 */
    dm.obs_stride = (int)((obs_bytes + 15) / 16 * 16);
    dm.action_stride = (2 + att_payload + 3) / 4 * 4;
    d.act_words = dm.action_stride / 4; d.ammo_offset = dm.ammo_offset; d.n_ammo = n_ammo; d.position_offset = dm.position_offset;
    d.obs_cells = (int)ncell;
    d.obs_h = dm.obs_h; d.obs_w = dm.obs_w; d.obs_c = dm.obs_c; d.obs_stride = dm.obs_stride; d.nchunks = dm.obs_stride / 16;

    /* ---- reset template: place the fixed-position entities once (state.py:107-109,143-150) ------- */
    d.hw_words = (HW + 31) / 32;
    {
        std::vector<uint16_t> cell(A, BGW_NONE), next(A, BGW_NONE), head(HW, BGW_NONE), tail(HW, BGW_NONE);
        std::vector<uint8_t> flags(A, 0);
        std::vector<uint32_t> avail((size_t)(max_enc + 1) * d.hw_words, 0);
        for (int e = 0; e <= max_enc; ++e)
            for (int i = 0; i < HW; ++i) avail[(size_t)e * d.hw_words + (i >> 5)] |= 1u << (i & 31);
        int err = 0;
        for (int a = 0; a < A; ++a) {
            if (init_cell[a] == BGW_NONE) continue;
            const int c = init_cell[a];
            const uint64_t row = sp->overlap[sp->encoding[a]];
            for (uint16_t o = head[c]; o != BGW_NONE; o = next[o])
                if (!((row >> sp->encoding[o]) & 1)) { err = 1; break; }          /* assert at state.py:147-149 */
            if (tail[c] != BGW_NONE) next[tail[c]] = (uint16_t)a; else head[c] = (uint16_t)a;
            tail[c] = (uint16_t)a; cell[a] = (uint16_t)c; flags[a] = BGW_ST_IN_GRID;
            for (int e = 1; e <= max_enc; ++e)                                       /* state.py:126-141 */
                if (sp->no_overlap_at_reset || !((row >> e) & 1)) avail[(size_t)e * d.hw_words + (c >> 5)] &= ~(1u << (c & 31));
        }
        d.tpl_error = err;
        int rc;
        if ((rc = upload(h, cell.data(), A, &d.tpl_cell)) || (rc = upload(h, next.data(), A, &d.tpl_next)) ||
            (rc = upload(h, flags.data(), A, &d.tpl_flags)) || (rc = upload(h, avail.data(), avail.size(), &d.tpl_avail)))
            return bail(rc);
    }
    {
        int rc;
        std::vector<unsigned long long> ov(BGW_MAX_ENCODING + 1), am(BGW_MAX_ENCODING + 1);
        for (int i = 0; i <= BGW_MAX_ENCODING; ++i) { ov[i] = sp->overlap[i]; am[i] = sp->attack_map[i]; }
        if ((rc = upload(h, sp->encoding, A, &d.enc)) || (rc = upload(h, sp->klass, A, &d.klass)) ||
            (rc = upload(h, sp->role, A, &d.role)) || (rc = upload(h, sp->init_orient, A, &d.init_orient)) ||
            (rc = upload(h, sp->simultaneous_attacks, A, &d.simatt)) || (rc = upload(h, sp->view_range, A, &d.view_r)) ||
            (rc = upload(h, sp->move_range, A, &d.move_r)) || (rc = upload(h, sp->attack_range, A, &d.attack_r)) ||
            (rc = upload(h, sp->target, A, &d.target)) || (rc = upload(h, learner_of.data(), A, &d.learner_of)) ||
            (rc = upload(h, agent_of.data(), L, &d.agent_of)) || (rc = upload(h, sp->init_health, A, &d.init_health)) ||
            (rc = upload(h, sp->attack_strength, A, &d.strength)) || (rc = upload(h, sp->attack_accuracy, A, &d.accuracy)) ||
            (rc = upload(h, ov.data(), ov.size(), &d.overlap)) || (rc = upload(h, am.data(), am.size(), &d.attack_map)) ||
            (rc = upload(h, blk.data(), blk.size(), &d.blk_agents)) || (rc = upload(h, var.data(), var.size(), &d.var_agents)))
            return bail(rc);
        d.init_ammo = nullptr;
        if (n_ammo && (rc = upload(h, sp->initial_ammo, A, &d.init_ammo))) return bail(rc);
        /* MazePlacementState on the device (bgw_maze.cuh) */
        h->maze_ok = false;
        if (sp->layout_kind == BGW_LAYOUT_MAZE || sp->layout_kind == BGW_LAYOUT_TARGET_BARRIERS_FREE) {
            if (sp->layout_target < 0 || sp->layout_target >= A) return bail(fail(1, "bgw_create: the placement state needs a target agent"));
            MazeParams &m = h->maze;
            m.kind = sp->layout_kind;
            m.rows = H; m.cols = W; m.A = A; m.max_enc = max_enc; m.no_overlap = sp->no_overlap_at_reset; m.target = sp->layout_target;
            m.cluster_barriers = sp->cluster_barriers; m.scatter_free = sp->scatter_free_agents;
            m.seed = sp->seed; m.barrier_encodings = sp->barrier_encodings; m.free_encodings = sp->free_encodings;
            m.enc = d.enc; m.overlap = d.overlap;
            if ((rc = upload(h, sp->init_row, A, &m.init_row)) || (rc = upload(h, sp->init_col, A, &m.init_col))) return bail(rc);
            h->maze_ok = maze_supported(H, W, max_enc, sp->barrier_encodings, sp->free_encodings);
            h->maze_small = maze_fits<MazeScratchSmall>(H, W, max_enc, sp->barrier_encodings, sp->free_encodings);
        } else if (sp->layout_kind != BGW_LAYOUT_POSITION_STATE) return bail(fail(1, "bgw_create: unknown layout_kind %d", sp->layout_kind));
    }

    /* ---- launch geometry and the shared-memory carve-up ------------------------------------------ */
    /* general kernel: one CTA per env; small CTAs keep more envs resident (measured: maze 2.4x, pacman 1.9x faster
     * than with 128 / 256 threads) */
    int T = A <= 128 ? 32 : A <= 1024 ? 64 : 128;
    if (const char *t = getenv("BGW_THREADS")) { const int v = atoi(t); if (v >= 32 && v <= 256 && v % 32 == 0) T = v; }   /* __launch_bounds__(256, 3) */
    h->threads = T;
    d.parallel_actors = ((sp->program == BGW_PROG_TEAM_BATTLE || sp->program == BGW_PROG_REACH_TARGET || sp->program == BGW_PROG_TRAFFIC) && (sp->move_actor == BGW_MOVE_BOX || sp->move_actor == BGW_MOVE_CROSS));
    if (sp->program == BGW_PROG_TRAFFIC)         /* the +1 looks at the target's cell right after the own move: rank order if a target can move */
        for (int a = 0; a < A; ++a) if (sp->target[a] >= 0 && (sp->klass[sp->target[a]] & BGW_AG_MOVING)) d.parallel_actors = 0;
    if (const char *t = getenv("BGW_SERIAL_ACTORS")) if (atoi(t)) d.parallel_actors = 0;
    int slots = std::min(std::max(pow2ceil(HW), 32), 2048);
    if (const char *t = getenv("BGW_SLOTS")) { const int v = atoi(t); if (v >= 32 && v <= 65536 && (v & (v - 1)) == 0) slots = v; }
    d.slot_mask = slots - 1;
    {
        int reff = rmax_obs;
        if (sp->observer == BGW_OBS_ABSOLUTE) reff = std::min(reff, std::max(H, W) - 1);
        const long long nbits = (long long)(2 * reff + 1) * (2 * reff + 1);
        d.mask_words = d.n_blk ? (int)((nbits + 31) / 32) : 0;
        d.mask_batch = 0;
        if (d.n_blk) {
            if ((long long)d.mask_words * 4 > 96 * 1024) return bail(fail(1, "bgw_create: view range %d with view-blocking entities needs a %lld-bit LOS mask, too large for shared memory", reff, nbits));
            d.mask_batch = std::max(1, std::min(L, 32 * 1024 / (d.mask_words * 4)));
        }
        /* static-blocker table: one mask per viewer cell, when every observing learner has the same view range */
        d.static_mask = nullptr;
        bool uniform = true;
        int ru = -1;
        for (int a = 0; a < A; ++a)
            if ((sp->klass[a] & BGW_AG_LEARNER) && (sp->klass[a] & BGW_AG_OBSERVING)) {
                if (ru < 0) ru = sp->view_range[a]; else if (sp->view_range[a] != ru) uniform = false;
            }
        const size_t table_words = (size_t)HW * d.mask_words;
        if (!blk_static.empty() && uniform && ru >= 0 && table_words * 4 <= (64u << 20) && !getenv("BGW_NO_STATIC_MASK")) {
            const int R = reff, n = 2 * R + 1;
            std::vector<uint32_t> table(table_words, 0xFFFFFFFFu);
            std::vector<uint8_t> one((size_t)n * n);
            for (int c = 0; c < HW; ++c) {
                uint32_t *row = table.data() + (size_t)c * d.mask_words;
                const int r0 = c / W, c0 = c % W;
                for (uint16_t b : blk_static) {
                    const int rd = sp->init_row[b] - r0, cd = sp->init_col[b] - c0;
                    if (rd < -R || rd > R || cd < -R || cd > R) continue;
                    memset(one.data(), 1, one.size());
                    los_apply_host(one.data(), R, rd, cd);
                    for (int i = 0; i < n * n; ++i) if (!one[i]) row[i >> 5] &= ~(1u << (i & 31));
                }
            }
            int rc = upload(h, table.data(), table.size(), &d.static_mask);
            if (rc) return bail(rc);
        }
    }
    int off = 0;
    auto take = [&](int bytes) { const int o = off; off += align16(bytes); return o; };
    d.o_head = take(HW * 2 + 2);
    d.o_slot = take(slots * 4);
    d.o_cell = take(A * 2); d.o_next = take(A * 2);
    d.o_flags = take(A); d.o_enc = take(A); d.o_klass = take(A); d.o_tmp = take(A);
    d.o_racc = take(A * 8);
    d.o_act = take(L * dm.action_stride);
    d.o_ragent = take(L * 2); d.o_plist = take(L * 2); d.o_pstate = take(L);
    d.o_avail = take((max_enc + 1) * d.hw_words * 4);
    d.o_mask = take(d.mask_batch * d.mask_words * 4);
    d.o_ctr = take(CTR_COUNT * 4);
    d.o_csum = take(HW);
    /* ---- specialised team-battle kernel (bgw_fast.cuh) when the sim qualifies: own launch geometry and its
     *      own shared-memory carve-up ------------------------------------------------------------------- */
    {
        FastSpec &f = h->fs;
        const int P = std::max(rmax_obs, rmax_att);
        bool fast = sp->program == BGW_PROG_TEAM_BATTLE && sp->manager == BGW_MANAGER_ALL_STEP &&
                    (sp->move_actor == BGW_MOVE_BOX || sp->move_actor == BGW_MOVE_CROSS) && d.n_blk == 0 &&
                    sp->observer == BGW_OBS_POSITION_CENTERED && sp->attack_actor == BGW_ATTACK_BINARY && n_ammo == 0 &&
                    !sp->ammo_observer && !sp->position_observer &&
                    (2 * rmax_att + 1) * (2 * rmax_att + 1) <= 32;
        if (const char *t = getenv("BGW_GENERIC_KERNEL")) if (atoi(t)) fast = false;
        int TF = A <= 32 ? 32 : A <= 64 ? 64 : 96;      /* 3 warps: 10 envs per SM fit (shared memory and registers) */
        if (A == FastStaticC5::A && H == FastStaticC5::H && W == FastStaticC5::W) TF = FastStaticC5::T;   /* 2 warps: 11 envs per SM */
        if (const char *t = getenv("BGW_THREADS")) { const int v = atoi(t); if (v >= 32 && v <= 1024 && v % 32 == 0) TF = std::min(v, 128); }   /* __launch_bounds__(128, 7) */
        if (fast) {
            f.P = P;
            f.PL = P;
            f.PW = (W + 2 * P + 3) / 4 * 4;
            f.PH = H + 2 * P;
            f.magic_w = (uint32_t)(((1ull << 32) + (uint64_t)W - 1) / (uint64_t)W);
            int fslots = std::min(std::max(pow2ceil(HW), 32), 256);   /* two tables of half that: only contested movers and effective attackers reserve */
            if (const char *t = getenv("BGW_SLOTS")) { const int v = atoi(t); if (v >= 32 && v <= 65536 && (v & (v - 1)) == 0) fslots = v; }
            h->dsf = d;
            h->dsf.slot_mask = fslots - 1;
            const long long cbytes = (long long)f.PH * f.PW + 32;
            const FastLayout ly = fast_layout(A, L, HW, f.PH, f.PW, fslots, TF, max_enc, d.hw_words, L == A);
            fast_apply_layout(f, ly);
            const int fo = ly.smem_bytes;
            f.async_ok = (A % 16 == 0) ? 1 : (A % 8 == 0) ? 2 : 0;   /* cp.async in 16- or 8-byte chunks (rows start at multiples of A bytes) */
            f.simd_ok = (A % 4 == 0);
            f.uniform_view = -1;
            bool first = true, uniform = true;
            for (int a = 0; a < A; ++a)
                if ((sp->klass[a] & BGW_AG_LEARNER) && (sp->klass[a] & BGW_AG_OBSERVING)) {
                    if (first) { f.uniform_view = sp->view_range[a]; first = false; }
                    else if (sp->view_range[a] != f.uniform_view) uniform = false;
                }
            if (!uniform) f.uniform_view = -1;
            f.uniform_att = -1;
            {
                bool firsta = true, unia = true;
                for (int a = 0; a < A; ++a)
                    if (sp->klass[a] & BGW_AG_ATTACKING) {
                        if (firsta) { f.uniform_att = sp->attack_range[a]; firsta = false; }
                        else if (sp->attack_range[a] != f.uniform_att) unia = false;
                    }
                if (!unia) f.uniform_att = -1;
            }
            f.identity_learners = (L == A);
            {   /* mixed cells need two DIFFERENT encodings that may overlap; accuracy draws need an accuracy below 1 */
                unsigned long long present = 0;
                for (int a = 0; a < A; ++a) present |= 1ull << sp->encoding[a];
                f.can_mix = 0; f.acc_lt1 = 0;
                for (int e = 1; e <= max_enc; ++e)
                    if (((present >> e) & 1ull) && (sp->overlap[e] & present & ~(1ull << e))) f.can_mix = 1;
                for (int a = 0; a < A; ++a)
                    if ((sp->klass[a] & BGW_AG_ATTACKING) && sp->attack_accuracy[a] < 1.0) f.acc_lt1 = 1;
            }
            f.epoch0 = 0xFFFFEu;
            if (const char *t = getenv("BGW_EPOCH0")) { const long v = atol(t); if (v >= 1 && v <= 0xFFFFE) f.epoch0 = (uint32_t)v; }
            if (cbytes > 96 * 1024 || fo > 227 * 1024) fast = false;
        }
        f.enabled = fast;
        h->threads_fast = TF;
        if (fast) {
            h->fast_shape = fast_shape_matches<FastStaticC5>(h->dsf, f, TF) ? 1 : fast_shape_matches<FastStaticC2>(h->dsf, f, TF) ? 2 : 0;
            if (const char *t = getenv("BGW_DYNAMIC_SHAPES")) if (atoi(t)) h->fast_shape = 0;
            h->fast_fn = bgw_fast_step_fn(h->fast_shape, f.head_elem);   /* the instantiation step_impl launches for this handle */
        }
    }
    d.smem_bytes = off;
    if (off > 227 * 1024) return bail(fail(1, "bgw_create: one environment needs %d bytes of shared memory (limit 232448): grid or entity count too large", off));
    cudaError_t ce;
    /* a user step program has no stock instantiation: its kernel comes from bgw_set_program */
    h->step_fn = d.program == BGW_PROG_USER ? nullptr : bgw_general_step_fn(d.program, d.attack_actor);
    if (const char *t = getenv("BGW_ALL_IN_ONE_KERNEL")) if (atoi(t) && h->step_fn) h->step_fn = bgw_general_step_fn(-1, -1);
    if ((h->step_fn && (ce = cudaFuncSetAttribute(h->step_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, off)) != cudaSuccess) ||
        (h->fs.enabled && (ce = cudaFuncSetAttribute(h->fast_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, h->fs.smem_bytes)) != cudaSuccess) ||
        (ce = cudaFuncSetAttribute(bgw_reset_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, off)) != cudaSuccess ||
        (ce = cudaFuncSetAttribute(bgw_observe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, off)) != cudaSuccess)
        return bail(fail(2, "bgw_create: cudaFuncSetAttribute: %s", cudaGetErrorString(ce)));
    /* bgw_observe: the observer alone.  The sims of the specialised kernel whose cells never mix encodings and whose learners
     * share a view range get the gather-only kernel (bgw_fast.cuh); the rest run observe_learners of the general kernel. */
    if (h->fs.enabled && !h->fs.can_mix && sp->observe_self && h->fs.uniform_view >= 1 && h->fs.uniform_view <= 5 && !getenv("BGW_GENERIC_OBSERVE")) {
        const ObserveLayout lay = observe_layout(d.A, d.L, h->fs.PH, h->fs.PW);
        int per_sm = 0, sms = 0;
        h->observe_fn = observe_fast_fn(h->fs.uniform_view);
        h->observe_smem = lay.bytes;
        if ((ce = cudaFuncSetAttribute(h->observe_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, lay.bytes)) != cudaSuccess ||
            (ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, h->observe_fn, 128, (size_t)lay.bytes)) != cudaSuccess ||
            (ce = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device)) != cudaSuccess)
            return bail(fail(2, "bgw_create: observe kernel set-up: %s", cudaGetErrorString(ce)));
        h->observe_grid = std::max(1, std::min(d.E, per_sm * sms));
        if (const char *t = getenv("BGW_OBSERVE_GRID")) { const int v = atoi(t); if (v >= 1) h->observe_grid = std::min(d.E, v); }
    }
    if (getenv("BGW_VERBOSE")) {
        if (h->observe_fn) fprintf(stderr, "[bgw] observe kernel: gather-only, view %d\n", h->fs.uniform_view);
        else fprintf(stderr, "[bgw] observe kernel: general\n");
    }
    if (h->fs.enabled) {
        int per_sm = 0, sms = 0;
        /* the instantiation step_impl launches for this handle */
        ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, h->fast_fn, h->threads_fast, (size_t)h->fs.smem_bytes);
        if (ce != cudaSuccess ||
            (ce = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device)) != cudaSuccess)
            return bail(fail(2, "bgw_create: occupancy query: %s", cudaGetErrorString(ce)));
        h->fs.grid_ctas = std::max(1, std::min(d.E, per_sm * sms));
        if (getenv("BGW_PROF_FILE")) {
            void *pp = nullptr;
            if (cudaMalloc(&pp, (size_t)h->fs.grid_ctas * 8 * 16 * sizeof(long long)) == cudaSuccess) { h->allocs.push_back(pp); cudaMemset(pp, 0, (size_t)h->fs.grid_ctas * 8 * 16 * sizeof(long long)); h->fs.prof = (long long *)pp; }
        }
        if (getenv("BGW_VERBOSE")) fprintf(stderr, "[bgw] fast kernel: shape %s, T=%d smem=%d B/CTA, %d CTAs/SM x %d SMs, grid=%d, slots=%d\n", h->fast_shape == 1 ? "C5 (compile-time)" : h->fast_shape == 2 ? "C2 (compile-time)" : "run-time", h->threads_fast, h->fs.smem_bytes, per_sm, sms, h->fs.grid_ctas, h->dsf.slot_mask + 1);
        if (const char *t = getenv("BGW_PDL")) h->pdl = atoi(t) != 0;
        if (const char *t = getenv("BGW_GRID")) { const int v = atoi(t); if (v >= 1) h->fs.grid_ctas = std::min(d.E, v); }
        {   /* env tickets + per-env launch stamps (bgw_fast.cuh, "env tickets and chained launches") */
            void *pp = nullptr;
            const size_t nb = ((size_t)d.E + BGW_TICKET_RING) * sizeof(uint32_t);
            if ((ce = cudaMalloc(&pp, nb)) != cudaSuccess || (ce = cudaMemset(pp, 0, nb)) != cudaSuccess)
                return bail(fail(2, "bgw_create: env stamps: %s", cudaGetErrorString(ce)));
            h->allocs.push_back(pp);
            h->ticket_ring = (uint32_t *)pp;
            h->fs.env_seq = (uint32_t *)pp + BGW_TICKET_RING;
        }
        /* chained launches: nothing may run between two steps (no layout kernel) */
        h->chain_ok = h->pdl && !(h->maze_ok && sp->auto_reset);
        if (const char *t = getenv("BGW_CHAIN")) if (!atoi(t)) h->chain_ok = false;
        if (const char *t = getenv("BGW_ROLLOUT_FUSED")) h->rollout_fused = atoi(t) != 0;
        h->fs.wait_limit_ns = 10ull * 1000ull * 1000ull * 1000ull;
        if (const char *t = getenv("BGW_WAIT_LIMIT_MS")) { const long long v = atoll(t); if (v > 0) h->fs.wait_limit_ns = (unsigned long long)v * 1000000ull; }
    }
    if (sp->randomize_action_input) {
        if (sp->manager != BGW_MANAGER_ALL_STEP) return bail(fail(1, "bgw_create: randomize_action_input is an AllStepManager option (all_step_manager.py:24-35)"));
        void *pp = nullptr;
        if ((ce = cudaMalloc(&pp, (size_t)d.E * std::max(L, 1) * sizeof(int16_t))) != cudaSuccess)
            return bail(fail(2, "bgw_create: order buffer: %s", cudaGetErrorString(ce)));
        h->allocs.push_back(pp);
        h->order_buf = (int16_t *)pp;
        h->randomize_action_input = true;
    }
    dm.device_layouts = h->maze_ok ? 1 : 0;
    dm.threads_per_env = h->fs.enabled ? h->threads_fast : T; dm.envs_per_cta = 1; dm.smem_bytes = h->fs.enabled ? h->fs.smem_bytes : off;
    *out = h;
    return 0;
}

int bgw_destroy(bgw_handle h)
{
    if (!h) return 0;
    DeviceGuard guard(h->device);
    if (h->jit.module) bgwjit::driver().ModuleUnload(h->jit.module);
    if (h->fast_jit.module) bgwjit::driver().ModuleUnload(h->fast_jit.module);
    for (void *p : h->allocs) cudaFree(p);
    delete h;
    return 0;
}

int bgw_specialize(bgw_handle h, const char *cache_dir)
{
    if (!h) return fail(1, "bgw_specialize: null handle");
    if (h->jit.function || h->fast_jit.function) return 0;
    if (h->ds.program == BGW_PROG_USER) return 0;             /* bgw_set_program compiles the program's kernel for the spec */
    /* nothing to gain (or not applicable): one of the shipped compile-time shapes; caller-supplied layouts (the compile-time
     * shapes have no layout path in their reset); the debug phase clocks (sized for the stock grid) */
    if (h->fs.enabled && (h->fast_shape != 0 || (h->bound && h->st.layout) || h->fs.prof)) return 0;
    DeviceGuard guard(h->device);
    CUDA_OK(cudaFree(nullptr));                              /* the runtime's primary context is current for the driver calls */
    if (!cache_dir) cache_dir = getenv("BGW_JIT_CACHE");
    std::string msg;
    if (!h->fs.enabled) {
        if (const char *e = bgwjit::build(h->ds, h->ds.init_ammo != nullptr, h->threads, cache_dir, h->jit, msg))
            return fail(2, "bgw_specialize: %s", e);
        return 0;
    }
    /* launch bounds as the shipped shapes choose them: as many CTAs per SM as the shared memory allows, at no fewer than 72
     * registers per thread */
    const int by_smem = (228 * 1024) / (h->fs.smem_bytes + 1024), by_regs = 65536 / (h->threads_fast * 72);
    const int lb_n = std::max(1, std::min(32, std::min(by_smem, by_regs)));
    if (const char *e = bgwjit::build_fast(h->dsf, h->fs, h->threads_fast, lb_n, cache_dir, h->fast_jit, msg))
        return fail(2, "bgw_specialize: %s", e);
    int per_sm = 0, sms = 0;
    const int rc = bgwjit::driver().OccupancyMaxActiveBlocks(&per_sm, h->fast_jit.function, h->threads_fast, (size_t)h->fs.smem_bytes);
    if (rc || per_sm < 1) { bgwjit::driver().ModuleUnload(h->fast_jit.module); h->fast_jit = bgwjit::Kernel(); return fail(2, "bgw_specialize: occupancy query of the compiled kernel failed (%d)", rc); }
    CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device));
    h->fs.grid_ctas = std::max(1, std::min(h->ds.E, per_sm * sms));
    if (const char *t = getenv("BGW_GRID")) { const int v = atoi(t); if (v >= 1) h->fs.grid_ctas = std::min(h->ds.E, v); }
    h->fast_jit_on = true;
    if (getenv("BGW_VERBOSE")) fprintf(stderr, "[bgw] fast kernel compiled for this spec's shape: %d CTAs/SM, grid=%d\n", per_sm, h->fs.grid_ctas);
    return 0;
}

int bgw_set_program(bgw_handle h, const char *source, const char *cache_dir)
{
    if (!h || !source) return fail(1, "bgw_set_program: null argument");
    if (h->ds.program != BGW_PROG_USER) return fail(1, "bgw_set_program: the handle's spec runs built-in program %d, not BGW_PROG_USER", h->ds.program);
    if (h->jit.function) return fail(1, "bgw_set_program: the handle has a step program already");
    DeviceGuard guard(h->device);
    CUDA_OK(cudaFree(nullptr));                              /* the runtime's primary context is current for the driver calls */
    if (!cache_dir) cache_dir = getenv("BGW_JIT_CACHE");
    std::string msg;
    if (const char *e = bgwjit::build(h->ds, h->ds.init_ammo != nullptr, h->threads, cache_dir, h->jit, msg, source))
        return fail(2, "bgw_set_program: %s", e);
    return 0;
}

int bgw_dims(bgw_handle h, BgwDims *out)
{
    if (!h || !out) return fail(1, "bgw_dims: null argument");
    *out = h->dims;
    return 0;
}

int bgw_bind_state(bgw_handle h, const BgwState *state)
{
    if (!h || !state) return fail(1, "bgw_bind_state: null argument");
    if (!state->cell || !state->next || !state->flags || !state->health || !state->reward_acc || !state->episode ||
        !state->step || !state->env_flags || !state->turn || !state->error || !state->stats)
        return fail(1, "bgw_bind_state: every array except `layout` and `ammo` is required");
    if (h->ds.n_ammo && !state->ammo) return fail(1, "bgw_bind_state: the simulation has AmmoAgents: `ammo` is required");
    h->st = *state;
    h->bound = true;
    if (state->layout && h->fs.enabled && (h->fast_shape != 0 || h->fast_jit_on)) {
        h->fast_jit_on = false;
        /* the compile-time-shape instantiations of the specialised kernel have no layout path in their inlined reset (code
         * size is what the instruction cache sees): a handle that is given layouts runs the run-time-shape instantiation */
        DeviceGuard guard(h->device);
        h->fast_shape = 0;
        h->fast_fn = bgw_fast_step_fn(0, h->fs.head_elem);
        CUDA_OK(cudaFuncSetAttribute(h->fast_fn, cudaFuncAttributeMaxDynamicSharedMemorySize, h->fs.smem_bytes));
        int per_sm = 0, sms = 0;
        CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, h->fast_fn, h->threads_fast, (size_t)h->fs.smem_bytes));
        CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device));
        h->fs.grid_ctas = std::max(1, std::min(h->ds.E, per_sm * sms));
    }
    return 0;
}

int bgw_reset(bgw_handle h, const uint8_t *env_mask, int8_t *obs, void *stream)
{
    if (!h) return fail(1, "bgw_reset: null handle");
    if (!h->bound) return fail(1, "bgw_reset: call bgw_bind_state first");
    DeviceGuard guard(h->device);
    bgw_reset_kernel<<<h->ds.E, h->threads, h->ds.smem_bytes, (cudaStream_t)stream>>>(h->ds, h->st, env_mask, obs);
    CUDA_OK(cudaGetLastError());
    h->launches += 1;
    return 0;
}

int bgw_observe(bgw_handle h, const uint8_t *env_mask, int8_t *obs, void *stream)
{
    if (!h) return fail(1, "bgw_observe: null handle");
    if (!h->bound) return fail(1, "bgw_observe: call bgw_bind_state first");
    if (!obs) return fail(1, "bgw_observe: obs is null");
    DeviceGuard guard(h->device);
    if (h->observe_fn) {
        void *args[] = {(void *)&h->dsf, (void *)&h->fs, (void *)&h->st, (void *)&env_mask, (void *)&obs};
        CUDA_OK(cudaLaunchKernel(h->observe_fn, dim3(h->observe_grid), dim3(128), args, (size_t)h->observe_smem, (cudaStream_t)stream));
    } else {
        bgw_observe_kernel<<<h->ds.E, h->threads, h->ds.smem_bytes, (cudaStream_t)stream>>>(h->ds, h->st, env_mask, obs);
        CUDA_OK(cudaGetLastError());
    }
    h->launches += 1;
    return 0;
}

/* debug builds (BGW_PROFILE): write the phase clocks of the last launch(es) to BGW_PROF_FILE.  With BGW_PROF_LAZY only
 * bgw_rollout_sampled dumps, after its last launch, so the per-env chaining of the launches is not broken by a synchronisation. */
static void dump_prof(bgw_handle h, void *stream)
{
    const size_t n = (size_t)h->fs.grid_ctas * 8 * 16;
    std::vector<long long> host(n);
    cudaStreamSynchronize((cudaStream_t)stream);
    cudaMemcpy(host.data(), h->fs.prof, n * sizeof(long long), cudaMemcpyDeviceToHost);
    if (FILE *fp = fopen(getenv("BGW_PROF_FILE"), "wb")) { fwrite(host.data(), sizeof(long long), n, fp); fclose(fp); }
}

static int step_impl(bgw_handle h, const int8_t *actions, int8_t *sampled, const int16_t *order, int8_t *obs, float *reward,
                     uint8_t *done, uint8_t *all_done, void *stream, bool chained = false, int n_steps = 1)
{
    if (h->ds.program == BGW_PROG_USER && !h->jit.function)
        return fail(1, "bgw_step: the handle runs a user step program and none is installed yet (bgw_set_program)");
    DeviceGuard guard(h->device);
    if (h->randomize_action_input && !order) {
        /* all_step_manager.py:62-65: the actions are processed in shuffled order -- the keyed order of this step, written
         * by bgw_order_kernel (the step kernels skip the learners that are done already) */
        if (n_steps != 1) return fail(1, "bgw_step: randomize_action_input needs one launch per step");
        const int L = h->ds.L, P = pow2ceil(std::max(L, 2));
        bgw_order_kernel<<<h->ds.E, std::min(1024, std::max(32, P / 2)), (size_t)P * sizeof(unsigned long long), (cudaStream_t)stream>>>(h->ds, h->st, P, h->order_buf);
        CUDA_OK(cudaGetLastError());
        h->launches += 1;
        order = h->order_buf;
        chained = false;                                  /* another kernel sits between this step launch and the one before */
    }
    if (h->fs.enabled) {
        if (h->poisoned) return fail(2, "bgw_step: an earlier step launch failed; the handle cannot be used any more");
        {   /* a launch that failed asynchronously (e.g. the bounded stamp wait trapped) leaves a sticky error: find it
             * before enqueueing more work on top of it (free: no synchronisation) */
            const cudaError_t pe = cudaPeekAtLastError();
            if (pe != cudaSuccess) { h->poisoned = true; return fail(2, "bgw_step: an earlier launch failed on the device (%s); the handle cannot be used any more", cudaGetErrorString(pe)); }
        }
        cudaStreamCaptureStatus capture = cudaStreamCaptureStatusNone;
        CUDA_OK(cudaStreamIsCapturing((cudaStream_t)stream, &capture));
        if (capture != cudaStreamCaptureStatusNone && n_steps != 1) return fail(1, "bgw_step: a captured launch is one manager step");
        h->fs.seq = h->seq + 1u;                       /* sequence number of this launch's first manager step */
        h->seq += (uint32_t)n_steps;
        h->fs.n_tickets = (uint32_t)n_steps * (uint32_t)h->ds.E;
        if (capture != cudaStreamCaptureStatusNone) {
            /* the launch goes into a CUDA graph and will run any number of times with these parameters: no ticket
             * counter (its base would be stale at the second replay) -- CTA c takes envs c, c + grid, ... -- and no
             * per-env chaining (the stamps it leaves carry this sequence number, which only ever makes a later
             * chained launch wait less than a whole launch, never less than it must: the first launch of every
             * rollout stamps all envs itself) */
            h->fs.chain = 0; h->fs.ticket = nullptr; h->fs.ticket_base = 0;
        } else {
            h->fs.chain = (chained && h->chain_ok) ? 1 : 0;
            if (h->ticket_next.empty()) h->ticket_next.assign(BGW_TICKET_RING, 0u);
            const uint32_t slot = h->fs.seq % BGW_TICKET_RING;
            h->fs.ticket = h->ticket_ring + slot;
            h->fs.ticket_base = h->ticket_next[slot];
            h->ticket_next[slot] += h->fs.n_tickets + (uint32_t)h->fs.grid_ctas;   /* every CTA draws one ticket past the end */
        }
        h->poisoned = true;                            /* until the launch below has been accepted */
        /* Programmatic dependent launch: when the previous operation on the stream is another step launch, the
         * CTAs of this one become resident as that one's CTAs retire and run their env-independent set-up (spec
         * tables, clean dense arrays) while its last envs finish; they read and write nothing of the step state
         * before griddepcontrol.wait, which returns once the previous grid has completed and its writes are visible.
         * After any other stream operation the attribute changes nothing.  BGW_PDL=0 turns it off (A/B). */
        cudaLaunchAttribute pdl_attr[1];
        pdl_attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        pdl_attr[0].val.programmaticStreamSerializationAllowed = h->pdl ? 1 : 0;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)h->fs.grid_ctas); cfg.blockDim = dim3((unsigned)h->threads_fast);
        cfg.dynamicSmemBytes = (size_t)h->fs.smem_bytes; cfg.stream = (cudaStream_t)stream;
        cfg.attrs = pdl_attr; cfg.numAttrs = 1;
        const uint32_t *act_arg = (const uint32_t *)actions;
        uint32_t *smp_arg = (uint32_t *)sampled;
        void *args[] = {&h->dsf, &h->fs, &h->st, &act_arg, &smp_arg, &order, &obs, &reward, &done, &all_done};
        if (h->fast_jit_on) {                          /* bgw_specialize: this spec's own compile-time shape, same launch */
            CUlaunchAttribute ja[1];
            memset(ja, 0, sizeof(ja));
            ja[0].id = CU_LAUNCH_ATTRIBUTE_PROGRAMMATIC_STREAM_SERIALIZATION;
            ja[0].value.programmaticStreamSerializationAllowed = h->pdl ? 1 : 0;
            CUlaunchConfig jc;
            memset(&jc, 0, sizeof(jc));
            jc.gridDimX = (unsigned)h->fs.grid_ctas; jc.gridDimY = jc.gridDimZ = 1;
            jc.blockDimX = (unsigned)h->threads_fast; jc.blockDimY = jc.blockDimZ = 1;
            jc.sharedMemBytes = (unsigned)h->fs.smem_bytes; jc.hStream = (CUstream)stream; jc.attrs = ja; jc.numAttrs = 1;
            const int rc = bgwjit::driver().LaunchKernelEx(&jc, h->fast_jit.function, args, nullptr);
            if (rc) { const char *es = nullptr; bgwjit::driver().GetErrorString(rc, &es); return fail(2, "bgw_step: cuLaunchKernelEx of the specialised kernel: %s", es ? es : "?"); }
        } else
            CUDA_OK(cudaLaunchKernelExC(&cfg, h->fast_fn, args));
        h->poisoned = false;
    } else {
        if (sampled) {                                 /* general kernel: sample, then step (two launches) */
            const size_t n = (size_t)h->ds.E * h->ds.L;
            bgw_sample_actions_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->ds, h->st, (uint32_t *)sampled);
            CUDA_OK(cudaGetLastError());
            h->launches += 1;
            actions = sampled;
        }
        if (h->jit.function) {                         /* bgw_specialize: this spec's own compilation of the same body */
            const uint32_t *act_arg = (const uint32_t *)actions;
            void *args[] = {&h->ds, &h->st, &act_arg, &order, &obs, &reward, &done, &all_done};
            const int rc = bgwjit::driver().LaunchKernel(h->jit.function, (unsigned)h->ds.E, 1, 1, (unsigned)h->threads, 1, 1,
                                                         (unsigned)h->ds.smem_bytes, stream, args, nullptr);
            if (rc) { const char *es = nullptr; bgwjit::driver().GetErrorString(rc, &es); return fail(2, "bgw_step: cuLaunchKernel of the specialised kernel: %s", es ? es : "?"); }
        } else
            h->step_fn<<<h->ds.E, h->threads, h->ds.smem_bytes, (cudaStream_t)stream>>>(
                h->ds, h->st, (const uint32_t *)actions, order, obs, reward, done, all_done);
    }
    CUDA_OK(cudaGetLastError());
    h->launches += 1;
    if (h->fs.enabled && h->fs.prof && !getenv("BGW_PROF_LAZY")) dump_prof(h, stream);   /* debug only: the phase clocks of this launch */
    return 0;
}

int bgw_step(bgw_handle h, const int8_t *actions, const int16_t *order, int8_t *obs, float *reward, uint8_t *done,
             uint8_t *all_done, void *stream)
{
    if (!h) return fail(1, "bgw_step: null handle");
    if (!h->bound) return fail(1, "bgw_step: call bgw_bind_state first");
    if (!actions || !reward || !done || !all_done) return fail(1, "bgw_step: actions, reward, done and all_done are required");
    return step_impl(h, actions, nullptr, order, obs, reward, done, all_done, stream);
}

int bgw_step_sampled(bgw_handle h, int8_t *actions_out, const int16_t *order, int8_t *obs, float *reward, uint8_t *done,
                     uint8_t *all_done, void *stream)
{
    if (!h) return fail(1, "bgw_step_sampled: null handle");
    if (!h->bound) return fail(1, "bgw_step_sampled: call bgw_bind_state first");
    if (!actions_out || !reward || !done || !all_done) return fail(1, "bgw_step_sampled: actions_out, reward, done and all_done are required");
    return step_impl(h, nullptr, actions_out, order, obs, reward, done, all_done, stream);
}

int bgw_rollout_sampled(bgw_handle h, int n_steps, int8_t *actions_out, const int16_t *order, int8_t *obs, float *reward,
                        uint8_t *done, uint8_t *all_done, void *stream)
{
    if (!h) return fail(1, "bgw_rollout_sampled: null handle");
    if (!h->bound) return fail(1, "bgw_rollout_sampled: call bgw_bind_state first");
    if (n_steps < 0) return fail(1, "bgw_rollout_sampled: n_steps < 0");
    if (!actions_out || !reward || !done || !all_done) return fail(1, "bgw_rollout_sampled: actions_out, reward, done and all_done are required");
    const bool layouts_between = h->maze_ok && h->st.layout && h->ds.auto_reset && h->use_device_layouts;
    cudaStreamCaptureStatus capture = cudaStreamCaptureStatusNone;
    if (h->fs.enabled) {
        DeviceGuard guard(h->device);
        CUDA_OK(cudaStreamIsCapturing((cudaStream_t)stream, &capture));
        if (capture == cudaStreamCaptureStatusNone) {
            /* the stream's status (no wait): a rollout whose bounded stamp wait trapped must not be followed by another */
            const cudaError_t qe = cudaStreamQuery((cudaStream_t)stream);
            if (qe != cudaSuccess && qe != cudaErrorNotReady) { h->poisoned = true; return fail(2, "bgw_rollout_sampled: the stream reports %s; the handle cannot be used any more", cudaGetErrorString(qe)); }
        }
    }
    if (h->fs.enabled && h->rollout_fused && !layouts_between && !(h->randomize_action_input && !order) && capture == cudaStreamCaptureStatusNone) {
        /* the specialised kernel runs the whole rollout in ONE launch: its CTAs draw (step, env) tickets and an env's step
         * k + 1 starts as soon as its step k is stamped (bgw_fast.cuh); the per-CTA set-up is paid once per rollout */
        const int kmax = std::max(1, (int)(0x7FFFFFFFu / (uint32_t)h->ds.E) - 1);
        for (int i = 0; i < n_steps; i += kmax) {
            const int rc = step_impl(h, nullptr, actions_out, order, obs, reward, done, all_done, stream, i > 0, std::min(kmax, n_steps - i));
            if (rc) return rc;
        }
    } else {
        for (int i = 0; i < n_steps; ++i) {
            /* launches 2..n follow a step launch of this handle directly: they may be chained per env */
            const int rc = step_impl(h, nullptr, actions_out, order, obs, reward, done, all_done, stream, i > 0 && !layouts_between);
            if (rc) return rc;
            if (layouts_between) {                                 /* next episode's layouts of the envs that just finished */
                const int rl = bgw_generate_layouts(h, nullptr, 1, stream);
                if (rl) return rl;
            }
        }
    }
    if (h->fs.enabled && h->fs.prof && getenv("BGW_PROF_LAZY")) dump_prof(h, stream);
    return 0;
}

int bgw_sample_actions(bgw_handle h, int8_t *actions, void *stream)
{
    if (!h || !actions) return fail(1, "bgw_sample_actions: null argument");
    if (!h->bound) return fail(1, "bgw_sample_actions: call bgw_bind_state first");
    DeviceGuard guard(h->device);
    const size_t n = (size_t)h->ds.E * h->ds.L;
    bgw_sample_actions_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(h->ds, h->st, (uint32_t *)actions);
    CUDA_OK(cudaGetLastError());
    h->launches += 1;
    return 0;
}

int bgw_gather_valid(bgw_handle h, const int8_t *obs, const float *reward, const uint8_t *done, const uint8_t *all_done,
                     int32_t *count, int32_t *index, int8_t *obs_c, float *reward_c, uint8_t *done_c, void *stream)
{
    if (!h || !obs || !reward || !done || !all_done || !count || !index || !obs_c || !reward_c || !done_c)
        return fail(1, "bgw_gather_valid: null argument");
    DeviceGuard guard(h->device);
    CUDA_OK(cudaMemsetAsync(count, 0, sizeof(int32_t), (cudaStream_t)stream));
    const int L = h->ds.L;
    bgw_gather_kernel<<<h->ds.E, 128, 16 + align16(L * 2), (cudaStream_t)stream>>>(
        L, h->ds.obs_stride, obs, reward, done, all_done, count, index, obs_c, reward_c, done_c);
    CUDA_OK(cudaGetLastError());
    h->launches += 1;
    return 0;
}

int bgw_generate_layouts(bgw_handle h, const uint8_t *env_mask, int only_done, void *stream)
{
    if (!h) return fail(1, "bgw_generate_layouts: null handle");
    if (!h->maze_ok) return fail(1, "bgw_generate_layouts: this simulation has no device-side layout generator (BgwDims.device_layouts == 0)");
    if (!h->bound || !h->st.layout) return fail(1, "bgw_generate_layouts: bind a state with a `layout` array first");
    DeviceGuard guard(h->device);
    int sms = 148;
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
    if (h->maze_small)                                             /* 5.5 KB of shared memory: the 32-CTA limit of an SM binds */
        bgw_layout_kernel<MazeScratchSmall><<<std::min(h->ds.E, sms * 32), 32, 0, (cudaStream_t)stream>>>(h->maze, h->st, h->ds.E, h->ds.env_offset, env_mask, only_done);
    else                                                           /* 14.7 KB: 15 CTAs per SM */
        bgw_layout_kernel<MazeScratch><<<std::min(h->ds.E, sms * 15), 32, 0, (cudaStream_t)stream>>>(h->maze, h->st, h->ds.E, h->ds.env_offset, env_mask, only_done);
    CUDA_OK(cudaGetLastError());
    h->launches += 1;
    return 0;
}

int bgw_use_device_layouts(bgw_handle h, int on)
{
    if (!h) return fail(1, "bgw_use_device_layouts: null handle");
    if (on && !h->maze_ok) return fail(1, "bgw_use_device_layouts: this simulation has no device-side layout generator");
    h->use_device_layouts = on != 0;
    return 0;
}

int bgw_maze_layout_host(const BgwSpec *sp, uint32_t global_env, uint32_t episode, uint16_t *layout)
{
    if (!sp || !layout) return fail(1, "bgw_maze_layout_host: null argument");
    if (sp->layout_kind != BGW_LAYOUT_MAZE && sp->layout_kind != BGW_LAYOUT_TARGET_BARRIERS_FREE)
        return fail(1, "bgw_maze_layout_host: the spec has no MazePlacementState / TargetBarriersFreePlacementState");
    int max_enc = 0;
    for (int a = 0; a < sp->n_agents; ++a) max_enc = std::max(max_enc, (int)sp->encoding[a]);
    if (!maze_supported(sp->rows, sp->cols, max_enc, sp->barrier_encodings, sp->free_encodings))
        return fail(1, "bgw_maze_layout_host: grid or encoding count above the generator's limits");
    std::vector<unsigned long long> ov(BGW_MAX_ENCODING + 1);
    for (int i = 0; i <= BGW_MAX_ENCODING; ++i) ov[i] = sp->overlap[i];
    MazeParams m{};
    m.kind = sp->layout_kind;
    m.rows = sp->rows; m.cols = sp->cols; m.A = sp->n_agents; m.max_enc = max_enc; m.no_overlap = sp->no_overlap_at_reset;
    m.target = sp->layout_target; m.cluster_barriers = sp->cluster_barriers; m.scatter_free = sp->scatter_free_agents;
    m.seed = sp->seed; m.barrier_encodings = sp->barrier_encodings; m.free_encodings = sp->free_encodings;
    m.enc = sp->encoding; m.init_row = sp->init_row; m.init_col = sp->init_col; m.overlap = ov.data();
    std::vector<MazeScratch> w(1);
    const int err = maze_layout(m, global_env, episode, w[0], layout);
    return err ? fail(10 + err, "bgw_maze_layout_host: no cell available for an entity (state.py:598-603)") : 0;
}

int bgw_rng_draw(uint64_t seed, uint32_t env, uint32_t episode, uint32_t step, uint32_t site, uint32_t slot, uint32_t k,
                 uint32_t out[4])
{
    bgw_draw4(seed, env, episode, step, site, slot, k, out);
    return 0;
}

int bgw_los_mask(int range, int r_diff, int c_diff, uint8_t *out)
{
    if (range < 0 || !out) return fail(1, "bgw_los_mask: bad argument");
    const int n = 2 * range + 1;
    memset(out, 1, (size_t)n * n);
    if (r_diff < -range || r_diff > range || c_diff < -range || c_diff > range) return 0;   /* utils.py:49-50 */
    los_apply_host(out, range, r_diff, c_diff);
    return 0;
}

uint64_t bgw_launch_count(bgw_handle h) { return h ? h->launches : 0; }

}  /* extern "C" */
