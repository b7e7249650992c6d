/*
 * bgw.cu -- host side of libbgw.so: the C-ABI declared in include/bgw.h.
 *
 * Plain C entry points over raw device pointers; kernels (bgw_dev.cuh) are enqueued on the caller's stream.
 * The library owns the opaque handle and the compiled spec tables only; there is no CPU fallback and no
 * dependency on the test oracle.
 */
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
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

/* the integer value of the environment knob `name`, or `fallback` when it is unset or outside lo..hi */
long long env_int(const char *name, long long lo, long long hi, long long fallback)
{
    const char *t = getenv(name);
    if (!t) return fallback;
    const long long v = atoll(t);
    return v >= lo && v <= hi ? v : fallback;
}

/* persistent grid of the specialised kernel: the resident set (per_sm CTAs on each of sms SMs), at most one CTA per env;
 * BGW_GRID=n runs n CTAs instead (tests: many envs per CTA) */
int fast_grid_ctas(int E, int per_sm, int sms)
{
    if (const long long v = env_int("BGW_GRID", 1, INT_MAX, 0)) return std::min<long long>(E, v);
    return std::max(1, std::min(E, per_sm * sms));
}

/* S, the consecutive steps of one env a ticket of the specialised kernel runs (bgw_fast.cuh, "env tickets and chained
 * launches"), for a launch of K manager steps over E envs on `grid` resident CTAs.  Every step of a block after its first
 * skips the env's hand-over (stamp wait, staging, list rebuild, write-back, summary clear, stamp), so a longer block is
 * cheaper per step; but the launch ends with a tail of up to one block per CTA.  When the envs fit the resident CTAs each
 * env is a serial chain anyway and has no tail to lengthen: the longest block.  Otherwise the block stays within a sixth
 * of a CTA's share of the launch (K E / grid env-steps).  Measured on a B200 (profiles/r03_block_sweep.txt, S = 1..16):
 * five episodes (K = 1000, share 2516) and configs[1] (K = 400, share 1384) are fastest at 16; K = 20 after a warm-up
 * (share 50) at 8, and slower at 16. */
int fast_block_steps(int K, int E, int grid)
{
    const long long share = (long long)K * E / std::max(grid, 1);
    int S = 16;
    if (E > grid)
        while (S > 1 && S * 6LL > share) S >>= 1;
    return std::max(1, std::min(S, K));
}

/* one kernel a handle launches, and how */
struct KernelLaunch {
    const void *fn = nullptr;   /* a stock kernel, or the cudaKernel_t of one compiled at run time (bgw_jit.h) */
    int grid = 0, threads = 0, smem = 0;
    bool pdl = false;           /* programmatic dependent launch (launch()) */
};

/* Launch `k`.  With `pdl`: when the previous operation on the stream is another step launch, the CTAs of this one become
 * resident as that one's CTAs retire and run their env-independent set-up (spec tables, clean dense arrays) while its last
 * envs finish; they read and write nothing of the step state before griddepcontrol.wait, which returns once the previous grid
 * has completed and its writes are visible.  After any other stream operation the attribute changes nothing. */
int launch(const KernelLaunch &k, void **args, void *stream)
{
    cudaLaunchAttribute pdl[1];
    pdl[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    pdl[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)k.grid); cfg.blockDim = dim3((unsigned)k.threads);
    cfg.dynamicSmemBytes = (size_t)k.smem; cfg.stream = (cudaStream_t)stream;
    cfg.attrs = pdl; cfg.numAttrs = k.pdl ? 1 : 0;
    (void)cudaLaunchKernelExC(&cfg, k.fn, args);
    CUDA_OK(cudaGetLastError());   /* as after a chevron launch: the launch's error, else one an earlier call left; cleared */
    return 0;
}

}  // namespace

struct BgwEngine {
    int device = 0;
    int sms = 0;                  /* the device's SM count */
    KernelLaunch step;            /* bgw_step_kernel of this sim's program, or compiled for this spec (bgw_specialize, bgw_set_program) */
    KernelLaunch fast;            /* bgw_step_fast_kernel of this sim's shape, or compiled with this spec's shape (bgw_specialize) */
    KernelLaunch observe;         /* bgw_observe_fast_kernel<view range> when the sim qualifies, else the general observe kernel */
    KernelLaunch reset;
    KernelLaunch program_vars;    /* bgw_program_vars_kernel: the initial values of the program's variables, after the reset kernel */
    ProgVars pv{};                /* the step program's variables (bgw_set_program_vars); all 0 without */
    cudaLibrary_t jit = nullptr;  /* the library of the kernel bgw_specialize / bgw_set_program compiled (step.fn or fast.fn) */
    MazeParams maze{};            /* device-side MazePlacementState (bgw_maze.cuh); device pointers */
    bool maze_ok = false, maze_small = false;
    DevSpec ds{}, dsf{};          /* general kernels / fast kernel (own slot table size) */
    FastSpec fs{};
    bool poisoned = false;        /* a step launch was rejected: the ticket counters are out of step */
    bool chain_ok = false;        /* consecutive launches of bgw_rollout_sampled may be chained per env (bgw_fast.cuh) */
    bool randomize_action_input = false;   /* AllStepManager(randomize_action_input): steps without a caller-given order use the keyed one */
    int16_t *order_buf = nullptr;     /* [E][L] device: the keyed order of the step (bgw_order_kernel) */
    bool use_device_layouts = true;   /* bgw_use_device_layouts(): the caller supplies its own layouts when false */
    uint32_t seq = 0;             /* sequence number of the last fast step launch */
    uint32_t *ticket_ring = nullptr;                /* [BGW_TICKET_RING] device: env ticket counters, one per launch in flight */
    std::vector<uint32_t> ticket_next;              /* value each counter will have when the launches that used it are done (a launch
                                                       draws exactly n_tickets + grid tickets) */
    BgwDims dims{};
    BgwState st{};
    bool bound = false;
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

/* the range that every entity with all of `klass_bits` has in `range` (validated: not negative), or -1 when they differ or
 * there is none */
int uniform_range(const BgwSpec *sp, int klass_bits, const int16_t *range)
{
    int r = -1;
    for (int a = 0; a < sp->n_agents; ++a)
        if ((sp->klass[a] & klass_bits) == klass_bits) {
            if (r >= 0 && range[a] != r) return -1;
            r = range[a];
        }
    return r;
}

/* the placement generator's parameters (bgw_maze.cuh) except its four arrays */
MazeParams maze_params(const BgwSpec *sp, int max_enc)
{
    MazeParams m{};
    m.kind = sp->layout_kind;
    m.rows = sp->rows; m.cols = sp->cols; m.A = sp->n_agents; m.max_enc = max_enc; m.no_overlap = sp->no_overlap_at_reset;
    m.target = sp->layout_target; m.cluster_barriers = sp->cluster_barriers; m.scatter_free = sp->scatter_free_agents;
    m.seed = sp->seed; m.barrier_encodings = sp->barrier_encodings; m.free_encodings = sp->free_encodings;
    return m;
}

/* Let `fn` launch with `smem` bytes of dynamic shared memory.  The limit belongs to the kernel, not to a handle, and the stock
 * kernels are shared by every handle of the process: it is only ever raised, so that creating a handle with a smaller working
 * set does not make the launches of a larger one fail. */
cudaError_t allow_smem(const void *fn, int smem)
{
    cudaFuncAttributes fa;
    cudaError_t ce = cudaFuncGetAttributes(&fa, fn);
    if (ce == cudaSuccess && fa.maxDynamicSharedSizeBytes < smem) ce = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    return ce;
}

/* Make `fn` the team-battle kernel step_impl launches: its dynamic shared memory, and the persistent grid of what fits the
 * device (per_sm: CTAs per SM).  On a failure the handle keeps the kernel it had, and the error is cleared so that
 * step_impl's cudaPeekAtLastError does not take it for a failed launch. */
int use_fast_kernel(BgwEngine *h, const void *fn, int &per_sm)
{
    cudaError_t ce = allow_smem(fn, h->fast.smem);
    if (ce == cudaSuccess) ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, h->fast.threads, (size_t)h->fast.smem);
    if (ce != cudaSuccess || per_sm < 1) {
        cudaGetLastError();
        return fail(2, "team-battle kernel set-up: %s", ce != cudaSuccess ? cudaGetErrorString(ce) : "no CTA fits on an SM");
    }
    h->fast.fn = fn;
    h->fast.grid = h->fs.grid_ctas = fast_grid_ctas(h->ds.E, per_sm, h->sms);
    return 0;
}

/* ---- the steps of bgw_create: each returns 0 or fail()'s code ------------------------------------------------------------ */

/* what the steps hand on to each other */
struct Plan {
    std::vector<uint16_t> init_cell;    /* per entity: its fixed start cell, or BGW_NONE */
    std::vector<uint16_t> blk_static;   /* blockers that never move, never die and have a fixed start cell (walls) */
    int rmax_obs = 0, rmax_att = 0;     /* largest view range of an observing learner, attack range of an attacker */
    int att_payload = 1;                /* attack bytes of the action row */
    int threads = 0, slots = 0;         /* BGW_THREADS / BGW_SLOTS, 0 when unset or not allowed; each kernel clamps them */
    int fast_shape = 0;                 /* team-battle kernel instantiation: 0 run-time shapes, 1 FastStaticC5, 2 FastStaticC2 */
};

/* validate the spec, fill DevSpec's scalars and upload the per-entity tables */
int check_spec(BgwEngine *h, const BgwSpec *sp, Plan &p)
{
    DevSpec &d = h->ds;
    const int A = sp->n_agents, H = sp->rows, W = sp->cols, HW = H * W;
    d.H = H; d.W = W; d.HW = HW; d.A = A; d.E = sp->n_envs; d.env_offset = sp->env_offset;
    d.program = sp->program; d.move_actor = sp->move_actor; d.attack_actor = sp->attack_actor;
    d.observer = sp->observer; d.observe_self = sp->observe_self; d.done_mask = sp->done_mask;
    d.manager = sp->manager; d.ravel = sp->ravel_actions; d.no_overlap = sp->no_overlap_at_reset;
    d.stacked = sp->stacked_attacks; d.horizon = sp->horizon; d.auto_reset = sp->auto_reset;
    d.randomize_placement_order = sp->randomize_placement_order;
    d.seed = sp->seed;
    memcpy(d.reward, sp->reward, sizeof(d.reward));

    std::vector<int16_t> learner_of(A, -1), agent_of;
    std::vector<uint16_t> blk, var;
    p.init_cell.assign(A, BGW_NONE);
    int max_enc = 0, n_ammo = 0;
    for (int a = 0; a < A; ++a) if (sp->encoding[a] > max_enc) max_enc = std::min((int)sp->encoding[a], BGW_MAX_ENCODING);
    if (sp->attack_actor < BGW_ATTACK_NONE || sp->attack_actor > BGW_ATTACK_SELECTIVE) return fail(1, "bgw_create: unknown attack actor %d", sp->attack_actor);
    for (int a = 0; a < A; ++a) {
        const int e = sp->encoding[a];
        if (e < 1 || e > BGW_MAX_ENCODING) return fail(1, "bgw_create: entity %d has encoding %d, must be 1..%d", a, e, BGW_MAX_ENCODING);
        if (sp->target && (sp->target[a] < -1 || sp->target[a] >= A)) return fail(1, "bgw_create: entity %d names target %d, must be -1 or an entity index below %d", a, (int)sp->target[a], A);
        if (sp->klass[a] & BGW_AG_LEARNER) { learner_of[a] = (int16_t)agent_of.size(); agent_of.push_back((int16_t)a); }
        if (sp->klass[a] & BGW_AG_BLOCKING) {
            /* static = never moves, never dies, fixed start cell (walls); dynamic blockers are listed first */
            const bool is_static = !(sp->klass[a] & (BGW_AG_MOVING | BGW_AG_HEALTH)) && sp->init_row[a] >= 0;
            (is_static ? p.blk_static : blk).push_back((uint16_t)a);
        }
        if (sp->init_row[a] < 0) var.push_back((uint16_t)a);
        else {
            if (sp->init_row[a] >= H || sp->init_col[a] < 0 || sp->init_col[a] >= W)
                return fail(1, "bgw_create: entity %d initial position off the grid", a);
            p.init_cell[a] = (uint16_t)(sp->init_row[a] * W + sp->init_col[a]);
        }
        if ((sp->klass[a] & BGW_AG_LEARNER) && (sp->klass[a] & BGW_AG_OBSERVING)) {
            int R = sp->view_range[a];
            if (R < 0) return fail(1, "bgw_create: negative view range");
            p.rmax_obs = std::max(p.rmax_obs, R);
        }
        if (sp->klass[a] & BGW_AG_AMMO) {
            ++n_ammo;
            if (!sp->initial_ammo || sp->initial_ammo[a] < 0) return fail(1, "bgw_create: entity %d is an AmmoAgent without a non-negative initial_ammo", a);
        }
        if ((sp->klass[a] & BGW_AG_ATTACKING) && sp->attack_actor != BGW_ATTACK_NONE) {
            const int R = sp->attack_range[a], n = 2 * R + 1, sim = sp->simultaneous_attacks[a];
            p.rmax_att = std::max(p.rmax_att, R);
            if (R < 0) return fail(1, "bgw_create: negative attack range");
            /* Binary / EncodingBased hand TeamBattleSim.step an ndarray: `not attacked_agents` raises for more than
             * one element (team_battle_example.py:41); the two selective actors return lists */
            if ((sp->program == BGW_PROG_TEAM_BATTLE || sp->program == BGW_PROG_REACH_TARGET) && sp->attack_actor == BGW_ATTACK_BINARY && sim > 1)
                return fail(1, "bgw_create: TeamBattleSim.step with the BinaryAttackActor is only defined for simultaneous_attacks == 1 (team_battle_example.py:41)");
            if (sim > BGW_MAX_SIMATT) return fail(1, "bgw_create: simultaneous_attacks %d exceeds %d", sim, BGW_MAX_SIMATT);
            /* attack bytes of the action row and the most agents one attack can name */
            int w = 1, groups = 1;
            if (sp->attack_actor == BGW_ATTACK_ENCODING) { w = max_enc; groups = 0; for (int e = 1; e <= max_enc; ++e) groups += (int)((sp->attack_map[sp->encoding[a]] >> e) & 1); }
            else if (sp->attack_actor == BGW_ATTACK_RESTRICTED) { w = sim; groups = 1; }
            else if (sp->attack_actor == BGW_ATTACK_SELECTIVE) { w = n * n; groups = n * n; }
            if (n * n > 256 && sp->attack_actor >= BGW_ATTACK_RESTRICTED) return fail(1, "bgw_create: attack range %d: a ravelled window cell must fit one byte (range <= 7)", R);
            if (groups * std::max(sim, 1) > BGW_MAX_VICTIMS)
                return fail(1, "bgw_create: entity %d could attack %d agents in one step, the limit is %d", a, groups * sim, BGW_MAX_VICTIMS);
            p.att_payload = std::max(p.att_payload, w);
        }
    }
    const int L = (int)agent_of.size();
    if (L < 1) return fail(1, "bgw_create: the simulation has no learning agent");
    d.n_dyn_blk = (int)blk.size();
    blk.insert(blk.end(), p.blk_static.begin(), p.blk_static.end());
    d.L = L; d.max_enc = max_enc; d.n_blk = (int)blk.size(); d.n_var = (int)var.size(); d.n_ammo = n_ammo;
    if (sp->attack_actor != BGW_ATTACK_NONE && d.n_blk > 0 && (2 * p.rmax_att + 1) * (2 * p.rmax_att + 1) > 32 * BGW_ATT_MASK_WORDS)
        return fail(1, "bgw_create: attack_range %d with view-blocking entities exceeds the attacker's LOS mask (range <= 7)", p.rmax_att);
    if (sp->observer == BGW_OBS_STACKED && A > 127) return fail(1, "bgw_create: stacked observer counts are int8 (at most 127 entities)");
    if (sp->ravel_actions && sp->move_actor != BGW_MOVE_BOX) return fail(1, "bgw_create: ravel_actions needs MoveActor");

    d.a_nav = first_role(sp, BGW_ROLE_NAVIGATOR); d.a_target = first_role(sp, BGW_ROLE_TARGET);
    d.a_pacman = first_role(sp, BGW_ROLE_PACMAN); d.has_food = first_role(sp, BGW_ROLE_FOOD) >= 0;
    if (sp->program == BGW_PROG_MAZE && (d.a_nav < 0 || d.a_target < 0 || learner_of[d.a_nav] < 0))
        return fail(1, "bgw_create: MazeNavigationSim needs a learning navigator and a target");
    if (sp->program == BGW_PROG_MULTI_MAZE && d.a_target < 0) return fail(1, "bgw_create: MultiMazeNavigationSim needs a target");
    for (int k = 0; k < 10; ++k) d.a_script[k] = first_role(sp, BGW_ROLE_SCRIPTED_BADDIE + k);
    if ((sp->program == BGW_PROG_PACMAN || sp->program == BGW_PROG_PACMAN_SIMPLE) && (d.a_pacman < 0 || learner_of[d.a_pacman] < 0 || H <= 9 || W <= 20))
        return fail(1, "bgw_create: PacmanSim needs a learning pacman and the (9,0)<->(9,20) tunnel (pacman.py:87-92)");
    if (sp->program == BGW_PROG_REACH_TARGET && (d.a_target < 0 || learner_of[d.a_target] < 0))
        return fail(1, "bgw_create: ReachTheTargetSim needs a learning target agent");
    if (sp->program < BGW_PROG_TEAM_BATTLE || sp->program > BGW_PROG_USER) return fail(1, "bgw_create: unknown program %d", sp->program);

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
        return rc;
    return n_ammo ? upload(h, sp->initial_ammo, A, &d.init_ammo) : 0;
}

/* observation geometry (same rule as the oracle's bgwo_dims) and the action row */
int observation_geometry(BgwEngine *h, const BgwSpec *sp, const Plan &p)
{
    DevSpec &d = h->ds;
    BgwDims &dm = h->dims;
    dm.n_envs = d.E; dm.n_agents = d.A; dm.n_learners = d.L;
    dm.obs_c = 1;
    if (sp->observer == BGW_OBS_ABSOLUTE) { dm.obs_h = d.H; dm.obs_w = d.W; }       /* observer.py:74 */
    else dm.obs_h = dm.obs_w = 2 * p.rmax_obs + 1;                                  /* observer.py:170,266 */
    if (sp->observer == BGW_OBS_STACKED) dm.obs_c = d.max_enc;                      /* observer.py:264 */
    const long long ncell = (long long)dm.obs_h * dm.obs_w * dm.obs_c;
    if (ncell > (1 << 24)) return fail(1, "bgw_create: observation of %lld cells is too large", ncell);
    dm.ammo_offset = -1;
    long long obs_bytes = ncell;
    if (sp->ammo_observer) { dm.ammo_offset = (int)((ncell + 3) / 4 * 4); obs_bytes = dm.ammo_offset + 4; }   /* observer.py:376-413 */
    dm.position_offset = -1;
    if (sp->position_observer) { dm.position_offset = (int)((obs_bytes + 3) / 4 * 4); obs_bytes = dm.position_offset + 4; }   /* observer.py:337-373 */
    dm.obs_stride = (int)((obs_bytes + 15) / 16 * 16);
    dm.action_stride = (2 + p.att_payload + 3) / 4 * 4;
    d.act_words = dm.action_stride / 4; d.ammo_offset = dm.ammo_offset; d.position_offset = dm.position_offset;
    d.obs_cells = (int)ncell;
    d.obs_h = dm.obs_h; d.obs_w = dm.obs_w; d.obs_c = dm.obs_c; d.obs_stride = dm.obs_stride; d.nchunks = dm.obs_stride / 16;
    return 0;
}

/* the reset template: place the fixed-position entities once (state.py:107-109,143-150); the MazePlacementState on the device */
int reset_template(BgwEngine *h, const BgwSpec *sp, const Plan &p)
{
    DevSpec &d = h->ds;
    const int A = d.A, HW = d.HW, max_enc = d.max_enc;
    d.hw_words = (HW + 31) / 32;
    std::vector<uint16_t> cell(A, BGW_NONE), next(A, BGW_NONE), head(HW, BGW_NONE), tail(HW, BGW_NONE);
    std::vector<uint8_t> flags(A, 0);
    std::vector<uint32_t> avail((size_t)(max_enc + 1) * d.hw_words, 0);
    for (int e = 0; e <= max_enc; ++e)
        for (int i = 0; i < HW; ++i) avail[(size_t)e * d.hw_words + (i >> 5)] |= 1u << (i & 31);
    int err = 0;
    for (int a = 0; a < A; ++a) {
        if (p.init_cell[a] == BGW_NONE) continue;
        const int c = p.init_cell[a];
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
        return rc;
    if (sp->layout_kind == BGW_LAYOUT_MAZE || sp->layout_kind == BGW_LAYOUT_TARGET_BARRIERS_FREE) {
        if (sp->layout_target < 0 || sp->layout_target >= A) return fail(1, "bgw_create: the placement state needs a target agent");
        MazeParams &m = h->maze;
        m = maze_params(sp, max_enc);
        m.enc = d.enc; m.overlap = d.overlap;
        if ((rc = upload(h, sp->init_row, A, &m.init_row)) || (rc = upload(h, sp->init_col, A, &m.init_col))) return rc;
        h->maze_ok = maze_supported(d.H, d.W, max_enc, sp->barrier_encodings, sp->free_encodings);
        h->maze_small = maze_fits<MazeScratchSmall>(d.H, d.W, max_enc, sp->barrier_encodings, sp->free_encodings);
    } else if (sp->layout_kind != BGW_LAYOUT_POSITION_STATE) return fail(1, "bgw_create: unknown layout_kind %d", sp->layout_kind);
    return 0;
}

/* the general kernel's LOS mask batches, and the static-blocker table: one mask per viewer cell, when every observing learner
 * has the same view range */
int static_los_table(BgwEngine *h, const BgwSpec *sp, const Plan &p)
{
    DevSpec &d = h->ds;
    const int H = d.H, W = d.W, HW = d.HW;
    int reff = p.rmax_obs;
    if (sp->observer == BGW_OBS_ABSOLUTE) reff = std::min(reff, std::max(H, W) - 1);
    const long long nbits = (long long)(2 * reff + 1) * (2 * reff + 1);
    d.mask_words = d.n_blk ? (int)((nbits + 31) / 32) : 0;
    d.mask_batch = 0;
    if (d.n_blk) {
        if ((long long)d.mask_words * 4 > 96 * 1024) return fail(1, "bgw_create: view range %d with view-blocking entities needs a %lld-bit LOS mask, too large for shared memory", reff, nbits);
        d.mask_batch = std::max(1, std::min(d.L, 32 * 1024 / (d.mask_words * 4)));
    }
    const size_t table_words = (size_t)HW * d.mask_words;
    if (p.blk_static.empty() || uniform_range(sp, BGW_AG_LEARNER | BGW_AG_OBSERVING, sp->view_range) < 0 ||
        table_words * 4 > (64u << 20) || getenv("BGW_NO_STATIC_MASK"))
        return 0;
    const int R = reff, n = 2 * R + 1;
    std::vector<uint32_t> table(table_words, 0xFFFFFFFFu);
    std::vector<uint8_t> one((size_t)n * n);
    for (int c = 0; c < HW; ++c) {
        uint32_t *row = table.data() + (size_t)c * d.mask_words;
        const int r0 = c / W, c0 = c % W;
        for (uint16_t b : p.blk_static) {
            const int rd = sp->init_row[b] - r0, cd = sp->init_col[b] - c0;
            if (rd < -R || rd > R || cd < -R || cd > R) continue;
            memset(one.data(), 1, one.size());
            los_apply_host(one.data(), R, rd, cd);
            for (int i = 0; i < n * n; ++i) if (!one[i]) row[i >> 5] &= ~(1u << (i & 31));
        }
    }
    return upload(h, table.data(), table.size(), &d.static_mask);
}

/* the general kernels: launch geometry and the shared-memory carve-up */
int general_kernel(BgwEngine *h, const BgwSpec *sp, const Plan &p)
{
    DevSpec &d = h->ds;
    const int A = d.A, L = d.L, HW = d.HW;
    /* one CTA per env; small CTAs keep more envs resident (measured: maze 2.4x, pacman 1.9x faster than with 128 / 256 threads) */
    int T = A <= 128 ? 32 : A <= 1024 ? 64 : 128;
    if (p.threads && p.threads <= 256) T = p.threads;   /* __launch_bounds__(256, 3) */
    d.parallel_actors = ((sp->program == BGW_PROG_TEAM_BATTLE || sp->program == BGW_PROG_REACH_TARGET || sp->program == BGW_PROG_TRAFFIC) && (sp->move_actor == BGW_MOVE_BOX || sp->move_actor == BGW_MOVE_CROSS));
    if (sp->program == BGW_PROG_TRAFFIC)         /* the +1 looks at the target's cell right after the own move: rank order if a target can move */
        for (int a = 0; a < A; ++a) if (sp->target[a] >= 0 && (sp->klass[sp->target[a]] & BGW_AG_MOVING)) d.parallel_actors = 0;
    if (env_int("BGW_SERIAL_ACTORS", LLONG_MIN, LLONG_MAX, 0)) d.parallel_actors = 0;
    const int slots = p.slots ? p.slots : std::min(std::max(pow2ceil(HW), 32), 2048);
    d.slot_mask = slots - 1;
    int off = 0;
    auto take = [&](int bytes) { const int o = off; off += align16(bytes); return o; };
    d.o_head = take(HW * 2 + 2);
    d.o_slot = take(slots * 4);
    d.o_cell = take(A * 2); d.o_next = take(A * 2);
    d.o_flags = take(A); d.o_enc = take(A); d.o_klass = take(A); d.o_tmp = take(A);
    d.o_racc = take(A * 8);
    d.o_act = take(L * h->dims.action_stride);
    d.o_ragent = take(L * 2); d.o_plist = take(L * 2); d.o_pstate = take(L);
    d.o_avail = take((d.max_enc + 1) * d.hw_words * 4);
    d.o_mask = take(d.mask_batch * d.mask_words * 4);
    d.o_ctr = take(CTR_COUNT * 4);
    d.o_csum = take(HW);
    d.smem_bytes = off;
    if (off > 227 * 1024) return fail(1, "bgw_create: one environment needs %d bytes of shared memory (limit 232448): grid or entity count too large", off);
    /* a user step program has no stock instantiation: its kernel comes from bgw_set_program */
    h->step = {d.program == BGW_PROG_USER ? nullptr : bgw_general_step_fn(d.program, d.attack_actor), d.E, T, off, false};
    h->reset = {(const void *)bgw_reset_kernel, d.E, T, off, false};
    for (const KernelLaunch *k : {&h->step, &h->reset})
        if (k->fn) CUDA_OK(allow_smem(k->fn, k->smem));
    return 0;
}

/* the specialised team-battle kernel (bgw_fast.cuh) when the sim qualifies: its FastSpec, threads and shared-memory carve-up */
int team_battle_kernel(BgwEngine *h, const BgwSpec *sp, Plan &p)
{
    const DevSpec &d = h->ds;
    FastSpec &f = h->fs;
    const int A = d.A, L = d.L, H = d.H, W = d.W, HW = d.HW;
    const int P = std::max(p.rmax_obs, p.rmax_att);
    bool fast = sp->program == BGW_PROG_TEAM_BATTLE && sp->manager == BGW_MANAGER_ALL_STEP &&
                (sp->move_actor == BGW_MOVE_BOX || sp->move_actor == BGW_MOVE_CROSS) && d.n_blk == 0 &&
                sp->observer == BGW_OBS_POSITION_CENTERED && sp->attack_actor == BGW_ATTACK_BINARY && d.n_ammo == 0 &&
                !sp->ammo_observer && !sp->position_observer &&
                (2 * p.rmax_att + 1) * (2 * p.rmax_att + 1) <= 32;
    if (env_int("BGW_GENERIC_KERNEL", LLONG_MIN, LLONG_MAX, 0)) fast = false;
    int TF = A <= 32 ? 32 : A <= 64 ? 64 : 96;      /* 3 warps: 10 envs per SM fit (shared memory and registers) */
    if (A == FastStaticC5::A && H == FastStaticC5::H && W == FastStaticC5::W) TF = FastStaticC5::T;   /* 2 warps: 11 envs per SM */
    if (p.threads) TF = std::min(p.threads, 128);   /* __launch_bounds__(128, 7) */
    if (fast) {
        f.P = P;
        f.PL = P;
        f.PW = (W + 2 * P + 3) / 4 * 4;
        f.PH = H + 2 * P;
        f.magic_w = (uint32_t)(((1ull << 32) + (uint64_t)W - 1) / (uint64_t)W);
        /* two tables of half that: only contested movers and effective attackers reserve */
        const int fslots = p.slots ? p.slots : std::min(std::max(pow2ceil(HW), 32), 256);
        h->dsf = d;
        h->dsf.slot_mask = fslots - 1;
        const long long cbytes = (long long)f.PH * f.PW + 32;
        const FastLayout ly = fast_layout(A, L, HW, f.PH, f.PW, fslots, TF, d.max_enc, d.hw_words, L == A);
        fast_apply_layout(f, ly);
        const int fo = ly.smem_bytes;
        f.async_ok = (A % 16 == 0) ? 1 : (A % 8 == 0) ? 2 : 0;   /* cp.async in 16- or 8-byte chunks (rows start at multiples of A bytes) */
        f.simd_ok = (A % 4 == 0);
        f.uniform_view = uniform_range(sp, BGW_AG_LEARNER | BGW_AG_OBSERVING, sp->view_range);
        f.uniform_att = uniform_range(sp, BGW_AG_ATTACKING, sp->attack_range);
        f.identity_learners = (L == A);
        {   /* mixed cells need two DIFFERENT encodings that may overlap; accuracy draws need an accuracy below 1 */
            unsigned long long present = 0;
            for (int a = 0; a < A; ++a) present |= 1ull << sp->encoding[a];
            f.can_mix = 0; f.acc_lt1 = 0;
            for (int e = 1; e <= d.max_enc; ++e)
                if (((present >> e) & 1ull) && (sp->overlap[e] & present & ~(1ull << e))) f.can_mix = 1;
            for (int a = 0; a < A; ++a)
                if ((sp->klass[a] & BGW_AG_ATTACKING) && sp->attack_accuracy[a] < 1.0) f.acc_lt1 = 1;
        }
        f.epoch0 = (uint32_t)env_int("BGW_EPOCH0", 1, 0xFFFFE, 0xFFFFE);
        f.wait_limit_ns = (unsigned long long)env_int("BGW_WAIT_LIMIT_MS", 1, LLONG_MAX, 10 * 1000) * 1000000ull;
        if (cbytes > 96 * 1024 || fo > 227 * 1024) fast = false;
    }
    f.enabled = fast;
    h->fast = {nullptr, 0, TF, f.smem_bytes, true};   /* the kernel and its grid: use_fast_kernel */
    if (fast) {
        p.fast_shape = fast_shape_matches<FastStaticC5>(h->dsf, f, TF) ? 1 : fast_shape_matches<FastStaticC2>(h->dsf, f, TF) ? 2 : 0;
        if (env_int("BGW_DYNAMIC_SHAPES", LLONG_MIN, LLONG_MAX, 0)) p.fast_shape = 0;
        h->chain_ok = !(h->maze_ok && sp->auto_reset);   /* chained launches: nothing may run between two steps (no layout kernel) */
    }
    return 0;
}

/* bgw_observe: the observer alone.  The sims of the specialised kernel whose cells never mix encodings and whose learners
 * share a view range get the gather-only kernel (bgw_fast.cuh); the rest run observe_learners of the general kernel. */
int observe_kernel(BgwEngine *h, const BgwSpec *sp)
{
    const FastSpec &f = h->fs;
    const void *const by_view[] = {nullptr, (const void *)bgw_observe_fast_kernel<1>, (const void *)bgw_observe_fast_kernel<2>,
        (const void *)bgw_observe_fast_kernel<3>, (const void *)bgw_observe_fast_kernel<4>, (const void *)bgw_observe_fast_kernel<5>};
    const bool gather = f.enabled && !f.can_mix && sp->observe_self && f.uniform_view >= 1 && f.uniform_view <= 5 && !getenv("BGW_GENERIC_OBSERVE");
    if (gather) h->observe = {by_view[f.uniform_view], 0, 128, observe_layout(h->ds.A, h->ds.L, f.PH, f.PW).bytes, false};
    else h->observe = {(const void *)bgw_observe_kernel, h->ds.E, h->step.threads, h->step.smem, false};
    CUDA_OK(allow_smem(h->observe.fn, h->observe.smem));
    if (gather) {
        int per_sm = 0;
        CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, h->observe.fn, h->observe.threads, (size_t)h->observe.smem));
        h->observe.grid = std::max(1, std::min(h->ds.E, per_sm * h->sms));
    }
    if (getenv("BGW_VERBOSE")) {
        if (gather) fprintf(stderr, "[bgw] observe kernel: gather-only, view %d\n", f.uniform_view);
        else fprintf(stderr, "[bgw] observe kernel: general\n");
    }
    return 0;
}

/* the team-battle kernel's persistent grid, env stamps and ticket ring; the order buffer of randomize_action_input */
int step_buffers(BgwEngine *h, const BgwSpec *sp, const Plan &p)
{
    const int E = h->ds.E;
    cudaError_t ce;
    if (h->fs.enabled) {
        int per_sm = 0;
        if (const int rc = use_fast_kernel(h, bgw_fast_step_fn(p.fast_shape, h->fs.head_elem), per_sm)) return rc;
        if (getenv("BGW_PROF_FILE")) {
            void *pp = nullptr;
            if (cudaMalloc(&pp, (size_t)h->fast.grid * 8 * 16 * sizeof(long long)) == cudaSuccess) { h->allocs.push_back(pp); cudaMemset(pp, 0, (size_t)h->fast.grid * 8 * 16 * sizeof(long long)); h->fs.prof = (long long *)pp; }
        }
        if (getenv("BGW_VERBOSE")) fprintf(stderr, "[bgw] fast kernel: shape %s, T=%d smem=%d B/CTA, %d CTAs/SM x %d SMs, grid=%d, slots=%d\n", p.fast_shape == 1 ? "C5 (compile-time)" : p.fast_shape == 2 ? "C2 (compile-time)" : "run-time", h->fast.threads, h->fast.smem, per_sm, h->sms, h->fast.grid, h->dsf.slot_mask + 1);
        /* env tickets + per-env launch stamps (bgw_fast.cuh, "env tickets and chained launches") */
        void *pp = nullptr;
        const size_t nb = ((size_t)E + BGW_TICKET_RING) * sizeof(uint32_t);
        if ((ce = cudaMalloc(&pp, nb)) != cudaSuccess || (ce = cudaMemset(pp, 0, nb)) != cudaSuccess)
            return fail(2, "bgw_create: env stamps: %s", cudaGetErrorString(ce));
        h->allocs.push_back(pp);
        h->ticket_ring = (uint32_t *)pp;
        h->fs.env_seq = (uint32_t *)pp + BGW_TICKET_RING;
    }
    if (sp->randomize_action_input) {
        if (sp->manager != BGW_MANAGER_ALL_STEP) return fail(1, "bgw_create: randomize_action_input is an AllStepManager option (all_step_manager.py:24-35)");
        void *pp = nullptr;
        if ((ce = cudaMalloc(&pp, (size_t)E * std::max(h->ds.L, 1) * sizeof(int16_t))) != cudaSuccess)
            return fail(2, "bgw_create: order buffer: %s", cudaGetErrorString(ce));
        h->allocs.push_back(pp);
        h->order_buf = (int16_t *)pp;
        h->randomize_action_input = true;
    }
    return 0;
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
    Plan p;
    p.threads = (int)env_int("BGW_THREADS", 32, 1024, 0);
    if (p.threads % 32) p.threads = 0;
    p.slots = (int)env_int("BGW_SLOTS", 32, 65536, 0);
    if (p.slots & (p.slots - 1)) p.slots = 0;
    const cudaError_t ce = cudaDeviceGetAttribute(&h->sms, cudaDevAttrMultiProcessorCount, device);
    int rc = ce == cudaSuccess ? 0 : fail(2, "bgw_create: SM count: %s", cudaGetErrorString(ce));
    if (rc || (rc = check_spec(h, sp, p)) || (rc = observation_geometry(h, sp, p)) || (rc = reset_template(h, sp, p)) ||
        (rc = static_los_table(h, sp, p)) || (rc = general_kernel(h, sp, p)) || (rc = team_battle_kernel(h, sp, p)) ||
        (rc = observe_kernel(h, sp)) || (rc = step_buffers(h, sp, p))) {
        bgw_destroy(h);
        return rc;
    }
    const KernelLaunch &k = h->fs.enabled ? h->fast : h->step;
    h->dims.device_layouts = h->maze_ok ? 1 : 0;
    h->dims.threads_per_env = k.threads; h->dims.envs_per_cta = 1; h->dims.smem_bytes = k.smem;
    *out = h;
    return 0;
}

int bgw_destroy(bgw_handle h)
{
    if (!h) return 0;
    DeviceGuard guard(h->device);
    if (h->jit) cudaLibraryUnload(h->jit);
    for (void *p : h->allocs) cudaFree(p);
    delete h;
    return 0;
}

int bgw_specialize(bgw_handle h, const char *cache_dir)
{
    if (!h) return fail(1, "bgw_specialize: null handle");
    if (h->jit) return 0;
    if (h->ds.program == BGW_PROG_USER) return 0;             /* bgw_set_program compiles the program's kernel for the spec */
    /* nothing to gain (or not applicable): one of the shipped compile-time shapes; caller-supplied layouts (the compile-time
     * shapes have no layout path in their reset); the debug phase clocks (sized for the stock grid) */
    if (h->fs.enabled && (h->fast.fn != bgw_fast_step_fn(0, h->fs.head_elem) || (h->bound && h->st.layout) || h->fs.prof)) return 0;
    DeviceGuard guard(h->device);
    if (!cache_dir) cache_dir = getenv("BGW_JIT_CACHE");
    std::string msg;
    bgwjit::Kernel k;
    if (!h->fs.enabled) {
        if (const char *e = bgwjit::build(h->ds, h->ds.init_ammo != nullptr, h->step.threads, cache_dir, k, msg))
            return fail(2, "bgw_specialize: %s", e);
        h->jit = k.lib;
        h->step.fn = k.fn;
        return 0;
    }
    /* launch bounds as the shipped shapes choose them: as many CTAs per SM as the shared memory allows, at no fewer than 72
     * registers per thread */
    const int by_smem = (228 * 1024) / (h->fast.smem + 1024), by_regs = 65536 / (h->fast.threads * 72);
    const int lb_n = std::max(1, std::min(32, std::min(by_smem, by_regs)));
    if (const char *e = bgwjit::build_fast(h->dsf, h->fs, h->fast.threads, lb_n, cache_dir, k, msg))
        return fail(2, "bgw_specialize: %s", e);
    int per_sm = 0;
    if (const int rc = use_fast_kernel(h, k.fn, per_sm)) { cudaLibraryUnload(k.lib); return rc; }
    h->jit = k.lib;
    if (getenv("BGW_VERBOSE")) fprintf(stderr, "[bgw] fast kernel compiled for this spec's shape: %d CTAs/SM, grid=%d\n", per_sm, h->fast.grid);
    return 0;
}

int bgw_set_program(bgw_handle h, const char *source, const char *cache_dir)
{
    if (!h || !source) return fail(1, "bgw_set_program: null argument");
    if (h->ds.program != BGW_PROG_USER) return fail(1, "bgw_set_program: the handle's spec runs built-in program %d, not BGW_PROG_USER", h->ds.program);
    if (h->step.fn) return fail(1, "bgw_set_program: the handle has a step program already");
    DeviceGuard guard(h->device);
    if (!cache_dir) cache_dir = getenv("BGW_JIT_CACHE");
    std::string msg;
    bgwjit::Kernel k;
    if (const char *e = bgwjit::build(h->ds, h->ds.init_ammo != nullptr, h->step.threads, cache_dir, k, msg, source, h->pv))
        return fail(2, "bgw_set_program: %s", e);
    h->jit = k.lib;
    h->step.fn = k.fn;
    return 0;
}

int bgw_set_program_vars(bgw_handle h, int n_env_vars, int n_agent_vars, const double *init, double *vars)
{
    if (!h) return fail(1, "bgw_set_program_vars: null handle");
    if (h->ds.program != BGW_PROG_USER) return fail(1, "bgw_set_program_vars: the handle's spec runs built-in program %d, not BGW_PROG_USER", h->ds.program);
    if (h->step.fn) return fail(1, "bgw_set_program_vars: the handle has a step program already (the counts are compiled into its kernel: call this first)");
    if (n_env_vars < 0 || n_env_vars > BGW_MAX_ENV_VARS || n_agent_vars < 0 || n_agent_vars > BGW_MAX_AGENT_VARS)
        return fail(1, "bgw_set_program_vars: %d env slots and %d agent variables, the limits are %d and %d", n_env_vars, n_agent_vars,
                    BGW_MAX_ENV_VARS, BGW_MAX_AGENT_VARS);
    const int stride = n_env_vars + h->ds.A * n_agent_vars;
    if (stride && (!init || !vars)) return fail(1, "bgw_set_program_vars: init and vars are required for %d slots per env", stride);
    DeviceGuard guard(h->device);
    ProgVars pv{n_env_vars, n_agent_vars, stride, nullptr, stride ? vars : nullptr};
    if (stride)
        if (const int rc = upload(h, init, (size_t)stride, &pv.init)) return rc;
    h->pv = pv;
    const size_t n = (size_t)h->ds.E * stride;
    h->program_vars = {(const void *)bgw_program_vars_kernel, (int)((n + 255) / 256), 256, 0, false};
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
    /* the compile-time-shape instantiations of the specialised kernel have no layout path in their inlined reset (code size is
     * what the instruction cache sees): a handle that is given layouts runs the run-time-shape instantiation */
    if (state->layout && h->fs.enabled && h->fast.fn != bgw_fast_step_fn(0, h->fs.head_elem)) {
        DeviceGuard guard(h->device);
        int per_sm = 0;
        return use_fast_kernel(h, bgw_fast_step_fn(0, h->fs.head_elem), per_sm);
    }
    return 0;
}

int bgw_reset(bgw_handle h, const uint8_t *env_mask, int8_t *obs, void *stream)
{
    if (!h) return fail(1, "bgw_reset: null handle");
    if (!h->bound) return fail(1, "bgw_reset: call bgw_bind_state first");
    DeviceGuard guard(h->device);
    void *args[] = {&h->ds, &h->st, &env_mask, &obs};
    if (const int rc = launch(h->reset, args, stream)) return rc;
    h->launches += 1;
    if (h->pv.stride) {                                   /* the program's variables: the reset kernel is compiled without them */
        void *vargs[] = {&h->pv, &h->ds.E, &env_mask};
        if (const int rc = launch(h->program_vars, vargs, stream)) return rc;
        h->launches += 1;
    }
    return 0;
}

int bgw_observe(bgw_handle h, const uint8_t *env_mask, int8_t *obs, void *stream)
{
    if (!h) return fail(1, "bgw_observe: null handle");
    if (!h->bound) return fail(1, "bgw_observe: call bgw_bind_state first");
    if (!obs) return fail(1, "bgw_observe: obs is null");
    DeviceGuard guard(h->device);
    void *general[] = {&h->ds, &h->st, &env_mask, &obs}, *gather[] = {&h->dsf, &h->fs, &h->st, &env_mask, &obs};
    if (const int rc = launch(h->observe, h->observe.fn == (const void *)bgw_observe_kernel ? general : gather, stream)) return rc;
    h->launches += 1;
    return 0;
}

/* debug builds (BGW_PROFILE): write the phase clocks of the last launch(es) to BGW_PROF_FILE.  With BGW_PROF_LAZY only
 * bgw_rollout_sampled dumps, after its last launch, so the per-env chaining of the launches is not broken by a synchronisation. */
static void dump_prof(bgw_handle h, void *stream)
{
    const size_t n = (size_t)h->fast.grid * 8 * 16;
    std::vector<long long> host(n);
    cudaStreamSynchronize((cudaStream_t)stream);
    cudaMemcpy(host.data(), h->fs.prof, n * sizeof(long long), cudaMemcpyDeviceToHost);
    if (FILE *fp = fopen(getenv("BGW_PROF_FILE"), "wb")) { fwrite(host.data(), sizeof(long long), n, fp); fclose(fp); }
}

static int step_impl(bgw_handle h, const int8_t *actions, int8_t *sampled, const int16_t *order, int8_t *obs, float *reward,
                     uint8_t *done, uint8_t *all_done, void *stream, bool chained = false, int n_steps = 1)
{
    if (h->ds.program == BGW_PROG_USER && !h->step.fn)
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
        h->fs.n_steps = (uint32_t)n_steps;
        h->fs.block_steps = (uint32_t)fast_block_steps(n_steps, h->ds.E, h->fast.grid);
        h->fs.n_tickets = (uint32_t)((n_steps + h->fs.block_steps - 1) / h->fs.block_steps) * (uint32_t)h->ds.E;
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
            h->ticket_next[slot] += h->fs.n_tickets + (uint32_t)h->fast.grid;   /* every CTA draws one ticket past the end */
        }
        h->poisoned = true;                            /* until the launch below has been accepted */
        const uint32_t *act_arg = (const uint32_t *)actions;
        uint32_t *smp_arg = (uint32_t *)sampled;
        void *args[] = {&h->dsf, &h->fs, &h->st, &act_arg, &smp_arg, &order, &obs, &reward, &done, &all_done};
        if (const int rc = launch(h->fast, args, stream)) return rc;
        h->poisoned = false;
    } else {
        if (sampled) {                                 /* general kernel: sample, then step (two launches) */
            if (const int rc = bgw_sample_actions(h, sampled, stream)) return rc;
            actions = sampled;
        }
        const uint32_t *act_arg = (const uint32_t *)actions;
        /* the kernel of a step program takes its variables last; the other kernels have eight parameters and ignore it */
        void *args[] = {&h->ds, &h->st, &act_arg, &order, &obs, &reward, &done, &all_done, &h->pv};
        if (const int rc = launch(h->step, args, stream)) return rc;
    }
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
    if (h->fs.enabled && !layouts_between && !(h->randomize_action_input && !order) && capture == cudaStreamCaptureStatusNone) {
        /* the specialised kernel runs the whole rollout in ONE launch: its CTAs draw (block of steps, env) tickets and an env's step
         * k + 1 starts as soon as its step k is stamped (bgw_fast.cuh); the per-CTA set-up is paid once per rollout */
        const int kmax = std::max(1, (int)(0x7FFFFFFFu / (uint32_t)h->ds.E) - 1);
        for (int i = 0; i < n_steps; i += kmax) {
            const int rc = step_impl(h, nullptr, actions_out, order, obs, reward, done, all_done, stream, i > 0, std::min(kmax, n_steps - i));
            if (rc) return rc;
        }
    } else {
        for (int i = 0; i < n_steps; ++i) {
            /* unchained: layouts run between steps, step_impl unchains the keyed order and capture, the general kernel never chains */
            const int rc = step_impl(h, nullptr, actions_out, order, obs, reward, done, all_done, stream, false);
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
    if (h->maze_small)                                             /* 5.5 KB of shared memory: the 32-CTA limit of an SM binds */
        bgw_layout_kernel<MazeScratchSmall><<<std::min(h->ds.E, h->sms * 32), 32, 0, (cudaStream_t)stream>>>(h->maze, h->st, h->ds.E, h->ds.env_offset, env_mask, only_done);
    else                                                           /* 14.7 KB: 15 CTAs per SM */
        bgw_layout_kernel<MazeScratch><<<std::min(h->ds.E, h->sms * 15), 32, 0, (cudaStream_t)stream>>>(h->maze, h->st, h->ds.E, h->ds.env_offset, env_mask, only_done);
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
    MazeParams m = maze_params(sp, max_enc);
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
