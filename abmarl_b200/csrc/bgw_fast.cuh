/*
 * bgw_fast.cuh -- the specialised step kernel for the headline path: TeamBattleSim under AllStepManager with
 * MoveActor / CrossMoveActor, BinaryAttackActor, PositionCenteredEncodingObserver and no view-blocking entities
 * (BASELINE configs 2 and 5).  Same semantics and same results as the general kernel in bgw_dev.cuh (the
 * parity tests run both against the oracle); what changes is the amount of work per env:
 *
 *   - PERSISTENT CTAs: the grid is sized to the number of co-resident CTAs and each CTA loops over envs.  The
 *     dense per-cell arrays (occupant list heads, reservation slots, encoding summary) are initialised once
 *     per CTA and left clean by every env (each env removes exactly what it inserted), so an env costs
 *     O(live entities), not O(cells);
 *   - DOUBLE-BUFFERED STAGING: while env e is processed, the agent store of the CTA's next env (cell / next /
 *     flags / health rows and the action row) streams HBM -> shared memory with cp.async (LDGSTS, 16-byte
 *     chunks), so no phase waits on a dependent global load;
 *   - only RELEVANT entities are touched (anything still in the grid, active, or not yet reported done); dead,
 *     removed and reported entities never change again and are not stored back.  One warp compacts the relevant
 *     entities and the acting learners (order preserving) with byte-parallel tests on the flag words and a
 *     shuffle scan, so every later phase costs O(live agents);
 *   - next to the per-cell occupant lists the env keeps `cenc`, a padded int8 summary of the grid
 *     (border = -1 out of bounds, 0 empty, e = every occupant has encoding e, BGW_MIXED = mixed encodings).
 *     The attack pre-pass, the move legality test and the observation gather read it instead of walking lists;
 *   - only attackers that have a possible victim in their window enter the ordered reservation rounds, and they
 *     reserve only their own cell and the cells that hold possible victims; attackers without one are settled
 *     afterwards from the rank of whoever killed them (an attacker is charged for a failed attempt iff it
 *     was still alive at its turn, team_battle_example.py:37-42);
 *   - the observation window is gathered from `cenc` with aligned 32-bit loads + funnel shifts, one thread per
 *     learner, assembled into the packed (2R+1)^2 row in registers (compile-time view range) and written to HBM
 *     straight from the registers with 256-bit stores (one full 32-byte sector per lane).  Envs that hold
 *     a mixed cell (or observers that do not observe themselves, or other view ranges) take the per-cell path
 *     with the keyed np.random.choice over the occupant list.
 */
#pragma once
#include "bgw_dev.cuh"

#define BGW_MIXED (-128)
/* -DBGW_JITTER: a test build that perturbs the interleavings -- a pseudo-random sleep (0..2 us, from the clock, the thread and
 * the site) in front of every reservation, table look-up, touch mark, ticket draw and stamp access.  The parity tests, the
 * chained / fused rollout tests and the soak run under it (profiles/gpu_jitter_r02.sh): results must not change.  (Stands in
 * for compute-sanitizer racecheck, which is closed on this pool.) */
#ifdef BGW_JITTER
__device__ __forceinline__ void bgw_jitter(unsigned site)
{
    unsigned x = (unsigned)clock64() * 2654435761u + threadIdx.x * 40503u + site * 2246822519u;
    x ^= x >> 15; x *= 2246822519u; x ^= x >> 13;
    if (x & 3u) __nanosleep(x & 0x7FFu);
}
#define BGW_JITTER_POINT(site) bgw_jitter(site)
#else
#define BGW_JITTER_POINT(site) do { } while (0)
#endif
#ifdef BGW_PROFILE   /* debug build (BGW_PROFILE=1 python -m abmarl_b200.csrc.build): clock64 at the phase boundaries */
#define BGW_PROF_MARK(k) do { if (f.prof && tid == 0 && it_no < 8) f.prof[((size_t)blockIdx.x * 8 + it_no) * 16 + (k)] = clock64(); } while (0)
#else
#define BGW_PROF_MARK(k) do { } while (0)
#endif

struct FastSpec {
    int enabled;
    int P, PL, PW, PH;        /* padding (max range), left padding (16-byte aligned interior when W % 16 == 0),
                                 padded width (multiple of 16) / height */
    uint32_t magic_w;         /* ceil(2^32 / W): r = umulhi(cell, magic_w) for cell < 65536 */
    int uniform_view;         /* view range shared by every observing learner, or -1 */
    int uniform_att;          /* attack range shared by every attacking entity, or -1 */
    int identity_learners;    /* every entity is a learner: learner index == entity index */
    int can_mix;              /* some encoding may share a cell with a DIFFERENT encoding (overlapping): mixed cells can exist */
    int acc_lt1;              /* some attacker has attack_accuracy < 1: _basic_criteria draws */
    int grid_ctas;            /* persistent grid size */
    int async_ok;             /* stage the rows with cp.async: 1 = 16-byte chunks (A % 16 == 0), 2 = 8-byte chunks (A % 8 == 0), 0 = plain loads */
    int simd_ok;              /* A % 4 == 0: byte-parallel compaction */
    uint32_t epoch0;          /* first reservation epoch of a launch (0xFFFFE; tests start lower to exercise the wrap guard) */
    int b_cell, b_next, b_flags, buf_bytes;   /* layout of one staging buffer */
    /* shared-memory carve-up of the fast kernel.  `scratch` is a union: during the actor phases it holds
     * rflag | slot | rkmask | eff | pstate | killrank, and in
     * the (general) reset path racc | avail. */
    int o_enc, o_klass, o_tmp, o_act, o_head, o_cenc, o_rel, o_ragent, o_plist, o_ctr, o_wsum, o_buf, o_scratch;
    int s_rflag, s_slot, s_rkmask, s_eff, s_pstate, s_killrank, s_touch, scratch_bytes, smem_bytes;
    int touch_words;          /* words of ONE touch bitmap (power of two; two bitmaps at s_touch) */
    int r_racc, r_avail;      /* reset arena (over cenc | head | scratch, from o_cenc): u16 heads at 0, then racc, avail */
    int head_elem;            /* bytes per list head: 1 when A <= 256, else 2 */
    long long *prof;          /* debug (BGW_PROF_FILE): clock64 at phase boundaries, [cta][8 envs][16 marks] */
    /* env scheduling across launches (see "env tickets and chained launches" below) */
    uint32_t *env_seq;        /* [E] sequence number of the last fast step launch that finished this env */
    uint32_t *ticket;         /* this launch's env ticket counter: one of a ring of BGW_TICKET_RING, never reset; NULL: CTA c takes
                                 envs c, c + grid, ... (launches captured into a CUDA graph) */
    uint32_t ticket_base;     /* value of *ticket before this launch: every launch draws exactly n_tickets + grid tickets */
    uint32_t seq;             /* sequence number of the first manager step of this launch (1, 2, ... per handle) */
    uint32_t n_steps;         /* manager steps in this launch, K (bgw_rollout_sampled runs a whole rollout in ONE launch;
                                 bgw_step / bgw_step_sampled: 1) */
    uint32_t block_steps;     /* S: one ticket runs the consecutive steps [b S, min((b + 1) S, K)) of one env (fast_block_steps) */
    uint32_t n_tickets;       /* ceil(K / S) x E: ticket g is block g / E of env g % E */
    unsigned long long wait_limit_ns;   /* longest legitimate wait for an env's stamp (env_wait_stamp) */
    int chain;                /* 1: the previous operation on the stream is the fast step launch seq - 1 of the same
                                 rollout (bgw_rollout_sampled): wait per env on env_seq, not for the whole grid */
};

/* The shared-memory carve-up of the fast kernel: ONE definition used by bgw_create (run-time shapes) and by the
 * compile-time-shape instantiation (where every offset folds into an immediate). */
struct FastLayout {
    int b_cell, b_next, b_flags, buf_bytes;
    int o_enc, o_klass, o_tmp, o_act, o_head, o_cenc, o_rel, o_ragent, o_plist, o_ctr, o_wsum, o_buf, o_scratch;
    int s_rflag, s_slot, s_rkmask, s_eff, s_pstate, s_killrank, s_touch, touch_words, scratch_bytes, smem_bytes;
    int r_racc, r_avail, head_elem;
};

__host__ __device__ constexpr int fl_align16(int x) { return (x + 15) & ~15; }
/* words of one touch bitmap: a bit per cell up to 4096 cells (larger grids alias: only more agents go through the rounds) */
__host__ __device__ constexpr int fl_touch_words(int HW)
{
    int w = 4;
    while (w * 32 < HW && w < 128) w <<= 1;
    return w;
}

__host__ __device__ constexpr FastLayout fast_layout(int A, int L, int HW, int PH, int PW, int slots, int T, int max_enc,
                                                     int hw_words, int identity)
{
    FastLayout y{};
    int fo = 0;
    y.o_enc = fo; fo += fl_align16(A);
    y.o_klass = fo; fo += fl_align16(A);
    y.o_tmp = fo; fo += fl_align16(A);
    y.o_rel = fo; fo += fl_align16(A * 2);
    y.o_ragent = fo; fo += fl_align16(L * 2);
    y.o_plist = identity ? y.o_ragent : fo;               /* learner index == entity index: one list serves as both */
    if (!identity) fo += fl_align16(L * 2);
    y.o_act = fo; fo += fl_align16(L * 4);                /* this env's action words (not double-buffered: read or drawn by the attack pre-pass) */
    y.o_ctr = fo; fo += fl_align16(CTR_COUNT * 4);
    y.o_wsum = fo; fo += fl_align16(32 * 4);             /* [0..1] totals, [2..5] / [8..11] per-warp counts (T <= 128), [12..13] env tickets,
                                                              [16..31] float: this step's reward by RF_* flag combination */
    int bo = 0;
    y.b_cell = bo; bo += fl_align16(A * 2);
    y.b_next = bo; bo += fl_align16(A * 2);
    y.b_flags = bo; bo += fl_align16(A);
    y.buf_bytes = bo;
    y.o_buf = fo; fo += 2 * bo;
    /* scratch union, actor phases: rflag | rkmask | eff | pstate | killrank | slot */
    int so = 0;
    y.s_rkmask = so; so += fl_align16(L * 4);
    y.s_eff = so; so += fl_align16(L * 2);
    y.s_pstate = so; so += fl_align16(L);
    y.s_killrank = so; so += fl_align16(A * 2);
    y.s_slot = so; so += fl_align16(slots * 4);
    y.touch_words = fl_touch_words(HW);
    y.s_touch = so; so += 2 * y.touch_words * 4;          /* move phase: cells touched once / more than once */
    y.s_rflag = so; so += fl_align16(A);
    const int actor_bytes = so;
    /* cenc | head | scratch are contiguous: the general reset path uses all three as one arena: u16 heads | racc | avail */
    const int cenc_bytes = fl_align16(PH * PW + 32);      /* + slack: the word gather reads past a row end */
    y.head_elem = A <= 256 ? 1 : 2;
    const int head_bytes = fl_align16(HW * y.head_elem + 2);
    y.r_racc = fl_align16(HW * 2 + 2);
    y.r_avail = y.r_racc + fl_align16(A * 8);
    const int reset_bytes = y.r_avail + fl_align16((max_enc + 1) * hw_words * 4);
    int sb = actor_bytes;
    if (reset_bytes - cenc_bytes - head_bytes > sb) sb = reset_bytes - cenc_bytes - head_bytes;
    y.scratch_bytes = sb;
    y.o_cenc = fo; fo += cenc_bytes;
    y.o_head = fo; fo += head_bytes;
    y.o_scratch = fo; fo += sb;
    y.smem_bytes = fo;
    return y;
}

__host__ __device__ inline void fast_apply_layout(FastSpec &f, const FastLayout &y)
{
    f.b_cell = y.b_cell; f.b_next = y.b_next; f.b_flags = y.b_flags; f.buf_bytes = y.buf_bytes;
    f.o_enc = y.o_enc; f.o_klass = y.o_klass; f.o_tmp = y.o_tmp; f.o_act = y.o_act; f.o_head = y.o_head;
    f.o_cenc = y.o_cenc; f.o_rel = y.o_rel; f.o_ragent = y.o_ragent; f.o_plist = y.o_plist; f.o_ctr = y.o_ctr;
    f.o_wsum = y.o_wsum; f.o_buf = y.o_buf; f.o_scratch = y.o_scratch;
    f.s_rflag = y.s_rflag; f.s_slot = y.s_slot; f.s_rkmask = y.s_rkmask; f.s_eff = y.s_eff; f.s_pstate = y.s_pstate;
    f.s_killrank = y.s_killrank; f.s_touch = y.s_touch; f.touch_words = y.touch_words; f.scratch_bytes = y.scratch_bytes; f.smem_bytes = y.smem_bytes;
    f.r_racc = y.r_racc; f.r_avail = y.r_avail; f.head_elem = y.head_elem;
}

/* what happened to an entity this step, in the order the reference adds the rewards (team_battle_example.py:38-59):
 * its own attack (failed attempt or kill, at its turn), its death (at the killer's turn), its failed move */
enum { RF_ATTACK_FAIL = 1, RF_KILL = 2, RF_DIED = 4, RF_MOVE_FAIL = 8 };

struct FastEnv {
    void *head;               /* [HW] first occupant of a cell, uint8_t when A <= 256 else uint16_t; an entry is
                                 meaningful only while the summary says the cell is occupied, so the array is
                                 never cleared */
    uint8_t *rflag;           /* [A] RF_* bits of this step (replaces float64 accumulators: the sum is formed once, in order) */
    int8_t *cenc;
    uint16_t *killrank, *eff, *rel;
    uint32_t *rkmask, *act;
    uint32_t *touch;          /* [2][touch_words]: cells named by one pending move / by more than one (move phase) */
    int *wsum;
};

__device__ __forceinline__ void cell_rc(const DevSpec &s, const FastSpec &f, int cell, int &r, int &c)
{
    r = (int)__umulhi((uint32_t)cell, f.magic_w);
    c = cell - r * s.W;
}

__device__ __forceinline__ int pad_index(const DevSpec &s, const FastSpec &f, int cell)
{
    int r, c;
    cell_rc(s, f, cell, r, c);
    return (r + f.P) * f.PW + (c + f.PL);
}

/* ---- occupant lists of the fast kernel: `next` threads the entities of a cell in arrival order (as everywhere),
 * the first occupant is head[cell], valid iff cenc says the cell is occupied ------------------------------------ */
template <typename HT>
__device__ __forceinline__ unsigned fl_first(const FastEnv &fe, int cell, int pidx)
{
    return fe.cenc[pidx] != 0 ? (unsigned)((const HT *)fe.head)[cell] : BGW_NONE16;
}

/* summary of the list that starts at `first` */
__device__ __forceinline__ int8_t fl_summary(const Env &ev, unsigned first, bool can_mix)
{
    if (first == BGW_NONE16) return 0;
    const int8_t e = ev.enc[first];
    if (can_mix)
        for (unsigned o = ev.next[first]; o != BGW_NONE16; o = ev.next[o]) if (ev.enc[o] != e) return (int8_t)BGW_MIXED;
    return e;
}

/* Grid.remove grid.py:131-140 for an entity that is in the grid; returns the first occupant that remains */
template <typename HT>
__device__ __forceinline__ unsigned fl_unlink(Env &ev, FastEnv &fe, int a)
{
    const int cell = ev.cell[a];
    unsigned first = ((const HT *)fe.head)[cell];
    if (first == (unsigned)a) {
        first = ev.next[a];
        if (first != BGW_NONE16) ((HT *)fe.head)[cell] = (HT)first;
    } else {
        unsigned p = first;
        while (ev.next[p] != (unsigned)a) p = ev.next[p];
        ev.next[p] = ev.next[a];
    }
    ev.next[a] = BGW_NONE16;
    ev.flags[a] &= ~BGW_ST_IN_GRID;
    return first;
}

/* dict insert of Grid.place grid.py:124-126 (append at the tail) */
template <typename HT>
__device__ __forceinline__ void fl_append(Env &ev, FastEnv &fe, int a, int cell, bool occupied)
{
    ev.next[a] = BGW_NONE16;
    if (!occupied) ((HT *)fe.head)[cell] = (HT)a;
    else {
        unsigned p = ((const HT *)fe.head)[cell];
        for (unsigned q = ev.next[p]; q != BGW_NONE16; q = ev.next[p]) p = q;
        ev.next[p] = (uint16_t)a;
    }
    ev.cell[a] = (uint16_t)cell;
    ev.flags[a] |= BGW_ST_IN_GRID;
}

__device__ __forceinline__ void cp_async16(void *smem_dst, const void *gmem_src)
{
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async8(void *smem_dst, const void *gmem_src)
{
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;\n" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory"); }

/* ---- env tickets and chained launches -----------------------------------------------------------------------
 * A CTA takes blockIdx.x as its first env and every further env from a ticket counter (arrival order), so CTAs
 * that drew cheap envs take more of them and a launch has no fixed 2-or-3-envs-per-CTA tail.  Every env a launch
 * finishes is stamped with the launch's sequence number (release).  Inside bgw_rollout_sampled, where the library
 * itself enqueues consecutive step launches with nothing in between, launch k+1 is a programmatic dependent launch
 * that does NOT wait for launch k as a whole: its CTAs become resident as k's CTAs retire and start an env as
 * soon as THAT env carries the stamp k (acquire) -- envs never interact, so this is the only dependency.
 * Launch k+1 is not scheduled before every CTA of k has started (griddepcontrol.launch_dependents), so a waiting
 * CTA only ever waits for envs that started or finished CTAs of the launch before own: the chain cannot deadlock.
 * Any number of launches can be in flight (a CTA of k that drew an expensive env -- one that resets -- is still
 * running while k+1, k+2, ... pass by, each leaving one CTA waiting for that env), at most one per resident CTA:
 * each launch has its own ticket counter in a ring of BGW_TICKET_RING > resident CTAs.  A launch draws exactly
 * n_tickets + grid tickets (one terminal ticket per CTA), so the counters are never reset: the host passes the value a
 * counter has before the launch.
 * Inside a launch a ticket is a BLOCK of S consecutive manager steps of one env (fast_block_steps): between two steps of
 * the block the env stays on its CTA with its rows, summary grid and occupant lists in shared memory, and only the
 * block's first step waits for a stamp (the one the env's previous block -- a smaller ticket, or the launch before --
 * leaves at its last step).  A CTA still blocks only for the env of its current ticket, whose awaited block has a smaller
 * ticket number than every ticket its own holder has not finished: the argument above holds for blocks as for steps. */
#define BGW_TICKET_RING 2048
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_u32(uint32_t *p, uint32_t v)
{
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
/* has env e been stamped with sequence number `need` (or a later one)? */
__device__ __forceinline__ bool env_stamped(const FastSpec &f, int e, uint32_t need)
{
    BGW_JITTER_POINT(6);
    return (int32_t)(ld_acquire_u32(f.env_seq + e) - need) >= 0;
}
/* wait until it has.  A legitimate wait ends within one env (tens of microseconds, milliseconds when envs reset).  The bound is
 * wall time on the device (%globaltimer, looked at every 1024 polls), not a poll count: under a debugger, compute-sanitizer or a
 * time-sliced GPU a poll can take arbitrarily long.  When FastSpec.wait_limit_ns (default 10 s, BGW_WAIT_LIMIT_MS) has passed,
 * something is broken: fail the launch instead of hanging the device (the host then finds the handle poisoned). */
__device__ __forceinline__ unsigned long long global_timer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
__device__ __forceinline__ void env_wait_stamp(const FastSpec &f, int e, uint32_t need)
{
    unsigned spins = 0;
    unsigned long long t0 = 0;
    while (!env_stamped(f, e, need)) {
        __nanosleep(64);
        if ((++spins & 1023u) == 0) {
            const unsigned long long now = global_timer_ns();
            if (t0 == 0) t0 = now;
            else if (now - t0 > f.wait_limit_ns) __trap();
        }
    }
}
#define BGW_TSLOT 12          /* wsum[12], wsum[13]: the env after this one / the one after that */
#define BGW_EFSLOT 14         /* wsum[14]: the env flags this step leaves, for the env's next step in the same block */

/* stream env e's rows into one staging buffer */
__device__ __forceinline__ void fast_issue_env(const DevSpec &s, const FastSpec &f, const BgwState &st, const uint32_t *actions,
                                               int e, unsigned char *buf, int tid, int T)
{
    /* the action row is read by the attack pre-pass straight from global memory: warm L2 a whole env ahead */
    if (actions)
        for (int i = tid; i < (s.L * 4 + 127) / 128; i += T)
            asm volatile("prefetch.global.L2 [%0];" ::"l"((const char *)(actions + (size_t)e * s.L) + (size_t)i * 128));
    const size_t off = (size_t)e * s.A;
    if (f.async_ok == 2) {                                         /* rows are only 8-byte aligned (e.g. 24 entities) */
        const unsigned char *g;
        g = (const unsigned char *)(st.cell + off);
        for (int i = tid; i < s.A / 4; i += T) cp_async8(buf + f.b_cell + i * 8, g + i * 8);
        g = (const unsigned char *)(st.next + off);
        for (int i = tid; i < s.A / 4; i += T) cp_async8(buf + f.b_next + i * 8, g + i * 8);
        g = (const unsigned char *)(st.flags + off);
        for (int i = tid; i < s.A / 8; i += T) cp_async8(buf + f.b_flags + i * 8, g + i * 8);
    } else if (f.async_ok) {
        const unsigned char *g;
        g = (const unsigned char *)(st.cell + off);
        for (int i = tid; i < s.A / 8; i += T) cp_async16(buf + f.b_cell + i * 16, g + i * 16);
        g = (const unsigned char *)(st.next + off);
        for (int i = tid; i < s.A / 8; i += T) cp_async16(buf + f.b_next + i * 16, g + i * 16);
        g = (const unsigned char *)(st.flags + off);
        for (int i = tid; i < s.A / 16; i += T) cp_async16(buf + f.b_flags + i * 16, g + i * 16);
    } else {
        uint16_t *c = (uint16_t *)(buf + f.b_cell), *n = (uint16_t *)(buf + f.b_next);
        uint8_t *fl = buf + f.b_flags;
        for (int a = tid; a < s.A; a += T) { c[a] = st.cell[off + a]; n[a] = st.next[off + a]; fl[a] = st.flags[off + a]; }
    }
}

/* BinaryAttackActor for one attacker with a candidate-cell bit mask (row-major window order, actor.py:489-496) */
template <typename HT>
__device__ void fast_exec_attack(const DevSpec &s, const FastSpec &f, Env &ev, FastEnv &fe, int rank, int a, uint32_t mask)
{
    if (!(ev.flags[a] & BGW_ST_ACTIVE)) return;                   /* team_battle_example.py:37 */
    const int R = f.uniform_att >= 0 ? f.uniform_att : __ldg(&s.attack_r[a]), n = 2 * R + 1;
    const int own = ev.cell[a];
    const unsigned long long row = __ldg(&s.attack_map[ev.enc[a]]);
    const double acc = f.acc_lt1 ? __ldg(&s.accuracy[a]) : 1.0;    /* 1.0: the accuracy draws fold away */
    int ncand = 0, v = -1, vcell = 0;                              /* v: the first candidate in scan order */
    for (uint32_t m = mask; m; m &= m - 1) {
        const int b = __ffs(m) - 1, wr = b / n, wc = b - wr * n;
        const int cc = own + (wr - R) * s.W + (wc - R);
        for (unsigned o = fl_first<HT>(fe, cc, pad_index(s, f, cc)); o != BGW_NONE16; o = ev.next[o])
            if (basic_criteria(s, ev, a, (int)o, row, acc) && ncand++ == 0) { v = (int)o; vcell = cc; }
    }
    if (ncand == 0) { fe.rflag[a] |= RF_ATTACK_FAIL; return; }
    if (ncand > 1) {
        /* _subset_attackables actor.py:394-414: one keyed draw over the candidate list (with a single candidate the
         * choice is forced and, the stream being keyed, the draw is skipped) */
        int j = (int)bgw_index(dev_draw(s, ev, BGW_SITE_SUBSET, (uint32_t)a, 0), (uint32_t)ncand);
        v = -1;
        for (uint32_t m = mask; m && v < 0; m &= m - 1) {
            const int b = __ffs(m) - 1, wr = b / n, wc = b - wr * n;
            vcell = own + (wr - R) * s.W + (wc - R);
            for (unsigned o = fl_first<HT>(fe, vcell, pad_index(s, f, vcell)); o != BGW_NONE16; o = ev.next[o])
                if (basic_criteria(s, ev, a, (int)o, row, acc) && j-- == 0) { v = (int)o; break; }
        }
    }
    /* actor.py:353-358; HealthAgent.health setter agent.py:192-196 (health stays in HBM, touched only on a hit) */
    {   /* the setter clamps health to [0, 1] (here and at reset), so a hit of strength >= 1 leaves 0 whatever the health was:
         * the common case needs no round trip to L2 on the critical path of the ordered rounds */
        const double hit = __ldg(&s.strength[a]);
        set_health(ev, v, hit >= 1.0 ? 0.0 : __ldcg(&ev.health[v]) - hit);
    }
    if (!(ev.flags[v] & BGW_ST_ACTIVE)) {
        fe.cenc[pad_index(s, f, vcell)] = fl_summary(ev, fl_unlink<HT>(ev, fe, v), f.can_mix);
        fe.killrank[v] = (uint16_t)rank;
        atomicAdd(&ev.ctr[CTR_KILLS], 1);
        fe.rflag[v] |= RF_DIED;                                   /* team_battle_example.py:44-47 */
        fe.rflag[a] |= RF_KILL;
    }
}

/* ---- ordered rounds ---------------------------------------------------------------------------------------
 * Agents whose actions touch disjoint cells commute; agents that share a cell must act in rank order.  Every
 * pending agent atomicMin()s a TAGGED rank (epoch << 12 | rank) into the slot of every cell its action may read
 * or write; after ONE barrier an agent that finds its own value in all its slots executes, the others retry in
 * the next round.  The epoch decreases from round to round, so whatever earlier rounds (or earlier phases, or
 * earlier envs of this CTA) left in a slot is larger than any current value and reads as free: slots are never
 * released or cleared.  The slot array is split in two tables used by alternate rounds: a loser reserves for the
 * next round right away, in the other table, while the winners of this round are still reading this one -- the
 * barrier that ends a round is the barrier that publishes the next round's reservations. */
#define BGW_TAG_SHIFT 12                      /* ranks < BGW_MAX_AGENTS = 4096 */

struct SlotTables {
    uint32_t *t0, *t1;
    uint32_t mask;
    __device__ __forceinline__ uint32_t *tab(int p) const { return p ? t1 : t0; }
};

__device__ __forceinline__ SlotTables slot_tables(const DevSpec &s, const Env &ev)
{
    SlotTables t;
    const uint32_t half = (uint32_t)(s.slot_mask + 1) >> 1;
    t.t0 = ev.slot; t.t1 = ev.slot + half; t.mask = half - 1u;
    return t;
}

/* reserve / test the slots of an attacker: its own cell and the cells of its candidate mask */
__device__ __forceinline__ void attack_reserve(const DevSpec &s, uint32_t *tab, uint32_t smask, int own, int R, uint32_t mask, uint32_t v)
{
    const int n = 2 * R + 1;
    BGW_JITTER_POINT(1);
    atomicMin(&tab[own & smask], v);
    for (uint32_t m = mask; m; m &= m - 1) {
        const int b = __ffs(m) - 1, wr = b / n, wc = b - wr * n;
        atomicMin(&tab[(own + (wr - R) * s.W + (wc - R)) & smask], v);
    }
}

__device__ __forceinline__ bool attack_holds(const DevSpec &s, const uint32_t *tab, uint32_t smask, int own, int R, uint32_t mask, uint32_t v)
{
    const int n = 2 * R + 1;
    BGW_JITTER_POINT(2);
    bool win = tab[own & smask] == v;
    for (uint32_t m = mask; m; m &= m - 1) {
        const int b = __ffs(m) - 1, wr = b / n, wc = b - wr * n;
        win &= tab[(own + (wr - R) * s.W + (wc - R)) & smask] == v;
    }
    return win;
}

/* Ordered rounds over the effective attackers eff[0..n_eff): all of them pending on entry, with their first
 * reservation already made in table 0 under `epoch` (by the attack pre-pass) and published by a barrier.
 * WARP = run by one warp with __syncwarp.  Returns the next unused epoch. */
/* The warp that runs the single-warp reservation rounds of an env: the LAST one; the first one compacts and keeps the books
 * (tickets, env flags, statistics).  With every single-warp job on warp 0 the sub-partitions that hold the first warps issued
 * 68 % of their slots and the others 38 %; measured with the rounds moved: 0.0423 -> 0.0408 ms per step (driver setting). */
#define BGW_ROUNDS_WARP(T) (((T) >> 5) - 1)

template <bool WARP, typename HT>
__device__ uint32_t fast_attack_rounds(const DevSpec &s, const FastSpec &f, Env &ev, FastEnv &fe, int n_eff, uint32_t epoch, int tid, int T)
{
    const int stride = WARP ? 32 : T;
    const SlotTables st = slot_tables(s, ev);
    int pending = 1, p = 0;
    while (pending) {
        const uint32_t tag = epoch << BGW_TAG_SHIFT, next_tag = (epoch - 1u) << BGW_TAG_SHIFT;
        int lost = 0;
        for (int x = tid; x < n_eff; x += stride) {
            const int i = fe.eff[x];
            if (ev.pstate[i] != 1) continue;
            const int a = ev.ragent[i], R = f.uniform_att >= 0 ? f.uniform_att : __ldg(&s.attack_r[a]), own = ev.cell[a];
            const uint32_t mask = fe.rkmask[i];
            if (!attack_holds(s, st.tab(p), st.mask, own, R, mask, tag | (uint32_t)i)) {
                lost = 1;
                attack_reserve(s, st.tab(p ^ 1), st.mask, own, R, mask, next_tag | (uint32_t)i);
                continue;
            }
            BGW_JITTER_POINT(9);
            fast_exec_attack<HT>(s, f, ev, fe, i, a, mask);
            ev.pstate[i] = 0;
        }
        if (WARP) { pending = __any_sync(0xFFFFFFFFu, lost); __syncwarp(); } else pending = __syncthreads_or(lost);
        p ^= 1; --epoch;
    }
    return epoch;
}

/* one move: Grid.query through the summary, then remove / place (actor.py:99-114).  The common move -- alone in its
 * cell, destination empty -- touches no occupant list; its four conditions are loaded and combined without
 * short-circuit branches. */
template <typename HT>
__device__ __forceinline__ void fast_exec_move(const DevSpec &s, const FastSpec &f, Env &ev, FastEnv &fe, int a, int from, int to)
{
    const int pto = pad_index(s, f, to);
    const int8_t summary = fe.cenc[pto], me = ev.enc[a];
    const unsigned fl = ev.flags[a], hd = ((const HT *)fe.head)[from], nx = ev.next[a];
    if ((summary == 0) & ((fl & BGW_ST_IN_GRID) != 0) & (hd == (unsigned)a) & (nx == BGW_NONE16)) {
        fe.cenc[pad_index(s, f, from)] = 0;                        /* Grid.remove: the cell is empty again */
        fe.cenc[pto] = me;                                         /* Grid.place into an empty cell */
        ((HT *)fe.head)[to] = (HT)a;
        ev.cell[a] = (uint16_t)to;
        return;
    }
    bool ok = true;
    if (summary != 0) {
        const unsigned long long row = __ldg(&s.overlap[me]);
        if (!f.can_mix || summary != (int8_t)BGW_MIXED) ok = (row >> summary) & 1ull;
        else                                                        /* Grid.query grid.py:81-105 over a mixed cell */
            for (unsigned o = ((const HT *)fe.head)[to]; o != BGW_NONE16; o = ev.next[o])
                if (!((row >> ev.enc[o]) & 1ull)) { ok = false; break; }
    }
    if (!ok) { fe.rflag[a] |= RF_MOVE_FAIL; return; }
    if (fl & BGW_ST_IN_GRID) fe.cenc[pad_index(s, f, from)] = fl_summary(ev, fl_unlink<HT>(ev, fe, a), f.can_mix);
    fl_append<HT>(ev, fe, a, to, summary != 0);
    /* (without mixed cells a move into an occupied cell is only legal among the mover's own encoding) */
    const int8_t ns = (!f.can_mix || summary == 0 || summary == me) ? me : (int8_t)BGW_MIXED;
    fe.cenc[pto] = ns;
    if (f.can_mix && ns == (int8_t)BGW_MIXED) ev.ctr[CTR_MIXED] = 1;
}

#define BGW_NO_MOVE 0xFFFFFFFFu
/* ---- the move phase -------------------------------------------------------------------------------------------
 * rkmask[i] = (source cell << 16 | destination cell) for a rank with a pending move, BGW_NO_MOVE otherwise (the attack
 * masks are dead by then).  A move reads and writes nothing but its source and its destination cell (their occupant
 * lists and summaries), so a move whose two cells are named by no other pending move commutes with every other move
 * and needs no ordering at all.  The classification loop marks every named cell in two bit maps (one bit per cell:
 * named once / named again); after one barrier a mover that finds neither of its cells named twice executes at once,
 * whatever its rank.  Only the CONTESTED movers (about one in ten on the headline workload) go through the ordered
 * reservation rounds; being few, they rarely alias in the hashed slot tables (round 1 had every mover reserve two of
 * 256 slots: half of them lost a round to an alias).  Contested movers are kept in two lists (the storage of eff[] /
 * killrank[], both dead by now): a round walks the losers of the round before. */
__device__ __forceinline__ void touch_mark(const FastSpec &f, FastEnv &fe, int cell)
{
    BGW_JITTER_POINT(3);
    const uint32_t bit = 1u << (cell & 31);
    uint32_t *w = fe.touch + ((cell >> 5) & (f.touch_words - 1));
    if (atomicOr(w, bit) & bit) atomicOr(w + f.touch_words, bit);
}

/* Ordered rounds over the n_cur contested movers listed in eff[], each with its first reservation made in table 0
 * under `epoch` and published by a barrier.  WARP = run by one warp with __syncwarp.  Returns the next unused epoch. */
template <bool WARP, typename HT>
__device__ uint32_t fast_move_rounds(const DevSpec &s, const FastSpec &f, Env &ev, FastEnv &fe, int n_cur, uint32_t epoch, int tid, int T)
{
    const int stride = WARP ? 32 : T;
    const SlotTables st = slot_tables(s, ev);
    uint32_t *cur = st.t0, *nxt = st.t1;                           /* this round's table / the next round's */
    int which = 0, base0 = 0, base1 = 0;                           /* the list counters only grow: entries before base are consumed */
    int pending = 1;
    while (pending) {
        const uint32_t tag = epoch << BGW_TAG_SHIFT, next_tag = (epoch - 1u) << BGW_TAG_SHIFT;
        const uint16_t *walk = which ? fe.killrank : fe.eff;
        uint16_t *losers = which ? fe.eff : fe.killrank;
        int *lctr = &ev.ctr[CTR_PA + (which ^ 1)];
        const int lbase = which ? base0 : base1;
        int lost = 0;
        for (int x = tid; x < n_cur; x += stride) {
            const int i = walk[x];
            const uint32_t ft = fe.rkmask[i];
            const int from = (int)(ft >> 16), to = (int)(ft & 0xFFFFu);
            const uint32_t mine = tag | (uint32_t)i, sf = (uint32_t)from & st.mask, sto = (uint32_t)to & st.mask;
            BGW_JITTER_POINT(4);
            const uint32_t hf = cur[sf], ht = cur[sto];                 /* both loads in flight, one test */
            if ((hf != mine) | (ht != mine)) {
                lost = 1;
                atomicMin(&nxt[sf], next_tag | (uint32_t)i);
                atomicMin(&nxt[sto], next_tag | (uint32_t)i);
                losers[atomicAdd(lctr, 1) - lbase] = (uint16_t)i;
                continue;
            }
            fast_exec_move<HT>(s, f, ev, fe, ev.ragent[i], from, to);
        }
        if (WARP) { pending = __any_sync(0xFFFFFFFFu, lost); __syncwarp(); }
        else pending = __syncthreads_or(lost);
        if (which) base1 += n_cur; else base0 += n_cur;            /* the list walked in this round is consumed */
        n_cur = *(volatile int *)lctr - lbase;                     /* the losers of this round */
        which ^= 1;
        { uint32_t *t = cur; cur = nxt; nxt = t; }
        --epoch;
    }
    return epoch;
}

/* All pending moves of an env (every thread of the CTA; the touch bit maps were filled by the classification loop and
 * published by a barrier).  Leaves the bit maps clean.  Returns the next unused epoch. */
template <typename HT>
__device__ uint32_t fast_move_phase(const DevSpec &s, const FastSpec &f, Env &ev, FastEnv &fe, int n_act, uint32_t epoch, int tid, int T)
{
    const SlotTables st = slot_tables(s, ev);
    const uint32_t *twice = fe.touch + f.touch_words;
    const uint32_t tw = (uint32_t)f.touch_words - 1u, tag = epoch << BGW_TAG_SHIFT;
    for (int i = tid; i < n_act; i += T) {
        const uint32_t ft = fe.rkmask[i];
        if (ft == BGW_NO_MOVE) continue;
        const int from = (int)(ft >> 16), to = (int)(ft & 0xFFFFu);
        BGW_JITTER_POINT(5);
        const uint32_t c = (twice[((uint32_t)from >> 5) & tw] >> (from & 31)) | (twice[((uint32_t)to >> 5) & tw] >> (to & 31));
        if (c & 1u) {                                               /* contested: first reservation, into the list */
            fe.eff[atomicAdd(&ev.ctr[CTR_PA], 1)] = (uint16_t)i;
            atomicMin(&st.t0[(uint32_t)from & st.mask], tag | (uint32_t)i);
            atomicMin(&st.t0[(uint32_t)to & st.mask], tag | (uint32_t)i);
        } else {
            fast_exec_move<HT>(s, f, ev, fe, ev.ragent[i], from, to);
        }
    }
    __syncthreads();
    {
        uint4 *t4 = reinterpret_cast<uint4 *>(fe.touch);
        for (int w = tid; w < f.touch_words / 2; w += T) t4[w] = make_uint4(0, 0, 0, 0);
    }
    const int n_con = ev.ctr[CTR_PA];
    if (n_con > 0) {                    /* few: one warp runs the rounds (also beyond 32); every thread keeps the same epoch */
        if ((tid >> 5) == BGW_ROUNDS_WARP(T)) {
            const uint32_t e2 = fast_move_rounds<true, HT>(s, f, ev, fe, n_con, epoch, tid & 31, T);
            if ((tid & 31) == 0) ev.ctr[CTR_EPOCH] = (int)e2;
        }
        __syncthreads();
        return (uint32_t)ev.ctr[CTR_EPOCH];
    }
    return epoch;
}

/* (re)initialise the dense per-cell arrays of this CTA: clean head-detection marks, free reservation slots, empty
 * summary with a -1 border (the list heads need no initialisation: the summary says which are meaningful) */
static __device__ void fast_init_dense(const DevSpec &s, const FastSpec &f, Env &ev, FastEnv &fe, int tid, int T)
{
    const uint4 ones = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
    for (int a = tid; a < s.A; a += T) ev.tmp[a] = 0;
    {   /* reservation slots: every round frees what it reserved, so they only need filling here (and after a
         * reset, whose availability maps share the scratch union) */
        uint4 *s4 = (uint4 *)ev.slot;
        for (int i = tid; i < (s.slot_mask + 1) / 4; i += T) s4[i] = ones;
        uint4 *t4 = (uint4 *)fe.touch;                             /* touch bit maps of the move phase: clean between envs */
        for (int i = tid; i < f.touch_words / 2; i += T) t4[i] = make_uint4(0, 0, 0, 0);
    }
    /* summary rows: word cw of an interior row has zeros where its 4 bytes fall inside the grid columns */
    uint32_t *c32 = (uint32_t *)fe.cenc;
    const int wpr = f.PW >> 2, lane = tid & 31, warp = tid >> 5, nwarp = T >> 5;
    for (int cw = lane; cw < wpr; cw += 32) {
        uint32_t inner = 0xFFFFFFFFu;
#pragma unroll
        for (int bb = 0; bb < 4; ++bb) {
            const int cc = cw * 4 + bb;
            if (cc >= f.PL && cc < f.PL + s.W) inner &= ~(0xFFu << (8 * bb));
        }
        for (int rr = warp; rr < f.PH; rr += nwarp)
            c32[rr * wpr + cw] = (rr >= f.P && rr < f.P + s.H) ? inner : 0xFFFFFFFFu;
    }
    if (tid < 8) c32[f.PH * wpr + tid] = 0xFFFFFFFFu;           /* slack words read by the row gather */
    __syncthreads();
}

/* the general per-cell observation chunk on top of the summary: used when the env holds a mixed cell, an
 * observer does not observe itself, or the compile-time gather does not apply */
template <typename HT>
__device__ void fast_obs_chunk_slow(const DevSpec &s, const FastSpec &f, const Env &ev, const FastEnv &fe, int a, int ch,
                                    uint32_t w[4])
{
    w[0] = w[1] = w[2] = w[3] = 0;
    if (!(ev.klass[a] & BGW_AG_OBSERVING)) return;
    const int R = __ldg(&s.view_r[a]), n = 2 * R + 1, valid = n * n, k0 = ch * 16;
    int r0, c0;
    cell_rc(s, f, ev.cell[a], r0, c0);
    const int8_t *win = fe.cenc + (r0 + f.P - R) * f.PW + (c0 + f.PL - R);
    int wr = k0 / n, wc = k0 - wr * n;
    for (int t = 0; t < 16 && k0 + t < valid; ++t) {
        int v = win[wr * f.PW + wc];
        const bool centre = (wr == R && wc == R);
        if (v == BGW_MIXED || (centre && !s.observe_self && v > 0)) {
            /* np.random.choice over the encodings of the occupants in arrival order (observer.py:233-246) */
            const int cell = (r0 - R + wr) * s.W + (c0 - R + wc), skip = s.observe_self ? -1 : a;
            const unsigned first = ((const HT *)fe.head)[cell];
            int cnt = 0;
            for (unsigned o = first; o != BGW_NONE16; o = ev.next[o]) cnt += ((int)o != skip);
            v = 0;
            if (cnt > 0) {
                int k = (cnt == 1) ? 0 : (int)bgw_index(dev_draw(s, ev, BGW_SITE_OBS, (uint32_t)a, (uint32_t)cell), (uint32_t)cnt);
                for (unsigned o = first; o != BGW_NONE16; o = ev.next[o]) {
                    if ((int)o == skip) continue;
                    if (k-- == 0) { v = ev.enc[o]; break; }
                }
            }
        }
        w[t >> 2] |= (uint32_t)(uint8_t)(int8_t)v << ((t & 3) * 8);
        if (++wc == n) { wc = 0; ++wr; }
    }
}

/* 32 contiguous bytes from one lane: STG.256 (sm_100), one full sector per lane and instruction */
__device__ __forceinline__ void st_global_256(void *p, const uint32_t *v)
{
#ifdef BGW_NO_ST256            /* a run-time compilation by an NVRTC older than 12.9 (PTX 8.8): two 128-bit stores */
    reinterpret_cast<uint4 *>(p)[0] = make_uint4(v[0], v[1], v[2], v[3]);
    reinterpret_cast<uint4 *>(p)[1] = make_uint4(v[4], v[5], v[6], v[7]);
    return;
#endif
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
                 "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}

/* ---- cooperative row gather (view ranges 5 and 3: the observation row is 4 / 2 chunks of 32 bytes) -----------------
 * LPA lanes share one learner: lane q of the group produces bytes [32q, 32q + 32) of the packed row and the group writes one
 * contiguous piece of a 128-byte line with a single 256-bit store per lane.  (One lane per learner -- fast_obs_rows_lane
 * below -- made every lane of a store instruction write into a line of its own: ncu counted 5.5 LSU data-pipe wavefronts per
 * row for the stores alone, more than for the window loads.)  Chunk q needs the window rows i = a*q + b + r, r = 0..NR-1
 * (rows outside 0..n-1 do not exist and read as nothing); they are packed at n*r into the register stream S exactly as the
 * one-lane gather packs a whole window, and the chunk is S from byte 32q - n*(a*q + b) on: a compile-time word offset plus a
 * lane-dependent shift of 0..4 bytes (shf.r.clamp), so every register index stays static. */
template <int R> struct ObsCoop { static constexpr bool on = false; static constexpr int LPA = 1, a = 0, b = 0, NR = 0; };
template <> struct ObsCoop<5> { static constexpr bool on = true; static constexpr int LPA = 4, a = 3, b = -1, NR = 4; };   /* start byte 11 - q */
template <> struct ObsCoop<3> { static constexpr bool on = true; static constexpr int LPA = 2, a = 4, b = 0, NR = 5; };    /* start byte 4q */

/* bytes [lo, hi) of window-row slot r that some lane of the group needs (compile time) */
template <int R>
__host__ __device__ constexpr int obs_coop_lo(int r)
{
    typedef ObsCoop<R> C;
    const int n = 2 * R + 1;
    int lo = n;
    for (int q = 0; q < C::LPA; ++q) {
        const int st = 32 * q - n * (C::a * q + C::b) - n * r;     /* chunk start relative to the row's first byte */
        const int l = st < 0 ? 0 : st;
        if (l < lo && st + 32 > 0 && st < n) lo = l;
    }
    return lo;
}
template <int R>
__host__ __device__ constexpr int obs_coop_hi(int r)
{
    typedef ObsCoop<R> C;
    const int n = 2 * R + 1;
    int hi = 0;
    for (int q = 0; q < C::LPA; ++q) {
        const int st = 32 * q - n * (C::a * q + C::b) - n * r;
        const int h = st + 32 > n ? n : st + 32;
        if (h > hi && st + 32 > 0 && st < n) hi = h;
    }
    return hi;
}

template <int R>
__device__ void fast_obs_rows_coop(const DevSpec &s, const FastSpec &f, const Env &ev, const FastEnv &fe, int n_act, int8_t *obs_env,
                                   int tid, int T)
{
    typedef ObsCoop<R> C;
    constexpr int n = 2 * R + 1, LPA = C::LPA, NR = C::NR;
    constexpr int RW = (n + 3) / 4;            /* words of an aligned row */
    constexpr int LW = (n + 6) / 4;            /* words to load: alignment shift (<= 3 bytes) + n bytes */
    constexpr int ST0 = -n * C::b, SLOPE = 32 - n * C::a;               /* chunk q starts at byte ST0 + SLOPE*q of S */
    constexpr int ST_MIN = SLOPE >= 0 ? ST0 : ST0 + SLOPE * (LPA - 1);
    constexpr int W0 = ST_MIN / 4;
    constexpr int SW = W0 + 9;                 /* words of S the chunk extraction reads */
    static_assert(ST_MIN >= 0 && (SLOPE >= 0 ? ST0 + SLOPE * (LPA - 1) : ST0) - 4 * W0 <= 4, "lane-dependent shift must stay within 0..4 bytes");
    static_assert((NR * n + 3) / 4 <= SW, "stream longer than the extraction window");
    const int q = tid & (LPA - 1);
    const int dyn = (ST0 + SLOPE * q - 4 * W0) * 8;
    const int pw4 = f.PW >> 2;
    const bool wide = ((s.obs_stride & 31) == 0) && ((reinterpret_cast<uintptr_t>(obs_env) & 31) == 0);
    for (int li = tid / LPA; li < n_act; li += T / LPA) {
        const int a = ev.ragent[li];
        const bool observing = ev.klass[a] & BGW_AG_OBSERVING;
        const int i0 = C::a * q + C::b;                                   /* first window row of this lane's chunk */
        const int o = pad_index(s, f, ev.cell[a]) - R * f.PW - R;
        const uint32_t *wp = reinterpret_cast<const uint32_t *>(fe.cenc + (o & ~3)) + i0 * pw4;
        const int sh = (o & 3) * 8;
        uint32_t S[SW + 1];
#pragma unroll
        for (int j = 0; j <= SW; ++j) S[j] = 0;
        if (observing) {
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                const int lo = obs_coop_lo<R>(r), hi = obs_coop_hi<R>(r);     /* compile-time after unrolling */
                if (hi <= lo) continue;
                const bool ok = (unsigned)(i0 + r) < (unsigned)n;             /* the window has this row */
                const uint32_t *rp = wp + r * pw4;
                uint32_t x[LW + 1], y[RW];
                /* aligned words j, j+1 of the padded row give bytes 4j..4j+3 of the window row; only the words some lane's
                 * chunk reaches are loaded, the last one only where the row's alignment reaches into it */
#pragma unroll
                for (int j = 0; j <= LW; ++j) {
                    const bool ny = j < RW && !(4 * j + 4 <= lo || 4 * j >= hi);
                    const bool nyp = j > 0 && j - 1 < RW && !(4 * (j - 1) + 4 <= lo || 4 * (j - 1) >= hi);
                    if (j < LW && (ny || nyp)) x[j] = (ok && (j < LW - 1 || sh + 8 * n > 32 * (LW - 1))) ? rp[j] : 0u;
                    else x[j] = 0;
                }
#pragma unroll
                for (int j = 0; j < RW; ++j)
                    y[j] = (4 * j + 4 <= lo || 4 * j >= hi) ? 0u : __funnelshift_r(x[j], x[j + 1], sh);
                constexpr int vb = n - 4 * (RW - 1);
                if (vb < 4) y[RW - 1] &= (1u << (8 * (vb & 3))) - 1u;
                const int d = n * r, qw = d >> 2, s8 = (d & 3) * 8;
#pragma unroll
                for (int j = 0; j < RW; ++j) {
                    if (4 * j + 4 <= lo || 4 * j >= hi) continue;
                    if (qw + j <= SW) S[qw + j] |= y[j] << s8;
                    if (s8 != 0 && qw + j + 1 <= SW) S[qw + j + 1] |= y[j] >> (32 - s8);
                }
            }
        }
        uint32_t out[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) out[j] = __funnelshift_rc(S[W0 + j], S[W0 + j + 1], dyn);
        if (32 * q < s.obs_stride) {
            int8_t *dg = obs_env + (size_t)ev.plist[li] * s.obs_stride + 32 * q;
            if (wide) st_global_256(dg, out);
            else {
                *reinterpret_cast<uint4 *>(dg) = make_uint4(out[0], out[1], out[2], out[3]);
                *reinterpret_cast<uint4 *>(dg + 16) = make_uint4(out[4], out[5], out[6], out[7]);
            }
        }
    }
}

/* Observation rows of the acting learners, view range R known at compile time.  One thread gathers one
 * learner's window: per window row LW aligned words, funnel-shifted to the row's first byte, then appended at
 * byte n*i of the packed output (all shifts are compile-time after unrolling).  The packed row is produced in
 * groups of 64 bytes held in registers and leaves the lane as two 256-bit stores per group (rows that are 32-byte
 * aligned; 128-bit stores otherwise): every store instruction writes 32 full sectors.  (Round 1 transposed the groups
 * through a shared-memory stage into coalesced 128-bit stores: half of the gather's instructions and a third of its
 * shared-memory wavefronts were that transposition.) */
template <int R>
__device__ void fast_obs_rows_lane(const DevSpec &s, const FastSpec &f, const Env &ev, const FastEnv &fe, int n_act, int8_t *obs_env,
                                   int tid, int T)
{
    constexpr int n = 2 * R + 1, NB = n * n;
    constexpr int RW = (n + 3) / 4;            /* words of an aligned row */
    constexpr int LW = (n + 6) / 4;            /* words to load: alignment shift (<= 3 bytes) + n bytes */
    constexpr int NG = (NB + 63) / 64;         /* 64-byte groups of the output row */
    const int pw4 = f.PW >> 2;
    const bool wide = ((s.obs_stride & 31) == 0) && ((reinterpret_cast<uintptr_t>(obs_env) & 31) == 0);
    for (int li = tid; li < n_act; li += T) {
        const int a = ev.ragent[li];
        const bool observing = ev.klass[a] & BGW_AG_OBSERVING;
        const int o = pad_index(s, f, ev.cell[a]) - R * f.PW - R;
        const uint32_t *wp = reinterpret_cast<const uint32_t *>(fe.cenc + (o & ~3));
        const int sh = (o & 3) * 8;
        int8_t *dst = obs_env + (size_t)ev.plist[li] * s.obs_stride;
#pragma unroll
        for (int g = 0; g < NG; ++g) {
            uint32_t out[16];
#pragma unroll
            for (int j = 0; j < 16; ++j) out[j] = 0;
            if (observing) {
#pragma unroll
                for (int i = 0; i < n; ++i) {
                    const int d = n * i;                              /* first output byte of window row i */
                    if (d + n <= 64 * g || d >= 64 * (g + 1)) continue;   /* row does not touch this group */
                    const uint32_t *rp = wp + i * pw4;
                    uint32_t x[LW + 1], y[RW];
                    /* the last aligned word only where the row reaches into it: a third of the gather's shared-memory
                       wavefronts are bank conflicts of 32 unrelated rows, fewer lanes, fewer conflicts */
#pragma unroll
                    for (int j = 0; j < LW; ++j) x[j] = (j < LW - 1 || sh + 8 * n > 32 * (LW - 1)) ? rp[j] : 0u;
                    x[LW] = 0;
#pragma unroll
                    for (int j = 0; j < RW; ++j) y[j] = __funnelshift_r(x[j], x[j + 1], sh);
                    constexpr int vb = n - 4 * (RW - 1);
                    if (vb < 4) y[RW - 1] &= (1u << (8 * (vb & 3))) - 1u;
                    const int q = (d >> 2) - 16 * g, s8 = (d & 3) * 8;
#pragma unroll
                    for (int j = 0; j < RW; ++j) {
                        if (q + j >= 0 && q + j < 16) out[q + j] |= y[j] << s8;
                        if (s8 != 0 && q + j + 1 >= 0 && q + j + 1 < 16) out[q + j + 1] |= y[j] >> (32 - s8);
                    }
                }
            }
            const int nchg = min(4, s.nchunks - 4 * g);                  /* 16-byte chunks of this group that exist */
            int8_t *dg = dst + 64 * g;
#pragma unroll
            for (int h = 0; h < 2; ++h) {                                 /* the two 32-byte halves of the group */
                if (wide && nchg >= 2 * h + 2) st_global_256(dg + 32 * h, out + 8 * h);
                else {
                    if (nchg >= 2 * h + 1) *reinterpret_cast<uint4 *>(dg + 32 * h) = make_uint4(out[8 * h], out[8 * h + 1], out[8 * h + 2], out[8 * h + 3]);
                    if (nchg >= 2 * h + 2) *reinterpret_cast<uint4 *>(dg + 32 * h + 16) = make_uint4(out[8 * h + 4], out[8 * h + 5], out[8 * h + 6], out[8 * h + 7]);
                }
            }
        }
    }
}

template <int R>
__device__ __forceinline__ void fast_obs_rows(const DevSpec &s, const FastSpec &f, const Env &ev, const FastEnv &fe, int n_act, int8_t *obs_env,
                                              int tid, int T)
{
    if constexpr (ObsCoop<R>::on) fast_obs_rows_coop<R>(s, f, ev, fe, n_act, obs_env, tid, T);
    else fast_obs_rows_lane<R>(s, f, ev, fe, n_act, obs_env, tid, T);
}

/* Compile-time shape of the headline workload (BASELINE configs[4]: 64x64 grid, 256 agents that are all learners,
 * view 5, MoveActor, observe_self, OneTeamRemainingDone).  bgw_create selects the instantiation of a shape when the
 * compiled spec matches it exactly; every other sim runs the FastDynamic instantiation with run-time shapes.  The
 * code is the same: the constants below only let the compiler fold divisions, strides and trip counts. */
struct FastStaticC5 {
    static constexpr bool is_static = true;
    static constexpr int A = 256, L = 256, H = 64, W = 64, P = 5, PL = 5, PW = 76, PH = 74, obs_stride = 128, nchunks = 8,
                         obs_h = 11, view = 5, move_actor = BGW_MOVE_BOX, ravel = 0, observe_self = 1, done_mask = BGW_DONE_ONE_TEAM,
                         max_enc = 4, simd_ok = 1, async_ok = 1, slots = 256, T = 64, att = 1, identity = 1, can_mix = 0, acc_lt1 = 0, rpo = 0,
                         LB_T = 64, LB_N = 8;
};
/* BASELINE configs[1] (examples/rllib_team_battle.py: 8x8 grid, 24 agents in 4 teams, view 3): one warp per env, 32 envs
 * per SM, each at its own place in the code -- the run-time-shape instantiation (9.3 k instructions) spends most of its
 * stall cycles waiting for instructions (ncu: no_instruction 5.4 per issue); this one is half the size. */
struct FastStaticC2 {
    static constexpr bool is_static = true;
    static constexpr int A = 24, L = 24, H = 8, W = 8, P = 3, PL = 3, PW = 16, PH = 14, obs_stride = 64, nchunks = 4,
                         obs_h = 7, view = 3, move_actor = BGW_MOVE_BOX, ravel = 0, observe_self = 1, done_mask = BGW_DONE_ONE_TEAM,
                         max_enc = 4, simd_ok = 1, async_ok = 2, slots = 64, T = 32, att = 1, identity = 1, can_mix = 0, acc_lt1 = 0, rpo = 0, LB_T = 128, LB_N = 7;
};
struct FastDynamic { static constexpr bool is_static = false; static constexpr int LB_T = 128, LB_N = 7; };

#ifndef __CUDACC_RTC__
/* does the compiled spec have exactly the compile-time shape C? (bgw_create) */
template <typename C>
inline bool fast_shape_matches(const DevSpec &q, const FastSpec &f, int threads)
{
    return q.A == C::A && q.L == C::L && q.H == C::H && q.W == C::W && q.obs_stride == C::obs_stride && q.obs_h == C::obs_h &&
           q.obs_c == 1 && q.move_actor == C::move_actor && q.ravel == C::ravel && q.observe_self == C::observe_self &&
           q.done_mask == C::done_mask && q.max_enc == C::max_enc && f.P == C::P && f.PL == C::PL && f.PW == C::PW &&
           f.PH == C::PH && f.uniform_view == C::view && f.simd_ok == C::simd_ok && f.async_ok == C::async_ok &&
           q.slot_mask == C::slots - 1 && threads == C::T && f.uniform_att == C::att && f.identity_learners == C::identity &&
           f.can_mix == C::can_mix && f.acc_lt1 == C::acc_lt1 && q.randomize_placement_order == C::rpo;
}
#endif

/* ---- phases of the per-env step (bgw_step_fast_body below), each run by every thread of the CTA ---------------------- */

/* Occupant lists and summary of the relevant entities.  Entry: compaction.  Exit: head / cenc describe the grid, rflag and
 * killrank of the relevant entities are clear (barrier).  `kept`: head / cenc still describe the grid from the env's step
 * before on this CTA (moves and kills keep them exact); only rflag / killrank are cleared, which nothing reads before the
 * attack pre-pass has ended with its barrier. */
template <typename HT>
__device__ __forceinline__ void fast_build_lists(const DevSpec &s, const FastSpec &f, Env &ev, FastEnv &fe, int n_rel, bool kept, int tid, int T)
{
    for (int x = tid; x < n_rel; x += T) {
        const int a = fe.rel[x];
        fe.rflag[a] = 0;
        fe.killrank[a] = BGW_NONE16;
        if (!kept && (ev.flags[a] & BGW_ST_IN_GRID)) {
            if (ev.next[a] != BGW_NONE16) ev.tmp[ev.next[a]] = 1;
            fe.cenc[pad_index(s, f, ev.cell[a])] = ev.enc[a];
        }
    }
    if (kept) return;
    __syncthreads();
    for (int x = tid; x < n_rel; x += T) {
        const int a = fe.rel[x];
        if (ev.flags[a] & BGW_ST_IN_GRID) {
            if (!ev.tmp[a]) ((HT *)fe.head)[ev.cell[a]] = (HT)a;
            ev.tmp[a] = 0;
            const int p = pad_index(s, f, ev.cell[a]);
            if (f.can_mix && fe.cenc[p] != ev.enc[a]) { fe.cenc[p] = (int8_t)BGW_MIXED; ev.ctr[CTR_MIXED] = 1; }
        }
    }
    __syncthreads();
}

/* Attack pre-pass (team_battle_example.py:35-47): each acting learner's learner index and action word, and for an attacker its
 * candidate cells; an effective attacker (one with a possible victim) makes its first reservation under `epoch`.  Entry: the
 * lists.  Exit: plist, act, rkmask, pstate and the effective attackers eff[0..ctr[CTR_NEMIT]) published (barrier). */
__device__ __forceinline__ void fast_attack_prepass(const DevSpec &s, const FastSpec &f, Env &ev, FastEnv &fe, const uint32_t *actions,
                                                    uint32_t *sampled, int n_act, uint32_t epoch, int tid, int T)
{
    const int e = ev.e;
    for (int i = tid; i < n_act; i += T) {
        const int a = ev.ragent[i], l = f.identity_learners ? a : __ldg(&s.learner_of[a]);
        ev.plist[i] = (uint16_t)l;
        if (sampled) {                                   /* bgw_step_sampled: the keyed random policy, fused */
            const uint32_t w = sample_action_word(s, a, ev.klass[a], ev.genv, ev.episode, ev.step - 1u);
            fe.act[l] = w;
            sampled[(size_t)e * s.L + l] = w;
        } else {
            fe.act[l] = __ldcg(&actions[(size_t)e * s.L + l]);   /* (prefetched to L2 while the env before ran) */
        }
        uint8_t p = 0;
        if ((ev.flags[a] & BGW_ST_ACTIVE) && (ev.klass[a] & BGW_AG_ATTACKING) && (int8_t)((fe.act[l] >> 16) & 0xFF) != 0) {
            /* candidate cells: the summary says an attackable encoding (or a mix) is present */
            const int R = f.uniform_att >= 0 ? f.uniform_att : __ldg(&s.attack_r[a]), n = 2 * R + 1;
            const unsigned long long row = __ldg(&s.attack_map[ev.enc[a]]);
            const int wo = pad_index(s, f, ev.cell[a]) - R * f.PW - R;
            const int8_t *w = fe.cenc + wo;
            uint32_t mask = 0;
            if (R == 1) {
                /* the three window rows as aligned word pairs, funnel-shifted to the window's first column; each of the nine
                 * bytes is tested from the register: v in 1..max_enc selects its bit of the attack map row, 0 (empty) and -1
                 * (border) select nothing (bit 0 of a row is never set; shifts clamp) */
                const uint32_t *wp = reinterpret_cast<const uint32_t *>(fe.cenc + (wo & ~3));
                const int sh = (wo & 3) * 8, pw4 = f.PW >> 2;
                uint32_t y[3];
#pragma unroll
                for (int k = 0; k < 3; ++k) y[k] = __funnelshift_r(wp[k * pw4], wp[k * pw4 + 1], sh);
                if (s.max_enc < 32) {
                    const uint32_t row32 = (uint32_t)row & ~1u;
#pragma unroll
                    for (int k = 0; k < 9; ++k) {
                        const uint32_t v = (y[k / 3] >> (8 * (k % 3))) & 0xFFu;
                        mask |= (__funnelshift_rc(row32, 0u, v) & 1u) << k;
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < 9; ++k) {
                        const uint32_t v = (y[k / 3] >> (8 * (k % 3))) & 0xFFu;
                        if (v < 64u && ((row >> v) & 1ull)) mask |= 1u << k;
                    }
                }
                if (f.can_mix && ev.ctr[CTR_MIXED]) {           /* a mixed cell is always a candidate (the walk decides) */
#pragma unroll
                    for (int k = 0; k < 9; ++k)
                        if (((y[k / 3] >> (8 * (k % 3))) & 0xFFu) == (uint32_t)(uint8_t)BGW_MIXED) mask |= 1u << k;
                }
            } else {
                for (int wr = 0; wr < n; ++wr)
                    for (int wc = 0; wc < n; ++wc) {
                        const int v = w[wr * f.PW + wc];
                        if (v > 0 ? (int)((row >> v) & 1ull) : (v == BGW_MIXED)) mask |= 1u << (wr * n + wc);
                    }
            }
            fe.rkmask[i] = mask;
            if (mask) {                                         /* effective attacker: first reservation right here */
                p = 1; fe.eff[atomicAdd(&ev.ctr[CTR_NEMIT], 1)] = (uint16_t)i;
                const SlotTables stt = slot_tables(s, ev);
                attack_reserve(s, stt.t0, stt.mask, ev.cell[a], R, mask, (epoch << BGW_TAG_SHIFT) | (uint32_t)i);
            }
            else p = 3;                                         /* no possible victim: settled after the rounds */
        }
        ev.pstate[i] = p;
    }
    __syncthreads();
}

/* The ordered rounds of the effective attackers.  Entry: the attack pre-pass.  Exit: every attack executed (barrier when there
 * was one); returns the next unused epoch, the same in every thread. */
template <typename HT>
__device__ __forceinline__ uint32_t fast_attack_phase(const DevSpec &s, const FastSpec &f, Env &ev, FastEnv &fe, uint32_t epoch, int lane, int warp, int T)
{
    const int n_eff = ev.ctr[CTR_NEMIT];
    if (n_eff > 0) {          /* few agents (an attack action AND a possible victim next to them): one warp runs the rounds, also
                                 beyond 32 of them; every thread keeps the same epoch */
        if (warp == BGW_ROUNDS_WARP(T)) {
            const uint32_t e2 = fast_attack_rounds<true, HT>(s, f, ev, fe, n_eff, epoch, lane, T);
            if (lane == 0) ev.ctr[CTR_EPOCH] = (int)e2;
        }
        __syncthreads();
        epoch = (uint32_t)ev.ctr[CTR_EPOCH];
    }
    else --epoch;
    return epoch;
}

/* launch bounds per instantiation: the headline shape runs 64 threads per env and is limited to 11 envs per SM by shared memory,
 * so it may use more registers than the run-time-shape code (up to 128 threads): 71 instead of 64 makes its code 5 % smaller
 * (3568 instructions; measured +1 %) */
#define BGW_FAST_LB __launch_bounds__(SHAPE::LB_T, SHAPE::LB_N)
template <typename SHAPE, typename HT>
__device__ __forceinline__ void bgw_step_fast_body(const DevSpec &s_in, const FastSpec &f_in, const BgwState &st, const uint32_t *actions,
                                                   uint32_t *sampled, const int16_t *order, int8_t *obs, float *reward, uint8_t *done,
                                                   uint8_t *all_done)
{
    DevSpec s = s_in;
    FastSpec f = f_in;
    if constexpr (SHAPE::is_static) {
        typedef SHAPE C;
        s.A = C::A; s.L = C::L; s.H = C::H; s.W = C::W; s.HW = C::H * C::W; s.obs_stride = C::obs_stride; s.nchunks = C::nchunks;
        s.obs_h = s.obs_w = C::obs_h; s.obs_c = 1; s.move_actor = C::move_actor; s.ravel = C::ravel; s.observe_self = C::observe_self;
        s.done_mask = C::done_mask; s.max_enc = C::max_enc; s.n_blk = 0; s.program = BGW_PROG_TEAM_BATTLE;
        s.randomize_placement_order = C::rpo;               /* (folds the shuffled-placement code out of the inlined reset) */
        s.manager = BGW_MANAGER_ALL_STEP; s.attack_actor = BGW_ATTACK_BINARY; s.hw_words = (C::H * C::W + 31) / 32;
        f.P = C::P; f.PL = C::PL; f.PW = C::PW; f.PH = C::PH; f.uniform_view = C::view; f.simd_ok = C::simd_ok; f.async_ok = C::async_ok;
        f.uniform_att = C::att; f.identity_learners = C::identity; f.can_mix = C::can_mix; f.acc_lt1 = C::acc_lt1;
        f.magic_w = (uint32_t)(((1ull << 32) + C::W - 1) / C::W);
        s.slot_mask = C::slots - 1;
        constexpr FastLayout LY = fast_layout(C::A, C::L, C::H * C::W, C::PH, C::PW, C::slots, C::T, C::max_enc, (C::H * C::W + 31) / 32, C::identity);
        fast_apply_layout(f, LY);
    }
    int T_ = (int)blockDim.x;
    if constexpr (SHAPE::is_static) T_ = SHAPE::T;
    const int tid = threadIdx.x, T = T_, lane = tid & 31, warp = tid >> 5, nwarp = T >> 5;
    unsigned char *scratch = bgw_smem + f.o_scratch;
    Env ev;
    ev.enc = (int8_t *)(bgw_smem + f.o_enc);
    ev.klass = bgw_smem + f.o_klass;
    ev.tmp = bgw_smem + f.o_tmp;
    ev.head = nullptr;                                     /* the fast kernel keeps its own typed heads (fe.head) */
    ev.ragent = (uint16_t *)(bgw_smem + f.o_ragent);
    ev.plist = (uint16_t *)(bgw_smem + f.o_plist);
    ev.ctr = (int *)(bgw_smem + f.o_ctr);
    ev.racc = nullptr;                                     /* float64 accumulators exist only in the reset arena */
    ev.slot = (uint32_t *)(scratch + f.s_slot);
    ev.pstate = scratch + f.s_pstate;
    ev.avail = nullptr;
    ev.mask = nullptr; ev.act = nullptr;
    ev.ammo = nullptr;                                     /* sims with AmmoAgents run the general kernel */
    FastEnv fe;
    fe.head = bgw_smem + f.o_head;
    fe.rflag = scratch + f.s_rflag;
    fe.cenc = (int8_t *)(bgw_smem + f.o_cenc);
    fe.rel = (uint16_t *)(bgw_smem + f.o_rel);
    fe.act = (uint32_t *)(bgw_smem + f.o_act);
    fe.wsum = (int *)(bgw_smem + f.o_wsum);
    fe.rkmask = (uint32_t *)(scratch + f.s_rkmask);
    fe.eff = (uint16_t *)(scratch + f.s_eff);
    fe.killrank = (uint16_t *)(scratch + f.s_killrank);
    fe.touch = (uint32_t *)(scratch + f.s_touch);
    const double *rw = s.reward;
    const int nch = s.nchunks;

    /* ---- once per CTA: spec tables, learner byte masks, clean dense arrays ------------------------- */
    if ((s.A & 3) == 0) {
        const uint32_t *e32 = (const uint32_t *)s.enc, *k32 = (const uint32_t *)s.klass;
        for (int w = tid; w < (s.A >> 2); w += T) {
            const uint32_t k = __ldg(&k32[w]);
            ((uint32_t *)ev.enc)[w] = __ldg(&e32[w]);
            ((uint32_t *)ev.klass)[w] = k;
        }
    } else {
        for (int a = tid; a < s.A; a += T) {
            const uint8_t k = __ldg(&s.klass[a]);
            ev.enc[a] = __ldg(&s.enc[a]); ev.klass[a] = k;
        }
    }
    /* Tickets: ticket g = block g / E (steps [b S, min((b + 1) S, K))) of env g % E, g < NT.  A CTA draws all its tickets from the launch's counter
     * (arrival order); without a counter (a launch captured into a CUDA graph: one step) CTA c takes c, c + grid, ... */
    uint32_t *const tk = f_in.ticket;                      /* this launch's ticket counter */
    const uint32_t NT = f_in.n_tickets, tbase = f_in.ticket_base;
    int *const tslot = fe.wsum + BGW_TSLOT;
    if (tid == 0) {
        const uint32_t g0 = tk ? atomicAdd(tk, 1u) - tbase : blockIdx.x;
        tslot[0] = (int)min(NT, g0);
        tslot[1] = (int)((g0 < NT) ? min(NT, tk ? atomicAdd(tk, 1u) - tbase : g0 + gridDim.x) : NT);
    }
    if (tid < 16) {
        /* the reference's float64 sum for every combination of what can happen to an entity in a step, term by term in the
         * order it adds them (team_battle_example.py:42,47,46,55,59), rounded to the float32 the reward row holds */
        double r = 0.0;
        if (tid & RF_ATTACK_FAIL) r += rw[BGW_RW_ATTACK_FAIL];
        if (tid & RF_KILL) r += rw[BGW_RW_KILL];
        if (tid & RF_DIED) r += rw[BGW_RW_DIE];
        if (tid & RF_MOVE_FAIL) r += rw[BGW_RW_MOVE_FAIL];
        r += rw[BGW_RW_ENTROPY];
        reinterpret_cast<float *>(fe.wsum + 16)[tid] = (float)r;
    }
    fast_init_dense(s, f, ev, fe, tid, T);
    /* Programmatic dependent launch (step_impl): everything above is env-independent and may run while the previous
     * step launch is still finishing; nothing of the step state is read or written before this point.  The next
     * launch may be scheduled as soon as every CTA of this one is running (its CTAs only become resident as
     * these retire, the grid being the resident set).  A chained launch waits per env instead (above). */
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    if (!f_in.chain) asm volatile("griddepcontrol.wait;" ::: "memory");

    /* (fast_init_dense ended with a barrier: the tickets are visible) */
    const uint32_t S = f_in.block_steps, K = f_in.n_steps;
    uint32_t g = (uint32_t)tslot[0], gn = 0;
    int e = 0, kstep = 0, kend = 0, b = 0;                /* this step, the end of its block (exclusive), the staging buffer */
    bool cont = false;                                     /* not the block's first step: the env's rows are staged in buffer b */
    uint8_t ef_cur = 0, ef_nxt = 0;
    uint32_t step_cur = 0, step_nxt = 0, epi_cur = 0, epi_nxt = 0;
    /* An env's rows may be read once the manager step before has stamped it.  A CTA only ever BLOCKS for the env of its
     * current ticket, with all its earlier tickets finished: the awaited ticket is smaller than every ticket its holder has
     * not finished, so the wait-for relation cannot close a cycle, whatever the number of steps in flight.  For the NEXT
     * ticket (prefetch) a thread merely looks; if the stamp is not there yet it fetches its share of the rows when the
     * ticket becomes current (`late`, per thread: cp.async groups are per thread). */
    bool late = false;
    int kn_carry = 0, en_carry = 0, kend_carry = 0;
    if (g < NT) {
        const uint32_t blk = g / (uint32_t)s.E;
        e = (int)(g - blk * (uint32_t)s.E); kstep = (int)(blk * S); kend = (int)min(blk * S + S, K);
        if (f_in.chain || kstep > 0) env_wait_stamp(f_in, e, f_in.seq + (uint32_t)kstep - 1u);
        fast_issue_env(s, f, st, actions, e, bgw_smem + f.o_buf, tid, T);
        ef_cur = __ldcg(&st.env_flags[e]); step_cur = __ldcg(&st.step[e]); epi_cur = __ldcg(&st.episode[e]);
    }
    cp_async_commit();

    uint32_t epoch = f_in.epoch0;                         /* tag of the next reservation round (ordered rounds, above) */
    int it_no = -1, sl = 1;
    /* end of an env-step.  Inside a block: the env's flags (written by thread 0 next to st.env_flags), step and episode
     * carry over to its next step.  At the block's end: hand the ticket drawn at its last step to the next iteration, and
     * once every thread's stores are behind a barrier, stamp the env (release: the barrier makes the other threads' stores
     * cumulative).  Thread T - 1 stamps: the fence of the release stalls its warp until the env's stores are performed, so
     * the stamp is on the LAST warp, not on the warp that leads the env (measured: five episodes 0.0295 -> 0.0276 ms per
     * step). */
#define BGW_END_ENV()                                                                \
    do {                                                                             \
        if (tid == 0 && last) tslot[sl ^ 1] = (int)tnew;                             \
        __syncthreads();                                                             \
        if (last) {                                                                  \
            BGW_JITTER_POINT(7);                                                     \
            if (tid == T - 1) st_release_u32(f_in.env_seq + e, f_in.seq + (uint32_t)kstep); \
            sl ^= 1; b ^= 1; g = gn; cont = false;                                   \
            kstep = kn_carry; kend = kend_carry; e = en_carry;                       \
            ef_cur = ef_nxt; step_cur = step_nxt; epi_cur = epi_nxt;                 \
        } else {                                                                     \
            ++kstep; cont = true;                                                    \
            ef_cur = (uint8_t)fe.wsum[BGW_EFSLOT]; step_cur = ev.step; epi_cur = ev.episode; \
        }                                                                            \
    } while (0)
    while (g < NT) {
        ++it_no;
        BGW_PROF_MARK(0);
        const bool last = kstep + 1 == kend;                       /* the block's last step: the env leaves the CTA after it */
        if (late) {                                                 /* this ticket's rows were not ready when it was `next` */
            env_wait_stamp(f_in, e, f_in.seq + (uint32_t)kstep - 1u);
            fast_issue_env(s, f, st, actions, e, bgw_smem + f.o_buf + b * f.buf_bytes, tid, T);
            ef_cur = __ldcg(&st.env_flags[e]); step_cur = __ldcg(&st.step[e]); epi_cur = __ldcg(&st.episode[e]);
            cp_async_commit();
            late = false;
        }
        uint32_t tnew = NT;                                         /* the ticket after `gn`: drawn now, needed after the next block */
        if (last) {                                                 /* look at the next ticket as late as possible */
            gn = (uint32_t)tslot[sl];
            BGW_JITTER_POINT(8);
            if (tid == 0 && gn < NT) tnew = min(NT, tk ? atomicAdd(tk, 1u) - tbase : gn + gridDim.x);
            if (gn < NT) {
                const uint32_t bn = gn / (uint32_t)s.E;
                const int kn = (int)(bn * S), en = (int)(gn - bn * (uint32_t)s.E);
                kn_carry = kn; en_carry = en; kend_carry = (int)min(bn * S + S, K);
                if ((f_in.chain || kn > 0) && !env_stamped(f_in, en, f_in.seq + (uint32_t)kn - 1u)) late = true;
                else {
                    fast_issue_env(s, f, st, actions, en, bgw_smem + f.o_buf + (b ^ 1) * f.buf_bytes, tid, T);
                    ef_nxt = __ldcg(&st.env_flags[en]); step_nxt = __ldcg(&st.step[en]); epi_nxt = __ldcg(&st.episode[en]);
                }
            }
        }
        cp_async_commit();                                          /* (an empty group inside a block: wait<1> below stays exact) */

        unsigned char *buf = bgw_smem + f.o_buf + b * f.buf_bytes;
        ev.cell = (uint16_t *)(buf + f.b_cell);
        ev.next = (uint16_t *)(buf + f.b_next);
        ev.flags = buf + f.b_flags;
        ev.health = st.health + (size_t)e * s.A;
        if (!cont)
            for (int i = tid; i < (s.A * 8 + 127) / 128; i += T)   /* hits read health from HBM on demand: warm L2 now */
                asm volatile("prefetch.global.L2 [%0];" ::"l"((const char *)ev.health + (size_t)i * 128));
        ev.e = e; ev.genv = (uint32_t)(s.env_offset + e);
        int8_t *obs_env = obs ? obs + (size_t)e * s.L * s.obs_stride : nullptr;
        float *rew = reward + (size_t)e * s.L;
        uint8_t *dn = done + (size_t)e * s.L;
        const size_t off = (size_t)e * s.A;
        const uint8_t ef0 = ef_cur;
        ev.episode = epi_cur;
        ev.step = step_cur + 1u;
        /* the env's next step runs on this CTA from the rows in shared memory (hold), and from this step's summary grid and
         * occupant lists (hold_lists).  Without auto-reset an env that ends takes no further steps that would store its rows or
         * clear the summary, so those sims store and clear every step; with mixed cells the lists are rebuilt every step
         * (ctr[CTR_MIXED] is set only by the rebuild and by the moves). */
        const bool hold = !last && s.auto_reset, hold_lists = hold && !f.can_mix;

        /* rows of learners that receive nothing this call read as zero; zero counters */
        if ((s.L & 15) == 0) {
            uint4 *d4 = (uint4 *)dn, *r4 = (uint4 *)rew;
            const uint4 z = make_uint4(0, 0, 0, 0);
            for (int i = tid; i < s.L / 16; i += T) d4[i] = z;
            for (int i = tid; i < s.L / 4; i += T) r4[i] = z;
        } else {
            for (int l = tid; l < s.L; l += T) { dn[l] = 0; rew[l] = 0.f; }
        }
        if (tid < CTR_COUNT) ev.ctr[tid] = 0;
        if (epoch < 4096u) {                                        /* (never in practice) the epochs are used up: start over */
            for (int i = tid; i <= s.slot_mask; i += T) ev.slot[i] = BGW_SLOT_FREE;
            epoch = 0xFFFFEu;
        }
        cp_async_wait<1>();
        __syncthreads();
        BGW_PROF_MARK(1);

        bool fresh = false;                                         /* this call resets the env instead of stepping it */
        if (__builtin_expect((ef0 & BGW_ENV_ALL_DONE) != 0, 0)) {     /* cold: once per episode */
            if (!s.auto_reset) {
                if (tid == 0) { all_done[e] = ef0; fe.wsum[BGW_EFSLOT] = ef0; }
                BGW_END_ENV();
                continue;
            }
            /* sim.reset() on this env's staging buffer (general code: placement, health, orientation), state to
             * HBM, then the first observations through the same summary + row-gather path as a step */
            {
                unsigned char *arena = bgw_smem + f.o_cenc;         /* cenc | head | scratch as one arena */
                Env evr = ev;
                evr.head = (uint16_t *)arena;
                evr.racc = (double *)(arena + f.r_racc);
                evr.avail = (uint32_t *)(arena + f.r_avail);
                BgwState st_r = st;
                if constexpr (SHAPE::is_static) st_r.layout = nullptr;   /* (bgw_bind_state moves a handle with caller-supplied layouts to the
                                                                            run-time-shape instantiation: the layout path folds away here) */
                sim_reset(s, st_r, evr, tid, T);
                store_env(s, st, evr, true, tid, T);
                ev.episode = evr.episode; ev.step = evr.step;
            }
            const bool bad = ev.ctr[CTR_ERR] != 0;                   /* (sim_reset ends with a barrier) */
            if (tid == 0) {
                const uint8_t fl = (uint8_t)((bad ? BGW_ENV_ERROR | BGW_ENV_ALL_DONE : 0) | BGW_ENV_RESET);
                st.error[e] = (uint32_t)ev.ctr[CTR_ERR];
                st.env_flags[e] = fl; all_done[e] = fl; fe.wsum[BGW_EFSLOT] = fl;
            }
            __syncthreads();
            fast_init_dense(s, f, ev, fe, tid, T);                  /* the reset arena ran over summary and slots */
            if (tid < CTR_COUNT) ev.ctr[tid] = 0;
            __syncthreads();
            if (bad) {
                /* the placement failed (the reference raises, state.py:147-149,161): an entity without a cell must not be
                 * touched; zero observations, the env stays inert until the next reset */
                if (obs_env)
                    for (int i = tid; i < s.L * nch; i += T) reinterpret_cast<uint4 *>(obs_env)[i] = make_uint4(0, 0, 0, 0);
                BGW_END_ENV();
                continue;
            }
            fresh = true;
        }
        BGW_PROF_MARK(2);

        /* ---- relevant entities and acting learners, both compacted in entity order ------------------ */
        int n_rel = 0, n_act = 0;
        if (f.simd_ok) {
            if (warp == 0) {
                const uint32_t *fw = (const uint32_t *)ev.flags, *kw = (const uint32_t *)ev.klass;
                const int nwords = s.A >> 2, wpl = (nwords + 31) >> 5;
                int cnt = 0;
                for (int j = 0; j < wpl; ++j) {
                    const int w = lane * wpl + j;
                    if (w < nwords) {
                        const uint32_t x = fw[w];
                        const uint32_t rel = ~__vcmpeq4(x & 0x07070707u, 0x04040404u);      /* not (dead, removed, reported) */
                        const uint32_t act = __vcmpne4(kw[w] & (0x01010101u * BGW_AG_LEARNER), 0u) & __vcmpeq4(x & 0x04040404u, 0u);   /* learner, not reported */
                        cnt += (__popc(rel) >> 3) + ((__popc(act) >> 3) << 16);
                    }
                }
                int incl = cnt;
#pragma unroll
                for (int dd = 1; dd < 32; dd <<= 1) { const int t = __shfl_up_sync(0xFFFFFFFFu, incl, dd); if (lane >= dd) incl += t; }
                int pr = (incl - cnt) & 0xFFFF, pa = (incl - cnt) >> 16;
                /* Acting learners are relevant, so equal counts mean equal lists: when every entity is a learner that is the
                 * rule (an entity leaves both when its death has been reported; the exception is one that was reported while
                 * still on the grid, e.g. placed with zero health).  Then ONE list is written and serves as both -- half the
                 * stores, and half the code of this unrolled loop on the env's critical path. */
                const int tot = __shfl_sync(0xFFFFFFFFu, incl, 31);
                const bool same = f.identity_learners && (tot & 0xFFFF) == (tot >> 16);
                if (same) {
                    for (int j = 0; j < wpl; ++j) {
                        const int w = lane * wpl + j;
                        if (w < nwords) {
                            const uint32_t act = __vcmpeq4(fw[w] & 0x04040404u, 0u);      /* (every entity is a learner) not reported */
#pragma unroll
                            for (int bb = 0; bb < 4; ++bb)
                                if ((act >> (8 * bb)) & 1u) ev.ragent[pa++] = (uint16_t)(4 * w + bb);
                        }
                    }
                } else {
#pragma unroll 1
                    for (int j = 0; j < wpl; ++j) {
                        const int w = lane * wpl + j;
                        if (w < nwords) {
                            const uint32_t x = fw[w];
                            const uint32_t rel = ~__vcmpeq4(x & 0x07070707u, 0x04040404u);
                            const uint32_t act = __vcmpne4(kw[w] & (0x01010101u * BGW_AG_LEARNER), 0u) & __vcmpeq4(x & 0x04040404u, 0u);
#pragma unroll 1
                            for (int bb = 0; bb < 4; ++bb) {
                                const int a = 4 * w + bb;
                                if ((rel >> (8 * bb)) & 1u) fe.rel[pr++] = (uint16_t)a;
                                if ((act >> (8 * bb)) & 1u) ev.ragent[pa++] = (uint16_t)a;
                            }
                        }
                    }
                }
                if (lane == 31) fe.wsum[3] = same;
                if (lane == 31) { fe.wsum[0] = incl & 0xFFFF; fe.wsum[1] = incl >> 16; }
            }
            __syncthreads();
            n_rel = fe.wsum[0]; n_act = fe.wsum[1];
            fe.rel = fe.wsum[3] ? ev.ragent : (uint16_t *)(bgw_smem + f.o_rel);   /* one list serves as both (above) */
        } else {
            for (int a0 = 0; a0 < s.A; a0 += T) {
                const int a = a0 + tid;
                bool rel = false, acting = false;
                if (a < s.A) {
                    const uint8_t fl = ev.flags[a];
                    rel = (fl & (BGW_ST_ACTIVE | BGW_ST_IN_GRID)) || !(fl & BGW_ST_DONE_REPORTED);
                    acting = (ev.klass[a] & BGW_AG_LEARNER) && !(fl & BGW_ST_DONE_REPORTED);
                }
                const unsigned br = __ballot_sync(0xFFFFFFFFu, rel), ba = __ballot_sync(0xFFFFFFFFu, acting);
                if (lane == 0) { fe.wsum[2 + warp] = __popc(br); fe.wsum[8 + warp] = __popc(ba); }
                __syncthreads();
                int before_r = n_rel, before_a = n_act;
                for (int w = 0; w < nwarp; ++w) {
                    const int cr = fe.wsum[2 + w], ca = fe.wsum[8 + w];
                    if (w < warp) { before_r += cr; before_a += ca; }
                    n_rel += cr; n_act += ca;
                }
                const unsigned lt = (1u << lane) - 1u;
                if (rel) fe.rel[before_r + __popc(br & lt)] = (uint16_t)a;
                if (acting) ev.ragent[before_a + __popc(ba & lt)] = (uint16_t)a;
                __syncthreads();
            }
        }
        if (order) {                                               /* all_step_manager.py:62-65: caller-given order */
            n_act = 0;
            for (int i0 = 0; i0 < s.L; i0 += T) {
                const int i = i0 + tid;
                int a = 0;
                bool acting = false;
                if (i < s.L) {
                    a = __ldg(&s.agent_of[order[(size_t)e * s.L + i]]);
                    acting = !(ev.flags[a] & BGW_ST_DONE_REPORTED);
                }
                __syncthreads();                                    /* wsum / ragent of the previous pass are consumed */
                const unsigned ba = __ballot_sync(0xFFFFFFFFu, acting);
                if (lane == 0) fe.wsum[2 + warp] = __popc(ba);
                __syncthreads();
                int before = n_act;
                for (int w = 0; w < nwarp; ++w) { const int c = fe.wsum[2 + w]; if (w < warp) before += c; n_act += c; }
                if (acting) ev.ragent[before + __popc(ba & ((1u << lane) - 1u))] = (uint16_t)a;
            }
            __syncthreads();
        }
        BGW_PROF_MARK(3);

        fast_build_lists<HT>(s, f, ev, fe, n_rel, cont && !fresh && s.auto_reset && !f.can_mix, tid, T);   /* (the step before held them) */
        BGW_PROF_MARK(4);

        if (fresh) {
            for (int i = tid; i < n_act; i += T) ev.plist[i] = f.identity_learners ? ev.ragent[i] : (uint16_t)__ldg(&s.learner_of[ev.ragent[i]]);
            /* the observation gather below reads entries other threads wrote (with every entity a learner, plist is ragent,
             * which the compaction's barrier published) */
            if (!f.identity_learners) __syncthreads();
        } else {
            fast_attack_prepass(s, f, ev, fe, actions, sampled, n_act, epoch, tid, T);
            BGW_PROF_MARK(5);
            epoch = fast_attack_phase<HT>(s, f, ev, fe, epoch, lane, warp, T);
            BGW_PROF_MARK(6);

            /* ---- settle attackers without candidates; classify the moves :50-55 --------------------------- */
            int pend = 0;
            for (int i = tid; i < n_act; i += T) {
                const int a = ev.ragent[i];
                const bool active = ev.flags[a] & BGW_ST_ACTIVE;
                if (ev.pstate[i] == 3) {
                    const unsigned kr = fe.killrank[a];
                    if (active || (kr != BGW_NONE16 && kr > (unsigned)i)) fe.rflag[a] |= RF_ATTACK_FAIL;   /* :41-42 */
                }
                uint32_t ft = BGW_NO_MOVE;                          /* (source << 16 | destination) of a pending move */
                if (active) {
                    bool ok = false;
                    if (ev.klass[a] & BGW_AG_MOVING) {
                        int dr, dc, r0, c0;
                        const int from = ev.cell[a];
                        decode_move(s, a, fe.act[ev.plist[i]], dr, dc);
                        cell_rc(s, f, from, r0, c0);
                        const int r = r0 + dr, c = c0 + dc;
                        if (r >= 0 && r < s.H && c >= 0 && c < s.W) {
                            if (dr == 0 && dc == 0) ok = true;
                            else ft = ((uint32_t)from << 16) | (uint32_t)(r * s.W + c);
                        }
                    }
                    if (ft == BGW_NO_MOVE && !ok) fe.rflag[a] |= RF_MOVE_FAIL;
                }
                fe.rkmask[i] = ft;
                if (ft != BGW_NO_MOVE) {                            /* name the two cells of the move (fast_move_phase) */
                    touch_mark(f, fe, (int)(ft >> 16));
                    touch_mark(f, fe, (int)(ft & 0xFFFFu));
                    pend = 1;
                }
            }
            pend = __syncthreads_or(pend);
            BGW_PROF_MARK(7);
            if (pend) epoch = fast_move_phase<HT>(s, f, ev, fe, n_act, epoch, tid, T);
            BGW_PROF_MARK(8);

            /* ---- entropy :58-59, rewards / dones of the acting learners (all_step_manager.py:68-87) -------- */
            for (int i = tid; i < n_act; i += T) {
                const int a = ev.ragent[i], l = ev.plist[i];
                const unsigned rf = fe.rflag[a];                     /* (table built once per CTA, above) */
                const bool dd = prog_done(s, ev, a);
                rew[l] = reinterpret_cast<const float *>(fe.wsum + 16)[rf & 15u];
                dn[l] = (uint8_t)(BGW_OUT_VALID | (dd ? BGW_OUT_DONE : 0));
                if (dd) ev.flags[a] |= BGW_ST_DONE_REPORTED; else atomicAdd(&ev.ctr[CTR_REMAINING], 1);
            }
        }
        /* entities whose accumulator persists (non-learners with health, never read): add this step's 'die' in HBM */
        if (!fresh)
            for (int x = tid; x < n_rel; x += T) {
                const int a = fe.rel[x];
                if (racc_persists(ev.klass[a]) && (fe.rflag[a] & RF_DIED)) st.reward_acc[off + a] = __ldcg(&st.reward_acc[off + a]) + rw[BGW_RW_DIE];
            }
        BGW_PROF_MARK(9);

        /* ---- observations ------------------------------------------------------------------------------ */
        if (obs_env) {
            const bool direct = s.observe_self && !(f.can_mix && ev.ctr[CTR_MIXED]);
            const int R = direct ? f.uniform_view : -1;
            switch (R) {
            case 1: fast_obs_rows<1>(s, f, ev, fe, n_act, obs_env, tid, T); break;
            case 2: fast_obs_rows<2>(s, f, ev, fe, n_act, obs_env, tid, T); break;
            case 3: fast_obs_rows<3>(s, f, ev, fe, n_act, obs_env, tid, T); break;
            case 4: fast_obs_rows<4>(s, f, ev, fe, n_act, obs_env, tid, T); break;
            case 5: fast_obs_rows<5>(s, f, ev, fe, n_act, obs_env, tid, T); break;
            default: {
                const int items = n_act * nch;
                for (int it = tid; it < items; it += T) {
                    const int li = it / nch, ch = it - li * nch;
                    const int l = ev.plist[li], a = ev.ragent[li];
                    uint32_t w[4];
                    fast_obs_chunk_slow<HT>(s, f, ev, fe, a, ch, w);
                    *reinterpret_cast<uint4 *>(obs_env + (size_t)l * s.obs_stride + ch * 16) = make_uint4(w[0], w[1], w[2], w[3]);
                }
            }
            }
        }
        __syncthreads();
        BGW_PROF_MARK(10);

        /* ---- store the relevant entities, get_all_done (done.py:49-56,147-153), clean the dense arrays ---- */
        {
            uint32_t lo = 0, hi = 0;
            int ok = 1;
            for (int x = tid; x < n_rel; x += T) {
                const int a = fe.rel[x];
                const uint8_t fl = ev.flags[a];
                /* held rows are stored at the block's end, except those of an entity that leaves the relevant set now (dead,
                 * removed and reported: the compaction's test), which no later step of the block visits */
                if (!fresh && (!hold || (fl & 7) == BGW_ST_DONE_REPORTED)) { st.cell[off + a] = ev.cell[a]; st.next[off + a] = ev.next[a]; st.flags[off + a] = fl; }
                if (fl & BGW_ST_ACTIVE) { const int en2 = ev.enc[a]; if (en2 < 32) lo |= 1u << en2; else hi |= 1u << (en2 - 32); }
                if (s.done_mask & (BGW_DONE_TARGET_AGENT | BGW_DONE_TARGET_DESTROYED)) {
                    const int t = __ldg(&s.target[a]);
                    if ((s.done_mask & BGW_DONE_TARGET_AGENT) && t >= 0 && !same_position(ev, a, t)) ok = 0;
                    if ((s.done_mask & BGW_DONE_TARGET_DESTROYED) && t >= 0 && (ev.flags[t] & BGW_ST_ACTIVE)) ok = 0;
                }
                if ((fl & BGW_ST_IN_GRID) && !hold_lists) fe.cenc[pad_index(s, f, ev.cell[a])] = 0;
            }
            lo = __reduce_or_sync(0xFFFFFFFFu, lo);
            hi = __reduce_or_sync(0xFFFFFFFFu, hi);
            ok = __all_sync(0xFFFFFFFFu, ok);
            if (lane == 0) {
                if (lo) atomicOr((unsigned *)&ev.ctr[CTR_ENC_LO], lo);
                if (hi) atomicOr((unsigned *)&ev.ctr[CTR_ENC_HI], hi);
                if (!ok) atomicOr((unsigned *)&ev.ctr[CTR_AND], 1u);   /* here: 1 = some target condition unmet */
            }
        }
        __syncthreads();
        if (tid == 0 && !fresh) {
            const unsigned long long encs = ((unsigned long long)(unsigned)ev.ctr[CTR_ENC_HI] << 32) | (unsigned)ev.ctr[CTR_ENC_LO];
            int d = !ev.ctr[CTR_AND];
            if (s.done_mask & BGW_DONE_ACTIVE) d &= (encs == 0);
            if (s.done_mask & BGW_DONE_ONE_TEAM) d &= ((encs & (encs - 1)) == 0);
            uint8_t ef = 0;
            if (d || ev.ctr[CTR_REMAINING] == 0) ef |= BGW_ENV_ALL_DONE;            /* all_step_manager.py:90-93 */
            if (s.horizon > 0 && (int)ev.step >= s.horizon) ef |= BGW_ENV_ALL_DONE | BGW_ENV_TRUNCATED;
            st.step[e] = ev.step;
            st.env_flags[e] = ef;
            all_done[e] = ef;
            fe.wsum[BGW_EFSLOT] = ef;
            unsigned long long *sr = (unsigned long long *)st.stats + (size_t)e * BGW_STAT_COUNT;
            /* reductions without a return value (the row belongs to this env: no contention): thread 0, which every
             * other thread of the CTA is about to wait for, does not sit out an L2 round trip */
            atomicAdd(&sr[BGW_STAT_AGENT_STEPS], (unsigned long long)n_act);
            atomicAdd(&sr[BGW_STAT_ENV_STEPS], 1ull);
            if (ev.ctr[CTR_KILLS]) atomicAdd(&sr[BGW_STAT_KILLS], (unsigned long long)ev.ctr[CTR_KILLS]);
            if (ef & BGW_ENV_ALL_DONE) atomicAdd(&sr[BGW_STAT_EPISODES], 1ull);
        }
        BGW_END_ENV();                                              /* ctr, scratch and the staging buffer are rewritten next */
        BGW_PROF_MARK(11);
    }
#undef BGW_END_ENV
    cp_async_wait<0>();
}

/* the stock instantiations (bgw_fastk.cu); a run-time compilation for one spec's shape (bgw_specialize, bgw_jit.h) wraps the
 * same body, with a shape struct of its own, in a kernel of its own */
template <typename SHAPE, typename HT>
__global__ void BGW_FAST_LB bgw_step_fast_kernel(const DevSpec s_in, const FastSpec f_in, const BgwState st, const uint32_t *actions,
                                     uint32_t *sampled, const int16_t *order, int8_t *obs, float *reward, uint8_t *done,
                                     uint8_t *all_done)
{
    bgw_step_fast_body<SHAPE, HT>(s_in, f_in, st, actions, sampled, order, obs, reward, done, all_done);
}

#ifdef BGW_SMALL_KERNELS
/* ------------------------------------------------------------------------------------------------- */
/* The observer on its own (bgw_observe): PositionCenteredEncodingObserver.get_obs observer.py:195-248  */
/* ------------------------------------------------------------------------------------------------- */
/* For the sims of the specialised kernel whose cells never hold two different encodings (FastSpec.can_mix == 0) and whose
 * learners share one view range.  Persistent CTAs; per env: the entities' cells and flags are read from HBM (3 bytes each),
 * their encodings scattered into the padded summary grid in shared memory, every learner's window gathered by
 * fast_obs_rows (the step kernel's gather: 256-bit stores), the scattered cells cleared again.  128 bytes written per
 * 3 read: the HBM-bound piece of the path (SURVEY.md 8(d): "K3"). */
struct ObserveLayout { int o_cell, o_flags, o_klass, o_enc, o_ragent, o_plist, bytes; };
inline __host__ __device__ ObserveLayout observe_layout(int A, int L, int PH, int PW)
{
    ObserveLayout o;
    int off = (PH * PW + 32 + 15) & ~15;             /* summary grid + the slack words the row gather reads */
    o.o_cell = off;   off += ((A + 7) & ~7) * 2;
    o.o_ragent = off; off += ((L + 7) & ~7) * 2;
    o.o_plist = off;  off += ((L + 7) & ~7) * 2;
    o.o_flags = off;  off += (A + 15) & ~15;
    o.o_klass = off;  off += (A + 15) & ~15;
    o.o_enc = off;    off += (A + 15) & ~15;
    o.bytes = off;
    return o;
}

template <int R>
__global__ void __launch_bounds__(128) bgw_observe_fast_kernel(const DevSpec s, const FastSpec f, const BgwState st, const uint8_t *env_mask,
                                                               int8_t *obs)
{
    const int tid = threadIdx.x, T = blockDim.x;
    const ObserveLayout lay = observe_layout(s.A, s.L, f.PH, f.PW);
    Env ev;
    FastEnv fe;
    fe.cenc = (int8_t *)bgw_smem;
    ev.cell = (uint16_t *)(bgw_smem + lay.o_cell);
    ev.ragent = (uint16_t *)(bgw_smem + lay.o_ragent);
    ev.plist = (uint16_t *)(bgw_smem + lay.o_plist);
    ev.flags = bgw_smem + lay.o_flags;
    ev.klass = bgw_smem + lay.o_klass;
    ev.enc = (int8_t *)(bgw_smem + lay.o_enc);
    {   /* once per CTA: the empty summary with its -1 border (as fast_init_dense), the per-entity constants */
        uint32_t *c32 = (uint32_t *)fe.cenc;
        const int wpr = f.PW >> 2;
        /* a thread keeps its column word (one division per CTA); rows_per_pass rows are written side by side.  A row with
         * more words than the CTA has threads is walked by all threads, one row at a time. */
        const int rows_per_pass = wpr <= T ? T / wpr : 1;
        const int r0 = wpr <= T ? tid / wpr : 0;
        for (int cw = wpr <= T ? tid - r0 * wpr : tid; cw < wpr && r0 < rows_per_pass; cw += T) {
            uint32_t inner = 0xFFFFFFFFu;
            for (int bb = 0; bb < 4; ++bb) {
                const int cc = cw * 4 + bb;
                if (cc >= f.PL && cc < f.PL + s.W) inner &= ~(0xFFu << (8 * bb));
            }
            for (int rr = r0; rr < f.PH; rr += rows_per_pass) c32[rr * wpr + cw] = (rr >= f.P && rr < f.P + s.H) ? inner : 0xFFFFFFFFu;
        }
        if (tid < 8) c32[f.PH * wpr + tid] = 0xFFFFFFFFu;           /* slack words read by the row gather */
        for (int a = tid; a < s.A; a += T) { ev.klass[a] = __ldg(&s.klass[a]); ev.enc[a] = __ldg(&s.enc[a]); }
        for (int l = tid; l < s.L; l += T) { ev.ragent[l] = (uint16_t)__ldg(&s.agent_of[l]); ev.plist[l] = (uint16_t)l; }
    }
    __syncthreads();
    for (int e = blockIdx.x; e < s.E; e += gridDim.x) {
        if (env_mask && !env_mask[e]) continue;
        const size_t off = (size_t)e * s.A;
        for (int a = tid; a < s.A; a += T) {
            const uint16_t c = __ldcs(&st.cell[off + a]);
            const uint8_t fl = __ldcs(&st.flags[off + a]);
            ev.cell[a] = c; ev.flags[a] = fl;
            if (fl & BGW_ST_IN_GRID) fe.cenc[pad_index(s, f, c)] = ev.enc[a];   /* same encoding from every occupant of a cell */
        }
        __syncthreads();
        fast_obs_rows<R>(s, f, ev, fe, s.L, obs + (size_t)e * s.L * s.obs_stride, tid, T);
        __syncthreads();
        for (int a = tid; a < s.A; a += T)
            if (ev.flags[a] & BGW_ST_IN_GRID) fe.cenc[pad_index(s, f, ev.cell[a])] = 0;
        __syncthreads();
    }
}
#endif  /* BGW_SMALL_KERNELS */

