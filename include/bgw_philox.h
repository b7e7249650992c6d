/*
 * bgw_philox.h -- counter-based Philox4x32-10 stream shared by the CUDA engine, the C-ABI host
 * entry point bgw_rng_draw(), and the CPU oracle (oracle/bgw_oracle.c).
 *
 * The reference (Abmarl 0.2.7) draws from ONE global numpy MT19937 stream in call order
 * (draw sites: state.py:159,641,675; actor.py:388,412; observer.py:131,234,246 -- see SURVEY.md
 * section 8(a) "RNG draw sites").  A lockstep batch of independent envs cannot share a stream, so
 * every stochastic outcome here is a pure function of the key
 *
 *     (seed, env, episode, step, site, slot, k)
 *
 * and the SAME draws are replayed INTO the unmodified reference by tests/refshim (it patches
 * numpy.random.{uniform,choice,randint} to return these values), which is what makes bit-exact
 * parity checkable.
 *
 *   key     = (seed_lo, seed_hi)
 *   counter = (env, episode, step, site<<28 | slot<<16 | k)       slot < 4096, k < 65536
 *
 * Mapping of a draw to the reference's value:
 *   uniform()          u = x0 * 2^-32            (float64, in [0,1))
 *   choice over n      index = (x0 * n) >> 32    (== floor(u*n), exact integer arithmetic)
 *   randint(lo, hi)    lo + ((x0 * (hi-lo)) >> 32)
 */
#ifndef BGW_PHILOX_H_
#define BGW_PHILOX_H_

#include "bgw_stdint.h"

#if defined(__CUDACC__)
#define BGW_HD __host__ __device__ __forceinline__
#else
#define BGW_HD static inline
#endif

/* draw sites */
enum {
    BGW_SITE_PLACE = 0,   /* PositionState._place_variable_position_agent   state.py:159  slot=agent k=0 */
    BGW_SITE_HEALTH = 1,  /* HealthState.reset                                state.py:641  slot=agent k=0 */
    BGW_SITE_ORIENT = 2,  /* OrientationState.reset                           state.py:675  slot=agent k=0 */
    BGW_SITE_ACC = 3,     /* AttackActorBaseComponent._basic_criteria         actor.py:388  slot=attacker
                             k = candidate + 4096 * (how often this step the pair was evaluated before; only the
                             RestrictedSelectiveAttackActor evaluates a pair more than once) */
    BGW_SITE_SUBSET = 4,  /* _subset_attackables actor.py:412 and RestrictedSelectiveAttackActor's choice :655
                             slot=attacker  k = group << 8 | draw#;  group = 0 (Binary), the encoding (EncodingBased),
                             window cell r*n+c (Selective), number of agents attacked so far (RestrictedSelective) */
    BGW_SITE_OBS = 5,     /* observers' np.random.choice            observer.py:131,234,246 slot=observer k=absolute cell */
    BGW_SITE_ACTION = 6,  /* synthetic random policy (bench / tests)          policies/policy.py:81-92 slot=agent */
    BGW_SITE_MAZE = 7,    /* MazePlacementState                               state.py:529, utils.py:193,198 */
    BGW_SITE_AMMO = 8,    /* ammo filter of process_action                    actor.py:346-350 slot=attacker k=draw# */
    BGW_SITE_SCRIPT = 9,  /* PacmanSimSimple's random baddie move             examples/sim/pacman.py:240 slot=baddie k=0 */
    /* random.shuffle (Python's own generator, not numpy's): the KEYED ORDER of a list of entities sorts them by
     * (first Philox word of the entity's key, entity index) -- a uniformly random permutation that does not depend on
     * the order the list had, and whose restriction to a sub-list is the keyed order of the sub-list */
    BGW_SITE_ORDER = 10,       /* AllStepManager(randomize_action_input) managers/all_step_manager.py:62-65 slot=agent k=0,
                                  step = the manager step that is being taken */
    BGW_SITE_PLACE_ORDER = 11, /* PositionState(randomize_placement_order)      state.py:97-101 slot=agent k=0, step 0 */
    BGW_SITE_PROGRAM = 12      /* bgwp_uniform of a user step program (bgw_program.h)   slot, k: the program's choice */
};

BGW_HD void bgw_philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                              uint32_t k0, uint32_t k1, uint32_t out[4])
{
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#if defined(__CUDACC__)
#pragma unroll
#endif
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)M0 * c0;
        uint64_t p1 = (uint64_t)M1 * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

BGW_HD void bgw_draw4(uint64_t seed, uint32_t env, uint32_t episode, uint32_t step,
                      uint32_t site, uint32_t slot, uint32_t k, uint32_t out[4])
{
    bgw_philox4x32_10(env, episode, step, (site << 28) | ((slot & 0xFFFu) << 16) | (k & 0xFFFFu),
                      (uint32_t)seed, (uint32_t)(seed >> 32), out);
}

/* first word only */
BGW_HD uint32_t bgw_draw(uint64_t seed, uint32_t env, uint32_t episode, uint32_t step,
                         uint32_t site, uint32_t slot, uint32_t k)
{
    uint32_t o[4];
    bgw_draw4(seed, env, episode, step, site, slot, k, o);
    return o[0];
}

/* uniform in [0,1): exactly representable in float64 */
BGW_HD double bgw_u01(uint32_t x) { return (double)x * (1.0 / 4294967296.0); }
/* index in [0,n) == floor(u01(x)*n) */
BGW_HD uint32_t bgw_index(uint32_t x, uint32_t n) { return (uint32_t)(((uint64_t)x * n) >> 32); }

#endif /* BGW_PHILOX_H_ */
