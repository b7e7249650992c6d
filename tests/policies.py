"""Structured policies for the parity tests, and measurements that show what they reach.

The keyed random policy (sample_actions) scatters uniform actions over a sparse board: on the headline shape its longest
chain of moves into cells vacated earlier in the same step is 2, and it rarely puts more than a few entities in one cell.
Trained policies herd, follow each other and gang up, and those are the inputs the kernels' ordered reservation rounds,
touch bit maps, hashed slot tables and occupant lists exist for.  Each policy here is a deterministic numpy function of
(spec, state, t, rng) that returns int8 actions [E, L, action_stride] in the layout of include/bgw.h (bgw_step), inside
the reference's action spaces; `state` is in the oracle's layout (OracleEnv.state, BatchedGridWorld.state_numpy()).
Rows of learners already reported done are zero.
"""
import numpy as np

from abmarl_b200 import _capi as K
from tests.kat_cases import make_spec, OBS, MOV, ATT, HEA, LRN

CROSS_DR = np.array([0, 0, 1, 0, -1])          # CrossMoveActor: 0 stay, 1 left, 2 down, 3 right, 4 up
CROSS_DC = np.array([0, -1, 0, 1, 0])
DIRS8 = np.array([(-1, -1), (-1, 0), (-1, 1), (0, 1), (1, 1), (1, 0), (1, -1), (0, -1)])
DIRS4 = np.array([(-1, 0), (0, 1), (1, 0), (0, -1)])


# ---------------------------------------------------------------------------------------------------
# layout helpers
# ---------------------------------------------------------------------------------------------------
def action_stride(spec):
    """bytes of one learner's action row: 2 move bytes + the widest attack action, rounded up to 4 (bgw.h, bgw_step)"""
    w = 1
    for a in range(spec.n_agents):
        if not spec.klass[a] & K.AG_ATTACKING:
            continue
        n = 2 * int(spec.attack_range[a]) + 1
        w = max(w, {K.ATTACK_ENCODING: spec.max_encoding, K.ATTACK_RESTRICTED: int(spec.simultaneous_attacks[a]),
                    K.ATTACK_SELECTIVE: n * n}.get(int(spec.attack_actor), 1))
    return (2 + w + 3) // 4 * 4


def learners(spec):
    return np.array(spec.learner_agents, dtype=np.int64)


def cells(spec, state):
    """row, col [E, A] of every entity in the grid, -1 for the others"""
    cell = state['cell'].astype(np.int64)
    ing = ((state['flags'] & K.ST_IN_GRID) != 0) & (cell != K.BGW_NONE)
    return np.where(ing, cell // spec.cols, -1), np.where(ing, cell % spec.cols, -1)


def occupancy(spec, state):
    """[E, max_encoding + 1, rows, cols]: active entities in the grid per cell and encoding"""
    r, c = cells(spec, state)
    E = r.shape[0]
    occ = np.zeros((E, spec.max_encoding + 1, spec.rows, spec.cols), dtype=np.int32)
    e, a = np.nonzero((r >= 0) & ((state['flags'] & K.ST_ACTIVE) != 0))
    np.add.at(occ, (e, spec.encoding[a].astype(np.int64), r[e, a], c[e, a]), 1)
    return occ


def blank(spec, state):
    return np.zeros((state['cell'].shape[0], spec.n_learners, action_stride(spec)), dtype=np.int8)


def finish(spec, state, act):
    """zero the rows of learners already reported done (bgw_step ignores them; the reference never receives them)"""
    act[(state['flags'][:, learners(spec)] & K.ST_DONE_REPORTED) != 0] = 0
    return act


def set_moves(spec, act, dr, dc):
    """Moves (dr, dc) [E, L] clipped to each learner's move range, in the spec's move action: the box (or its ravelled
    index) or the cross actor's 0..4 (the larger component wins, rows before columns)."""
    lrn = learners(spec)
    m = spec.move_range[lrn].astype(np.int64)
    moving = (spec.klass[lrn] & K.AG_MOVING) != 0
    dr = np.where(moving, np.clip(dr, -m, m), 0)
    dc = np.where(moving, np.clip(dc, -m, m), 0)
    if spec.move_actor == K.MOVE_BOX:
        if spec.ravel_actions:
            act[..., 0] = ((dr + m) * (2 * m + 1) + dc + m).astype(np.uint8).view(np.int8)
        else:
            act[..., 0], act[..., 1] = dr, dc
    elif spec.move_actor == K.MOVE_CROSS:
        vert = (np.abs(dr) >= np.abs(dc)) & (dr != 0)
        act[..., 0] = np.where(vert, np.where(dr > 0, 2, 4), np.where(dc > 0, 3, np.where(dc < 0, 1, 0)))
    return act


def toward(spec, state, gr, gc):
    """(dr, dc) [E, L] from each learner's cell toward the goal cells gr, gc (broadcast to [E, L]); 0 off the grid"""
    r, c = cells(spec, state)
    lrn = learners(spec)
    r, c = r[:, lrn], c[:, lrn]
    off = r < 0
    return np.where(off, 0, gr - r), np.where(off, 0, gc - c)


def enemies_of(spec):
    """[L, max_encoding + 1] bool: learner l may attack encoding e"""
    enc = spec.encoding[learners(spec)].astype(np.int64)
    bits = np.arange(spec.max_encoding + 1, dtype=np.uint64)
    return ((spec.attack_map[enc][:, None] >> bits[None, :]) & np.uint64(1)).astype(bool)


def best_window_cell(spec, state):
    """[E, L]: index r * n + c of the cell of each learner's attack window (n = 2 * attack_range + 1) that holds the most
    enemies (the first in row-major order among equals; the centre when the window holds none)"""
    occ = occupancy(spec, state)
    foe = np.einsum('eihw,li->elhw', occ, enemies_of(spec).astype(np.int32))
    r, c = cells(spec, state)
    lrn = learners(spec)
    E, L = r.shape[0], len(lrn)
    best = np.zeros((E, L), dtype=np.int64)
    for l, a in enumerate(lrn):
        R = int(spec.attack_range[a])
        n = 2 * R + 1
        counts = np.zeros((E, n * n), dtype=np.int32)
        for k in range(n * n):
            gr, gc = r[:, a] - R + k // n, c[:, a] - R + k % n
            ok = (r[:, a] >= 0) & (gr >= 0) & (gr < spec.rows) & (gc >= 0) & (gc < spec.cols)
            counts[ok, k] = foe[np.nonzero(ok)[0], l, gr[ok], gc[ok]]
        best[:, l] = np.where(counts.max(axis=1) > 0, counts.argmax(axis=1), R * n + R)
    return best


def max_attack(spec, state, act):
    """Every attacking learner attacks at the maximum of its attack action: Binary byte 2 = simultaneous_attacks;
    EncodingBased every attackable encoding at simultaneous_attacks; Selective all attacks on the window cell holding the
    most enemies; RestrictedSelective that cell named simultaneous_attacks times."""
    lrn = learners(spec)
    att = (spec.klass[lrn] & K.AG_ATTACKING) != 0
    sim = np.where(att, spec.simultaneous_attacks[lrn].astype(np.int64), 0)
    kind = int(spec.attack_actor)
    if kind == K.ATTACK_BINARY:
        act[..., 2] = sim
    elif kind == K.ATTACK_ENCODING:
        foe = enemies_of(spec)
        for e in range(1, spec.max_encoding + 1):
            act[..., 2 + e - 1] = np.where(foe[:, e], sim, 0)
    elif kind in (K.ATTACK_SELECTIVE, K.ATTACK_RESTRICTED):
        best = best_window_cell(spec, state)
        for l, a in enumerate(lrn):
            if not att[l]:
                continue
            n = 2 * int(spec.attack_range[a]) + 1
            if kind == K.ATTACK_SELECTIVE:
                act[np.arange(act.shape[0]), l, 2 + best[:, l]] = sim[l]
            else:                                  # the ravelled index counts rows fastest (actor.py:641-643)
                act[:, l, 2:2 + sim[l]] = ((best[:, l] % n) * n + best[:, l] // n + 1)[:, None]
    return act


# ---------------------------------------------------------------------------------------------------
# the policies
# ---------------------------------------------------------------------------------------------------
def convoy(dr=0, dc=1):
    """every learner moves by (dr, dc) every step (for formations built with fixed positions)"""
    def policy(spec, state, t, rng):
        act = blank(spec, state)
        shape = act.shape[:2]
        return finish(spec, state, set_moves(spec, act, np.full(shape, dr), np.full(shape, dc)))
    return policy


def corners(spec):
    return [(0, 0), (0, spec.cols - 1), (spec.rows - 1, 0), (spec.rows - 1, spec.cols - 1)]


class Rendezvous:
    """Each team (encoding e) walks to its own corner, corners(spec)[(e - 1) % 4]; a learner away from its goal that did
    not move in the last step takes a random step drawn from `rng` instead (a fresh draw for every learner every step,
    so the stream does not depend on who is stuck).  `attack`: max_attack on top."""

    def __init__(self, attack=False):
        self.attack, self.last = attack, None

    def __call__(self, spec, state, t, rng):
        lrn = learners(spec)
        goal = np.array(corners(spec))[(spec.encoding[lrn].astype(np.int64) - 1) % 4]
        dr, dc = toward(spec, state, goal[:, 0], goal[:, 1])
        act = blank(spec, state)
        jit = rng.integers(-2, 3, size=(2,) + act.shape[:2])
        cell = state['cell'][:, lrn].copy()
        if self.last is not None and self.last.shape == cell.shape:
            stuck = (cell == self.last) & ((dr != 0) | (dc != 0))
            dr, dc = np.where(stuck, jit[0], dr), np.where(stuck, jit[1], dc)
        self.last = cell
        set_moves(spec, act, dr, dc)
        if self.attack:
            max_attack(spec, state, act)
        return finish(spec, state, act)


def disperse(spec, state, t, rng):
    """every learner steps away by its full move range in the direction its index names: the 8 neighbours of the box
    actor or the 4 of the cross actor in turn.  From a pile every mover names the same source cell."""
    act = blank(spec, state)
    L = act.shape[1]
    dirs = DIRS8 if spec.move_actor == K.MOVE_BOX else DIRS4
    d = dirs[np.arange(L) % len(dirs)] * spec.move_range[learners(spec)][:, None].astype(np.int64)
    return finish(spec, state, set_moves(spec, act, np.broadcast_to(d[:, 0], act.shape[:2]), np.broadcast_to(d[:, 1], act.shape[:2])))


def melee(goal=None):
    """every team heads for one common cell (default: the centre) and attacks at the maximum every step"""
    def policy(spec, state, t, rng):
        gr, gc = goal if goal is not None else (spec.rows // 2, spec.cols // 2)
        act = blank(spec, state)
        set_moves(spec, act, *toward(spec, state, gr, gc))
        return finish(spec, state, max_attack(spec, state, act))
    return policy


def wall_herding(spec, state, t, rng):
    """Learners of even index head for their nearest corner, the others for their nearest edge, and keep pushing against
    it: at the wall their moves leave the grid."""
    r, c = cells(spec, state)
    lrn = learners(spec)
    r, c = r[:, lrn], c[:, lrn]
    big = spec.rows + spec.cols
    up, left = r <= spec.rows - 1 - r, c <= spec.cols - 1 - c
    dr, dc = np.where(up, -big, big), np.where(left, -big, big)
    row_wall = np.minimum(r, spec.rows - 1 - r) <= np.minimum(c, spec.cols - 1 - c)
    edge = (np.arange(len(lrn)) % 2 == 1)[None, :]
    dr, dc = np.where(edge & ~row_wall, 0, dr), np.where(edge & row_wall, 0, dc)
    act = blank(spec, state)
    off = r < 0
    return finish(spec, state, set_moves(spec, act, np.where(off, 0, dr), np.where(off, 0, dc)))


def swap(partner):
    """learner l moves into the cell of learner partner[l] (pairs: each other's; triples: a rotation)"""
    partner = np.asarray(partner)

    def policy(spec, state, t, rng):
        r, c = cells(spec, state)
        lrn = learners(spec)
        pr, pc = r[:, lrn[partner]], c[:, lrn[partner]]
        dr, dc = toward(spec, state, pr, pc)
        gone = pr < 0
        act = blank(spec, state)
        return finish(spec, state, set_moves(spec, act, np.where(gone, 0, dr), np.where(gone, 0, dc)))
    return policy


def schedule(*phases):
    """(steps, policy), ... run one after the other; the last one runs on"""
    def policy(spec, state, t, rng):
        t0 = 0
        for n, p in phases:
            if t < t0 + n or p is phases[-1][1]:
                return p(spec, state, t - t0, rng)
            t0 += n
    return policy


# ---------------------------------------------------------------------------------------------------
# formations (fixed positions)
# ---------------------------------------------------------------------------------------------------
def _battler(enc, pos, view=5, att=1, move=1):
    return dict(enc=enc, pos=pos, klass=LRN | OBS | MOV | ATT | HEA, view=view, att_range=att, move=move, strength=1.0)


def convoy_spec(n_envs=2, seed=0xC0, band=48):
    """The headline shape (64 x 64, 256 learners of 4 teams, view 5, attack range 1: the C5 compile-time instantiation)
    in bands of `band` learners along rows 10, 12, ... (rows r and r + 2 share the reservation slots of a 128-slot
    table), teams alternating along each band.  Learner 0 leads band 0 at column band - 1, learner 1 follows it, and so
    on: in dict order the learners are processed front to back."""
    agents = []
    for i in range(256):
        b, k = divmod(i, band)
        agents.append(_battler(i % 4 + 1, (10 + 2 * b, band - 1 - k)))
    teams = {1, 2, 3, 4}
    sp = make_spec(64, 64, agents, overlapping={t: {t} for t in teams}, attack_mapping={t: teams - {t} for t in teams},
                   attack_actor=K.ATTACK_BINARY, done_mask=K.DONE_ONE_TEAM, n_envs=n_envs, seed=seed)
    sp.horizon, sp.auto_reset = 100, 1
    return sp


def swap_spec(n_envs=8, seed=0x5A, cross=False):
    """Pairs and triples of different teams side by side on a 15 x 16 grid, returned with the partner table of swap():
    a pair moves into each other's cells, a triple (an L of three cells) rotates.  Teams 1 and 2 may share a cell (so
    some exchanges succeed), team 3 may not; attack range 1 and view 2."""
    agents, partner = [], []
    for g in range(20):
        r0, c0 = 3 * (g // 5), 3 * (g % 5) + 1
        base = len(agents)
        if g % 2 == 0 or cross:                    # a pair (the cross actor cannot rotate an L)
            agents += [_battler(1 + g % 3, (r0, c0), view=2), _battler(1 + (g + 1) % 3, (r0, c0 + 1), view=2)]
            partner += [base + 1, base]
        else:                                      # a triple: (r0, c0) -> (r0, c0 + 1) -> (r0 + 1, c0) -> (r0, c0)
            agents += [_battler(1, (r0, c0), view=2), _battler(2, (r0, c0 + 1), view=2), _battler(3, (r0 + 1, c0), view=2)]
            partner += [base + 1, base + 2, base]
    sp = make_spec(15, 16, agents, overlapping={1: {1, 2}, 2: {2}, 3: {3}}, attack_mapping={1: {2, 3}, 2: {1, 3}, 3: {1, 2}},
                   attack_actor=K.ATTACK_BINARY, move_actor=K.MOVE_CROSS if cross else K.MOVE_BOX,
                   done_mask=K.DONE_ONE_TEAM, n_envs=n_envs, seed=seed)
    sp.horizon, sp.auto_reset = 30, 1
    return sp, np.array(partner)


# ---------------------------------------------------------------------------------------------------
# measurements, from the state before and after one step (and the actions)
# ---------------------------------------------------------------------------------------------------
def _same_episode(before, after):
    return before['episode'] == after['episode']


def move_chains(spec, before, after):
    """[E]: the longest chain of cross-team moves in the step, where each move enters a cell that the mover ahead (of
    another team) vacated in the same step.  0 for envs that were reset by the step."""
    r0, c0 = cells(spec, before)
    r1, c1 = cells(spec, after)
    enc = spec.encoding.astype(np.int64)
    out = np.zeros(r0.shape[0], dtype=np.int64)
    for e in np.nonzero(_same_episode(before, after))[0]:
        moved = np.nonzero((r0[e] >= 0) & (r1[e] >= 0) & ((r0[e] != r1[e]) | (c0[e] != c1[e])))[0]
        left = {}
        for a in moved:
            left.setdefault((r0[e, a], c0[e, a]), []).append(a)
        depth = {}

        def chain(a, seen=()):
            if a not in depth:
                ahead = [b for b in left.get((r1[e, a], c1[e, a]), ()) if enc[b] != enc[a] and b not in seen]
                depth[a] = 1 + max((chain(b, seen + (a,)) for b in ahead), default=0)
            return depth[a]
        out[e] = max((chain(a) for a in moved), default=0)
    return out


def largest_pile(spec, state):
    """[E]: the most entities in one cell"""
    r, c = cells(spec, state)
    cell = np.where(r >= 0, r * spec.cols + c, spec.rows * spec.cols)
    return np.array([np.bincount(row, minlength=spec.rows * spec.cols + 1)[:-1].max() for row in cell])


def kills(spec, before, after):
    """[E]: entities active before the step and inactive after it (envs not reset by the step)"""
    was = (before['flags'] & K.ST_ACTIVE) != 0
    now = (after['flags'] & K.ST_ACTIVE) != 0
    return np.where(_same_episode(before, after), (was & ~now).sum(axis=1), 0)


def overlapping_attackers(spec, state, actions):
    """[E]: the learners that attack (any attack byte set) from the grid whose attack windows overlap the window of
    another such learner"""
    r, c = cells(spec, state)
    lrn = learners(spec)
    r, c = r[:, lrn], c[:, lrn]
    R = spec.attack_range[lrn].astype(np.int64)
    attacking = ((actions[..., 2:] != 0).any(axis=-1)) & (r >= 0) & ((spec.klass[lrn] & K.AG_ATTACKING) != 0)
    reach = R[:, None] + R[None, :]
    near = (np.abs(r[:, :, None] - r[:, None, :]) <= reach) & (np.abs(c[:, :, None] - c[:, None, :]) <= reach)
    near &= attacking[:, :, None] & attacking[:, None, :]
    near &= ~np.eye(len(lrn), dtype=bool)[None]
    return near.any(axis=2).sum(axis=1)


def off_grid_moves(spec, state, actions):
    """[E]: learners in the grid whose move would leave it"""
    r, c = cells(spec, state)
    lrn = learners(spec)
    r, c = r[:, lrn], c[:, lrn]
    m = spec.move_range[lrn].astype(np.int64)
    if spec.move_actor == K.MOVE_CROSS:
        k = actions[..., 0].astype(np.int64)
        dr, dc = CROSS_DR[k], CROSS_DC[k]
    elif spec.ravel_actions:
        v = actions[..., 0].view(np.uint8).astype(np.int64)
        dr, dc = v // (2 * m + 1) - m, v % (2 * m + 1) - m
    else:
        dr, dc = actions[..., 0].astype(np.int64), actions[..., 1].astype(np.int64)
    nr, nc = r + dr, c + dc
    return ((r >= 0) & ((nr < 0) | (nr >= spec.rows) | (nc < 0) | (nc >= spec.cols))).sum(axis=1)


def exchanges(spec, before, after):
    """[E]: learners of different teams that took each other's cells in the step (counted once per learner)"""
    r0, c0 = cells(spec, before)
    r1, c1 = cells(spec, after)
    lrn = learners(spec)
    enc = spec.encoding[lrn]
    a0, a1 = r0[:, lrn] * spec.cols + c0[:, lrn], r1[:, lrn] * spec.cols + c1[:, lrn]
    ok = (r0[:, lrn] >= 0) & (r1[:, lrn] >= 0) & (a0 != a1)
    sw = ok[:, :, None] & ok[:, None, :] & (a1[:, :, None] == a0[:, None, :]) & (a1[:, None, :] == a0[:, :, None])
    sw &= (enc[:, None] != enc[None, :])[None]
    return np.where(_same_episode(before, after), sw.any(axis=2).sum(axis=1), 0)


def assert_in_action_space(spec, actions):
    """every row inside the reference's action spaces: box moves within move_range (or the ravelled index below
    (2m+1)^2), cross moves 0..4, attack bytes within each actor's bounds (zero beyond an actor's width)"""
    lrn = learners(spec)
    assert actions.dtype == np.int8 and actions.shape[1:] == (len(lrn), action_stride(spec))
    m = spec.move_range[lrn].astype(np.int64)
    a = actions.astype(np.int64)
    u = actions.view(np.uint8).astype(np.int64)
    if spec.move_actor == K.MOVE_BOX and spec.ravel_actions:
        assert (u[..., 0] < (2 * m + 1) ** 2).all() and (a[..., 1] == 0).all()
    elif spec.move_actor == K.MOVE_BOX:
        assert (np.abs(a[..., 0]) <= m).all() and (np.abs(a[..., 1]) <= m).all()
    else:
        assert ((a[..., 0] >= 0) & (a[..., 0] <= 4)).all() and (a[..., 1] == 0).all()
    kind = int(spec.attack_actor)
    for l, ag in enumerate(lrn):
        sim = int(spec.simultaneous_attacks[ag]) if spec.klass[ag] & K.AG_ATTACKING else 0
        n = 2 * int(spec.attack_range[ag]) + 1
        row = u[:, l, 2:]
        if sim == 0 or kind == K.ATTACK_NONE:
            width, hi = 0, 0
        elif kind == K.ATTACK_BINARY:
            width, hi = 1, sim
        elif kind == K.ATTACK_ENCODING:
            width, hi = spec.max_encoding, sim
            assert (row[:, :width][:, ~enemies_of(spec)[l, 1:]] == 0).all(), 'attack on an encoding outside the mapping'
        elif kind == K.ATTACK_RESTRICTED:
            width, hi = sim, n * n
        else:
            width, hi = n * n, sim
        assert (row[:, :width] <= hi).all() and (row[:, width:] == 0).all(), f'learner {l}: attack bytes out of bounds'
