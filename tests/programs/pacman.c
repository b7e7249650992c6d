/* PacmanSim (pacman.py:29-151) as a step program, with raw Grid.remove / Grid.place for the tunnel and cell iteration for
 * the overlaps.  Constants: PACMAN (agent), BAD_MOVE, ENTROPY, EAT_FOOD, KILL, DIE.  Roles: 4 food, 5 baddie. */
#define ROLE_FOOD 4
#define ROLE_BADDIE 5

BGWP_FN void teleport(bgwp_ctx *c, int a)                  /* :87-92, :116-121: (9,0) <-> (9,20) */
{
    if (bgwp_row(c, a) != 9 || (bgwp_col(c, a) != 0 && bgwp_col(c, a) != 20)) return;
    const int to = bgwp_col(c, a) == 0 ? 20 : 0;
    bgwp_remove(c, a);
    bgwp_place(c, a, 9, to);
}

BGWP_FN void overlaps(bgwp_ctx *c, int p, int eat_food)  /* :94-105, :123-131 (over a copy of the cell: read next first) */
{
    if (!bgwp_in_grid(c, p)) return;
    int o = bgwp_first_occupant(c, bgwp_row(c, p), bgwp_col(c, p));
    while (o >= 0) {
        const int nx = bgwp_next_occupant(c, o);
        if (o != p) {
            if (eat_food && bgwp_role(c, o) == ROLE_FOOD) {
                bgwp_add_reward(c, p, EAT_FOOD);
                bgwp_remove(c, o);
                bgwp_set_health(c, o, 0.0);
            } else if (bgwp_role(c, o) == ROLE_BADDIE) {
                bgwp_add_reward(c, p, DIE);
                bgwp_add_reward(c, o, KILL);
                bgwp_set_health(c, p, 0.0);
            }
        }
        o = nx;
    }
}

BGWP_FN void bgwp_step(bgwp_ctx *c)                        /* :80-135 */
{
    if (!bgwp_move(c, PACMAN)) bgwp_add_reward(c, PACMAN, BAD_MOVE);
    else bgwp_add_reward(c, PACMAN, ENTROPY);
    teleport(c, PACMAN);
    overlaps(c, PACMAN, 1);
    for (int i = 0; i < bgwp_n_acting(c); ++i) {
        const int a = bgwp_acting(c, i);
        if (a < 0 || a == PACMAN) continue;
        if (!bgwp_move(c, a)) bgwp_add_reward(c, a, BAD_MOVE);
        else bgwp_add_reward(c, a, ENTROPY);
        teleport(c, a);
    }
    overlaps(c, PACMAN, 0);
    if (!bgwp_active(c, PACMAN)) bgwp_remove(c, PACMAN);  /* :134-135 */
}

#define BGWP_HAS_GET_ALL_DONE
BGWP_FN int bgwp_get_all_done(const bgwp_ctx *c)          /* :140-151: pacman dead, or no FoodAgent left in the sim */
{
    if (!bgwp_active(c, PACMAN)) return 1;
    for (int a = 0; a < bgwp_n_agents(c); ++a) if (bgwp_role(c, a) == ROLE_FOOD) return 0;
    return 1;
}

#define BGWP_HAS_GET_DONE
BGWP_FN int bgwp_get_done(const bgwp_ctx *c, int a) { (void)a; return bgwp_get_all_done(c); }   /* :137-138 */
