/*
 * cc_oracle_np.c — the C oracle (oracle/cc_oracle.c, included whole) with the placements of CC_RESET_RNG_NUMPY:
 * the auto-reset and the masked reset continue each env's numpy generator, as the reference's reset() without a
 * seed does.  TEST INFRASTRUCTURE: tests/np_oracle.py compiles it into a temporary directory and binds it.
 *
 * gen: [N][6] uint64 per env, the layout of cc_oracle_reset_seeded / cc_get_rng_state:
 * {state hi, state lo, inc hi, inc lo, buffered uint32, has_buffered}.
 */
#include "../../oracle/cc_oracle.c"

static void np_gen_load(const uint64_t *s, orc_pcg64 *g) {
    g->state = ((unsigned __int128)s[0] << 64) | s[1];
    g->inc = ((unsigned __int128)s[2] << 64) | s[3];
    g->uinteger = (uint32_t)s[4];
    g->has_uint32 = s[5] != 0;
}
static void np_gen_store(const orc_pcg64 *g, uint64_t *s) {
    s[0] = (uint64_t)(g->state >> 64); s[1] = (uint64_t)g->state;
    s[2] = (uint64_t)(g->inc >> 64); s[3] = (uint64_t)g->inc;
    s[4] = g->uinteger; s[5] = g->has_uint32 ? 1 : 0;
}

/* collectivecrossing.py:91-150 reset() drawing from the env's numpy generator (the device's np_place_agent, the
 * loop of cc_oracle_reset_seeded): per agent, candidates until one is a valid, free cell; at the attempt cap the last
 * candidate is kept.  Returns 0, or 1 if the cap was hit. */
static int np_place(const cc_config *cfg, orc_env *e, orc_pcg64 *g) {
    int stuck = 0;
    e->step = 0;                                        /* :97 */
    for (int i = 0; i < e->A; ++i) { e->active[i] = 0; e->terminated[i] = 0; e->truncated[i] = 0; }
    for (int i = 0; i < e->A; ++i) {
        int px = 0, py = 0, ok = 0;
        for (int attempt = 0; attempt < ORC_RESET_ATTEMPT_CAP && !ok; ++attempt) {
            if (i < e->B) {
                px = (int)pcg_integers(g, 0, cfg->width);
                py = (int)pcg_integers(g, 0, cfg->division_y);
                ok = orc_is_valid_position(cfg, px, py) && !orc_is_position_occupied(e, i, px, py, -1) &&
                     !(cfg->door_left <= px && px <= cfg->door_right && py == cfg->division_y - 1);
            } else {
                px = (int)pcg_integers(g, cfg->tram_left, cfg->tram_right + 1);
                py = (int)pcg_integers(g, cfg->division_y, cfg->height);
                ok = orc_is_valid_position(cfg, px, py) && !orc_is_position_occupied(e, i, px, py, -1);
            }
        }
        if (!ok) stuck = 1;
        e->x[i] = px; e->y[i] = py; e->active[i] = 1;
    }
    return stuck;
}

/* cc_oracle_step whose auto-reset places env n from gen[n] and advances it; random actions still come from Philox
 * (seed, global env, t).  The step itself is the oracle's, run without auto-reset; an env whose episode ended is
 * then placed here, its return zeroed and its rows rewritten — what orc_step_env does with the Philox placement. */
int cc_oracle_np_step(const cc_config *cfg, int64_t n_envs, int64_t global_env_offset, uint64_t seed, uint64_t t,
                      int8_t *x, int8_t *y, uint8_t *flags, int32_t *step, float *episode_return, const cc_step_io *io,
                      cc_stats *stats, uint64_t *gen) {
    int A = cfg->num_boarding + cfg->num_exiting;
    if (A < 1 || A > ORC_MAX_A) return CC_ERR_UNSUPPORTED;
    if (!gen) return CC_ERR_INVALID_ARG;
    cc_step_io plain = *io;
    plain.auto_reset = 0;
    int status = 0;
    cc_stats total;
    memset(&total, 0, sizeof total);
#pragma omp parallel
    {
        cc_stats local;
        memset(&local, 0, sizeof local);
        int lstatus = 0;
#pragma omp for schedule(static)
        for (int64_t n = 0; n < n_envs; ++n) {
            orc_env e;
            orc_load(cfg, &e, x, y, flags, step, n);
            lstatus |= orc_step_env(cfg, &e, &plain, n, seed, (uint64_t)(global_env_offset + n), (uint32_t)t, episode_return, &local);
            if (io->auto_reset && (io->env_flags[n] & (CC_E_TERMINATED_ALL | CC_E_TRUNCATED_ALL))) {
                orc_pcg64 g;
                np_gen_load(gen + 6 * n, &g);
                if (np_place(cfg, &e, &g)) lstatus |= 2;
                np_gen_store(&g, gen + 6 * n);
                io->env_flags[n] |= CC_E_WAS_RESET;
                episode_return[n] = 0.0f;
                orc_write_obs(cfg, &e, io->obs, io->obs_dtype, n);
            }
            orc_store(&e, x, y, flags, step, n);
        }
#pragma omp critical
        { orc_stats_add(&total, &local); status |= lstatus; }
    }
    if (stats) orc_stats_add(stats, &total);
    if (status & 1) return CC_ERR_INVALID_ACTION;
    if (status & 2) return CC_ERR_RESET_STUCK;
    return CC_OK;
}

/* reset() without a seed for the envs with mask[n] != 0 (mask NULL: all): each continues its generator; the other
 * envs, their generators and their observation rows are untouched (cc_reset under CC_RESET_RNG_NUMPY) */
int cc_oracle_np_reset(const cc_config *cfg, int64_t n_envs, const uint8_t *mask, uint64_t *gen, int8_t *x, int8_t *y,
                       uint8_t *flags, int32_t *step, float *episode_return, void *obs, int32_t obs_dtype) {
    int A = cfg->num_boarding + cfg->num_exiting;
    if (A < 1 || A > ORC_MAX_A || !gen) return CC_ERR_INVALID_ARG;
    int stuck = 0;
    for (int64_t n = 0; n < n_envs; ++n) {
        if (mask && !mask[n]) continue;
        orc_pcg64 g;
        np_gen_load(gen + 6 * n, &g);
        orc_env e;
        orc_load(cfg, &e, x, y, flags, step, n);
        stuck |= np_place(cfg, &e, &g);
        orc_store(&e, x, y, flags, step, n);
        episode_return[n] = 0.0f;
        orc_write_obs(cfg, &e, obs, obs_dtype, n);
        np_gen_store(&g, gen + 6 * n);
    }
    return stuck ? CC_ERR_RESET_STUCK : CC_OK;
}
