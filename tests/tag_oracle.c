/* TEST INFRASTRUCTURE ONLY -- reference for the tagging-out timers (DESIGN.md §3 item 11), in plain sequential C.
 *
 * The reference env has no tagging; this file is the executable form of the spec the CUDA kernels are pinned to.  It builds
 * on the pinned restatement of the reference (oracle/ssd_oracle.c, compiled into this translation unit so that its static
 * phase functions can be reused unchanged): a phase runs on a copy of the env that holds only the agents in play, in index
 * order, so every "last index wins" / "index order" rule of the reference keeps its meaning among them.  Timers live in a
 * separate array, tag_out[n] (0 = in play).
 *
 * Build: gcc -O2 -ffp-contract=off -fPIC -shared -I oracle tests/tag_oracle.c   (tests/tag_oracle.py)
 */
#include "ssd_oracle.c"

/* subs[k] = *m with n = k agents and hit_penalty = 1 (fire_beam then counts hits into the reward array it is given) */
void ssdt_submaps(const ssdo_map* m, ssdo_map* subs) {
    for (int k = 0; k <= m->n; ++k) { subs[k] = *m; subs[k].n = k; subs[k].hit_penalty = 1; }
}

/* copy of e holding the agents with keep[i] set, in index order; idx[j] = original index of agent j */
static int compact(const ssdo_env* e, int n, const uint8_t* keep, ssdo_env* s, int* idx) {
    int k = 0;
    memcpy(s->grid, e->grid, sizeof(s->grid));
    for (int i = 0; i < n; ++i) {
        if (!keep[i]) continue;
        idx[k] = i; s->pos[k] = e->pos[i]; s->orient[k] = e->orient[i]; s->ep_ret[k] = 0;
        ++k;
    }
    s->t = e->t; s->tick = e->tick; s->error = e->error;
    return k;
}

static int occupied_in_play(const ssdo_map* m, const ssdo_env* e, const uint8_t* tag_out, int cell) {
    for (int j = 0; j < m->n; ++j) if (!tag_out[j] && e->pos[j] == cell) return 1;
    return 0;
}

/* respawn of agent i by the reset rules (map_env.py:771-793): the free spawn point with the largest (key, cell), where free
 * means no agent in play stands there (agents respawned earlier in the same step included) */
static void respawn(const ssdo_map* m, ssdo_env* e, const uint8_t* tag_out, int i, int random_spawn_point, int spawn_rotation,
                    const ssdo_draws* d, uint64_t seed, uint32_t env_gid) {
    const int S = m->n_spawn;
    int best = -1; uint32_t best_key = 0;
    for (int s = 0; s < S; ++s) {
        int c = m->spawn_pts[s];
        if (occupied_in_play(m, e, tag_out, c)) continue;
        uint32_t key = 0;
        if (random_spawn_point)
            key = d && d->spawn_key ? d->spawn_key[i * m->G + c] : philox_word(seed, env_gid, e->tick, 3, (uint32_t)(i * S + s));
        if (best < 0 || key >= best_key) { best = c; best_key = key; }
    }
    e->pos[i] = best;
    if (spawn_rotation >= 0) e->orient[i] = (uint8_t)spawn_rotation;
    else e->orient[i] = d && d->rot ? d->rot[i] : (uint8_t)(philox_word(seed, env_gid, e->tick, 4, (uint32_t)i) >> 30);
}

void ssdt_step(const ssdo_map* m, const ssdo_map* subs, ssdo_env* e, uint8_t* tag_out, const uint8_t* actions,
               const ssdo_draws* d, uint64_t seed, uint32_t env_gid, int tag_timeout, int random_spawn_point, int spawn_rotation,
               int8_t* reward, uint8_t* clean, uint16_t* apple_cnt, uint8_t* done) {
    const int n = m->n;
    uint8_t was_out[SSDO_MAX_AGENTS], keep[SSDO_MAX_AGENTS], act[SSDO_MAX_AGENTS];
    int idx[SSDO_MAX_AGENTS];
    uint32_t prio[SSDO_MAX_AGENTS];
    int8_t r[SSDO_MAX_AGENTS], neg_hits[SSDO_MAX_AGENTS];
    for (int i = 0; i < n; ++i) { was_out[i] = tag_out[i] > 0; keep[i] = !was_out[i]; reward[i] = 0; clean[i] = 0; }

    /* 1. moves, consume and beams among the agents in play; an agent out of play does nothing */
    ssdo_env s;
    const int k = compact(e, n, keep, &s, idx);
    const ssdo_map* sm = &subs[k];
    for (int j = 0; j < k; ++j) {
        act[j] = actions[idx[j]];
        prio[j] = d && d->prio ? d->prio[idx[j]] : philox_word(seed, env_gid, e->tick, 0, (uint32_t)idx[j]);
        r[j] = 0; neg_hits[j] = 0;
    }
    update_moves(sm, &s, act, prio);
    for (int j = 0; j < k; ++j)
        if (s.grid[s.pos[j]] == SSDO_APPLE) { r[j] += 1; s.grid[s.pos[j]] = SSDO_EMPTY; }
    for (int j = 0; j < k; ++j) {
        if (act[j] == 7) { r[j] -= (int8_t)m->fire_cost; fire_beam(sm, &s, j, 0, neg_hits); }
        else if (act[j] == 8 && m->kind == SSDO_KIND_CLEANUP) clean[idx[j]] = (uint8_t)fire_beam(sm, &s, j, 1, neg_hits);
    }
    for (int j = 0; j < k; ++j) {                                 /* 2. hit = tagged; hit_penalty per hit */
        const int i = idx[j];
        reward[i] = (int8_t)(r[j] + neg_hits[j] * m->hit_penalty);
        e->pos[i] = s.pos[j]; e->orient[i] = s.orient[j];
        if (tag_timeout > 0 && neg_hits[j]) { tag_out[i] = (uint8_t)tag_timeout; keep[i] = 0; }   /* 3. leaves the map */
    }
    memcpy(e->grid, s.grid, sizeof(e->grid));
    e->error = s.error;

    /* 4. spawning sees only the agents still in play */
    ssdo_env s2;
    const int k2 = compact(e, n, keep, &s2, idx);
    custom_map_update(&subs[k2], &s2, d, seed, env_gid);
    memcpy(e->grid, s2.grid, sizeof(e->grid));

    /* 5. the agents out at the start count down; those reaching 0 respawn in index order */
    for (int i = 0; i < n; ++i) {
        if (!was_out[i]) continue;
        if (tag_out[i] == 1) respawn(m, e, tag_out, i, random_spawn_point, spawn_rotation, d, seed, env_gid);   /* still out */
        tag_out[i] -= 1;                                          /* here, so its old cell does not block its own respawn */
    }

    int apples = 0;                                               /* map_env.py:291-292, agents in play */
    for (int c = 0; c < m->G; ++c) apples += e->grid[c] == SSDO_APPLE && !occupied_in_play(m, e, tag_out, c);
    *apple_cnt = (uint16_t)apples;
    for (int i = 0; i < n; ++i) e->ep_ret[i] += reward[i];
    e->t += 1; e->tick += 1;
    *done = e->t >= m->episode_limit;
}

/* render: agents out of play are not drawn, and their own view is all zero */
static void overlay_in_play(const ssdo_map* m, const ssdo_env* e, const uint8_t* tag_out, uint8_t* idx) {
    for (int c = 0; c < m->G; ++c) idx[c] = e->grid[c];
    for (int i = 0; i < m->n; ++i) if (!tag_out[i]) idx[e->pos[i]] = (uint8_t)(6 + agent_char(i));   /* later index overwrites */
}

void ssdt_render_state(const ssdo_map* m, const ssdo_env* e, const uint8_t* tag_out, uint8_t* out) {
    uint8_t idx[SSDO_MAX_CELLS];
    overlay_in_play(m, e, tag_out, idx);
    for (int ch = 0; ch < 3; ++ch) for (int c = 0; c < m->G; ++c) out[ch * m->G + c] = m->color[idx[c]][ch];
}

void ssdt_render_obs(const ssdo_map* m, const ssdo_env* e, const uint8_t* tag_out, uint8_t* obs) {
    const int N = m->N, V = m->V, W = m->W, H = m->H;
    uint8_t idx[SSDO_MAX_CELLS];
    overlay_in_play(m, e, tag_out, idx);
    for (int i = 0; i < m->n; ++i) {
        uint8_t* o = obs + (long)i * 3 * N * N;
        if (tag_out[i]) { memset(o, 0, (size_t)3 * N * N); continue; }
        int pr = e->pos[i] / W, pc = e->pos[i] % W;
        for (int y = 0; y < N; ++y) for (int x = 0; x < N; ++x) {
            int a, b;                                            /* np.rot90 k = 1, 3, 0, 2 (map_env.py:806-813) */
            switch (e->orient[i]) {
                case SSDO_LEFT:  a = x;         b = N - 1 - y; break;
                case SSDO_RIGHT: a = N - 1 - x; b = y;         break;
                case SSDO_UP:    a = y;         b = x;         break;
                default:         a = N - 1 - y; b = N - 1 - x; break;
            }
            int r = pr - V + a, c = pc - V + b;
            int ci = (r >= 0 && r < H && c >= 0 && c < W) ? idx[r * W + c] : 6;
            for (int ch = 0; ch < 3; ++ch) o[(ch * N + y) * N + x] = m->color[ci][ch];
        }
    }
}

void ssdt_batch_step(const ssdo_map* m, const ssdo_map* subs, ssdo_env* envs, uint8_t* tag_out /* [B][SSDO_MAX_AGENTS] */,
                     int B, const uint8_t* actions, uint64_t seed, uint32_t env_gid0, int tag_timeout, int random_spawn_point,
                     int spawn_rotation, int8_t* reward, uint8_t* clean, uint16_t* apple_cnt, uint8_t* done, uint8_t* obs,
                     int threads) {
    (void)threads;
    const int n = m->n;
    const long obs_env = (long)n * 3 * m->N * m->N;
#pragma omp parallel for num_threads(threads) schedule(static)
    for (int b = 0; b < B; ++b) {
        uint8_t* to = tag_out + (long)b * SSDO_MAX_AGENTS;
        ssdt_step(m, subs, &envs[b], to, actions + (long)b * n, 0, seed, env_gid0 + (uint32_t)b, tag_timeout,
                  random_spawn_point, spawn_rotation, reward + (long)b * n, clean + (long)b * n, apple_cnt + b, done + b);
        if (obs) ssdt_render_obs(m, &envs[b], to, obs + b * obs_env);
    }
}
