/* TEST INFRASTRUCTURE ONLY -- reference for the per-agent episode counters (DESIGN.md §3 item 16), in plain sequential C.
 *
 * ssds_step is ssdt_step (tests/tag_oracle.c, compiled into this translation unit the way that file compiles in the pinned
 * restatement) with the seven counters added; the phase functions are reused unchanged.  stats is [SSDS_N_STATS][SSDO_MAX_AGENTS],
 * field-major like the device buffer.  Hits dealt by a shooter are the change of the hit counts around its fire_beam call:
 * fire_beam is run on the sub-map whose hit_penalty is 1, so it counts one -1 per ray that hits an agent into neg_hits.
 *
 * Build: gcc -O2 -ffp-contract=off -fPIC -shared -I oracle -I tests tests/stats_oracle.c   (tests/stats_oracle.py)
 */
#include "tag_oracle.c"

enum { SSDS_APPLES, SSDS_APPLE_T, SSDS_FIRES, SSDS_HITS_DEALT, SSDS_HITS_TAKEN, SSDS_OUT_STEPS, SSDS_CLEANED, SSDS_N_STATS };
#define ST(f, i) stats[(f) * SSDO_MAX_AGENTS + (i)]

static int sum_hits(const int8_t* neg_hits, int k) {
    int s = 0;
    for (int j = 0; j < k; ++j) s += neg_hits[j];
    return s;
}

void ssds_step(const ssdo_map* m, const ssdo_map* subs, ssdo_env* e, uint8_t* tag_out, uint32_t* stats, const uint8_t* actions,
               const ssdo_draws* d, uint64_t seed, uint32_t env_gid, int tag_timeout, int random_spawn_point, int spawn_rotation,
               int8_t* reward, uint8_t* clean, uint16_t* apple_cnt, uint8_t* done) {
    const int n = m->n;
    const uint32_t t = (uint32_t)e->t + 1;                        /* the step's 1-based index in the episode */
    uint8_t was_out[SSDO_MAX_AGENTS], keep[SSDO_MAX_AGENTS], act[SSDO_MAX_AGENTS];
    int idx[SSDO_MAX_AGENTS];
    uint32_t prio[SSDO_MAX_AGENTS];
    int8_t r[SSDO_MAX_AGENTS], neg_hits[SSDO_MAX_AGENTS];
    for (int i = 0; i < n; ++i) { was_out[i] = tag_out[i] > 0; keep[i] = !was_out[i]; reward[i] = 0; clean[i] = 0; }
    for (int i = 0; i < n; ++i) ST(SSDS_OUT_STEPS, i) += was_out[i];

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
        if (s.grid[s.pos[j]] == SSDO_APPLE) {
            r[j] += 1; s.grid[s.pos[j]] = SSDO_EMPTY;
            ST(SSDS_APPLES, idx[j]) += 1; ST(SSDS_APPLE_T, idx[j]) += t;
        }
    for (int j = 0; j < k; ++j) {
        if (act[j] == 7) {
            r[j] -= (int8_t)m->fire_cost;
            const int before = sum_hits(neg_hits, k);
            fire_beam(sm, &s, j, 0, neg_hits);
            ST(SSDS_FIRES, idx[j]) += 1;
            ST(SSDS_HITS_DEALT, idx[j]) += (uint32_t)(before - sum_hits(neg_hits, k));
        } else if (act[j] == 8 && m->kind == SSDO_KIND_CLEANUP) {
            clean[idx[j]] = (uint8_t)fire_beam(sm, &s, j, 1, neg_hits);
            ST(SSDS_CLEANED, idx[j]) += clean[idx[j]];
        }
    }
    for (int j = 0; j < k; ++j) {                                 /* 2. hit = tagged; hit_penalty per hit */
        const int i = idx[j];
        reward[i] = (int8_t)(r[j] + neg_hits[j] * m->hit_penalty);
        ST(SSDS_HITS_TAKEN, i) += (uint32_t)(-neg_hits[j]);
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
        if (tag_out[i] == 1) respawn(m, e, tag_out, i, random_spawn_point, spawn_rotation, d, seed, env_gid);
        tag_out[i] -= 1;
    }

    int apples = 0;
    for (int c = 0; c < m->G; ++c) apples += e->grid[c] == SSDO_APPLE && !occupied_in_play(m, e, tag_out, c);
    *apple_cnt = (uint16_t)apples;
    for (int i = 0; i < n; ++i) e->ep_ret[i] += reward[i];
    e->t += 1; e->tick += 1;
    *done = e->t >= m->episode_limit;
}

void ssds_batch_step(const ssdo_map* m, const ssdo_map* subs, ssdo_env* envs, uint8_t* tag_out /* [B][SSDO_MAX_AGENTS] */,
                     uint32_t* stats /* [B][SSDS_N_STATS][SSDO_MAX_AGENTS] */, int B, const uint8_t* actions, uint64_t seed,
                     uint32_t env_gid0, int tag_timeout, int random_spawn_point, int spawn_rotation, int8_t* reward,
                     uint8_t* clean, uint16_t* apple_cnt, uint8_t* done, uint8_t* obs, int threads) {
    (void)threads;
    const int n = m->n;
    const long obs_env = (long)n * 3 * m->N * m->N;
#pragma omp parallel for num_threads(threads) schedule(static)
    for (int b = 0; b < B; ++b) {
        uint8_t* to = tag_out + (long)b * SSDO_MAX_AGENTS;
        ssds_step(m, subs, &envs[b], to, stats + (long)b * SSDS_N_STATS * SSDO_MAX_AGENTS, actions + (long)b * n, 0, seed,
                  env_gid0 + (uint32_t)b, tag_timeout, random_spawn_point, spawn_rotation, reward + (long)b * n,
                  clean + (long)b * n, apple_cnt + b, done + b);
        if (obs) ssdt_render_obs(m, &envs[b], to, obs + b * obs_env);
    }
}
