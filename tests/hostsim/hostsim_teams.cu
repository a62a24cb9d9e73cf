/*
 * hostsim_teams.cu -- TEST INFRASTRUCTURE ONLY.  The host harness of hostsim.cu (included whole: the same handle,
 * reset, state and statistics entry points) plus hsim_step_teams, the host build of msoc_step_teams: the same flow as
 * hsim_step through env_step's TEAMS instances, reward (N,4) with red's reward in columns 2, 3.
 *
 * Build: nvcc -O2 -std=c++17 --shared -Xcompiler -fPIC -o libhostsim_teams.so hostsim_teams.cu   (host code only)
 */
#include "hostsim.cu"

extern "C" void hsim_step_teams(HostSim *h, const float *actions, float *obs_out, float *reward, uint8_t *done,
                                int8_t *goal, int32_t *score, uint32_t flags)
{
    h->last_contacts.assign((size_t)h->n, 0); h->last_load.assign((size_t)h->n, -1);
    const int step = h->step;
    for (int64_t e = 0; e < h->n; e++) {
        const float4 *rec = h->A.pose[buf_cur(step)] + e * POSE_F4;
        const bool injected = (f2u(rec[7].z) & FLAG_INJECT) != 0u;
        Env E;
        load_env(h->A, rec, e, E);
        StepOut out;
        /* the kernels' flow: contact-free fast pass first, the pass of the env's work class if it declines */
        int load = 0;
        float body[BODY_FIELDS * 5], con[CON_FIELDS * CON_FAST], geom[GEOM_WORDS], oldc[3 * OLD_FAST], isl[ISL_FIELDS * ISL_SLOTS];
        float ovf_store[MAXC - CON_FAST][CON_FIELDS];
        Work W;
        W.ovf = ovf_store;
        int pool_count = 0;
        W.body = body; W.pool = con; W.pool_count = &pool_count; W.geom = geom; W.old = oldc; W.isl = isl;
        const uint64_t gidx = h->global_offset + (uint64_t)e;
        if (!env_step<true>(MODE_FAST, 1 << MODE_FAST, E, actions + e * 12, h->cfg, h->A, cache_half(step), e, gidx, flags, W, out, load)) {
            load_env(h->A, (injected && load != 0) ? h->A.inject + e * POSE_F4 : rec, e, E);
            h->last_load[(size_t)e] = load;
            int dummy;
            pool_count = 0;
            env_step<true>(mode_of_load(load), 31, E, actions + e * 12, h->cfg, h->A, cache_half(step), e, gidx, flags, W, out, dummy);
        }
        h->last_contacts[(size_t)e] = out.n_contacts;
        store_env(h->A, buf_next(step), e, E, out.score_dirty);
        if (out.fresh_episode) {
            store_env_record(h->A.pose[buf_cur(step)] + e * POSE_F4, E);
            store_env_record(h->A.pose[buf_prev(step)] + e * POSE_F4, E);
        }
        reward[4 * e] = out.reward; reward[4 * e + 1] = out.reward;
        reward[4 * e + 2] = out.reward_r; reward[4 * e + 3] = out.reward_r;
        done[e] = out.done; goal[e] = out.goal;
        if (score) { score[2 * e] = out.score_b; score[2 * e + 1] = out.score_r; }
        write_obs(h, e, obs_out + e * 4 * OBS);
        if (out.done) { h->stats[0] += 1.0; h->stats[1] += out.finished_return; }
        if (out.goal > 0) h->stats[2] += 1.0;
        if (out.goal < 0) h->stats[3] += 1.0;
        h->stats[4] += 1.0; h->stats[5] += out.n_contacts; h->stats[6] += out.overflow;
    }
    h->step = (h->step + 1) % 6;
}
