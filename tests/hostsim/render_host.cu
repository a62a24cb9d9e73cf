/*
 * render_host.cu -- TEST INFRASTRUCTURE ONLY.  Compiles the render kernel's per-env scene and per-pixel colour code
 * (marl_soccer_b200/csrc/render_core.cuh, all __host__ __device__) for the HOST, so that the fp32 rasteriser can be
 * checked against the fp64 reference (tests/render_ref.py) on a machine without a GPU.  The product never loads it;
 * tests/test_gpu_render.py checks the real kernel through msoc_render.
 *
 * The envs arrive as msoc_env_state (what msoc_get_state returns) and are laid out as the handle lays them out: the
 * current record holds the pose behind the newest frame (hist_*[1]); where the state's own pose differs from it, the
 * state goes to the injected record and the current record is flagged FLAG_INJECT, as msoc_set_state does.
 *
 * Build: nvcc -O2 -std=c++17 --shared -Xcompiler -fPIC -o librender_host.so render_host.cu   (host code only)
 */
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>
#include <vector>

#include "../../include/msoc.h"
#include "../../marl_soccer_b200/csrc/render_core.cuh"

using namespace msoc;

static void pack_state(const msoc_env_state &S, float4 *r)
{
    Pose Q;
    for (int i = 0; i < 5; i++) { Q.px[i] = S.pos[i][0]; Q.py[i] = S.pos[i][1]; }
    for (int i = 0; i < 4; i++) { Q.vx[i] = S.vel[i][0]; Q.vy[i] = S.vel[i][1]; Q.ang[i] = S.ang[i]; Q.w[i] = S.angvel[i]; }
    pose_pack(Q, 0.0f, 0.0f, r);
}
static void pack_hist(const msoc_env_state &S, int k, float4 *r)
{
    Pose Q;
    for (int i = 0; i < 5; i++) { Q.px[i] = S.hist_pos[k][i][0]; Q.py[i] = S.hist_pos[k][i][1]; }
    for (int i = 0; i < 4; i++) { Q.vx[i] = S.hist_vel[k][i][0]; Q.vy[i] = S.hist_vel[k][i][1]; Q.ang[i] = S.hist_ang[k][i]; Q.w[i] = S.hist_angvel[k][i]; }
    pose_pack(Q, 0.0f, 0.0f, r);
}
/* the floats an image is drawn from: positions and agent angles */
static bool same_drawing(const float4 *a, const float4 *b)
{
    for (int i = 0; i < 5; i++)
        if (f2u(a[i].x) != f2u(b[i].x) || f2u(a[i].y) != f2u(b[i].y)) return false;
    return memcmp(&a[5], &b[5], sizeof(float4)) == 0;
}

extern "C" {

/* Images (n, height, width, 3) of the envs idx[0..n) (null: 0..n-1) out of the n_states states, through the same
   32-pixel segments of the flat pixel stream as msoc_render_kernel.  An index outside [0, n_states) gives a zero image. */
void rhost_render(const msoc_env_state *states, int64_t n_states, const int64_t *idx, int64_t n, int height, int width, uint8_t *out)
{
    std::vector<float4> cur((size_t)n_states * POSE_F4), inj((size_t)n_states * POSE_F4);
    for (int64_t e = 0; e < n_states; e++) {
        float4 *rec = cur.data() + e * POSE_F4, *ir = inj.data() + e * POSE_F4;
        const msoc_env_state &S = states[e];
        pack_state(S, ir);
        if (S.hist_valid) pack_hist(S, 1, rec);
        else pack_state(S, rec);
        const bool injected = !same_drawing(rec, ir);
        rec[7] = make_float4(0.0f, u2f((uint32_t)S.steps), u2f(injected ? FLAG_INJECT : 0u), 0.0f);
    }
    Arrays A;
    memset(&A, 0, sizeof A);
    A.n = n_states;
    A.pose[0] = A.pose[1] = A.pose[2] = cur.data();
    A.inject = inj.data();
    const int step = 0;

    RenderGeom G;
    render_geom(height, width, G);
    std::vector<RenderScene> scenes((size_t)n);
    for (int64_t i = 0; i < n; i++) {
        const int64_t e = idx ? idx[i] : i;
        render_scene(G, (e >= 0 && e < n_states) ? render_record(A, step, e) : nullptr, scenes[(size_t)i]);
    }
    const int64_t hw = (int64_t)height * width, total = n * hw;
    for (int64_t g0 = 0; g0 < total; g0 += RENDER_SEG) {
        const int64_t img = g0 / hw, rem = g0 - img * hw;
        const int count = total - g0 < RENDER_SEG ? (int)(total - g0) : RENDER_SEG;
        uint32_t wm, bm, rm, ym, zm, w[RENDER_SEG_WORDS];
        render_segment_masks(G, scenes.data() + img, 0, (int)(rem / width), (int)(rem % width), count, wm, bm, rm, ym, zm);
        render_pack(wm, bm, rm, ym, zm, w);
        memcpy(out + g0 * 3, w, (size_t)count * 3);
    }
}

} /* extern "C" */
