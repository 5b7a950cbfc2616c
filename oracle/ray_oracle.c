/*
 * ray_oracle.c -- CPU restatement of vr_render_rays / vr_camera_rays (TEST INFRASTRUCTURE ONLY, like
 * march_oracle.c, whose functions it reuses unchanged by including it).
 *
 * orc_render_rays is render_pixel (offscreen) with screen2worlddir replaced by a loaded ray: normalise
 * with normalize3 (common.cuh:18-23 _normalize), keep the unit direction as view direction, maybe_world2ndc,
 * tree offset/scale, rodrigues, trace_ray with the ray's depth limit, background compositing.  A ray with a
 * non-finite component or a direction of fp32 length 0 or infinity is a miss (background, alpha 0; alpha 1 in
 * depth mode) and is not counted.  orc_camera_rays writes screen2worlddir's direction before normalize3.
 */
#include "march_oracle.c"

#include "ray_oracle.h"

/* volrend.cu:22-29: screen2worlddir up to its _normalize */
static void camera_dir(int ix, int iy, const orc_camera* cam, float* dir) {
    const float* m = cam->c2w;
    float vx = ((float)ix - (float)cam->width * 0.5f) / cam->fx;
    float vy = -((float)iy - (float)cam->height * 0.5f) / cam->fy;
    dir[0] = fmaf(vx, m[0], vy * m[3]) - m[6];
    dir[1] = fmaf(vx, m[1], vy * m[4]) - m[7];
    dir[2] = fmaf(vx, m[2], vy * m[5]) - m[8];
}

void orc_camera_rays(const orc_camera* cam, int x0, int y0, int w, int h, float* origins, float* dirs) {
    for (int r = 0; r < h; ++r)
        for (int c = 0; c < w; ++c) {
            const size_t i = (size_t)r * w + c;
            camera_dir(x0 + c, y0 + r, cam, dirs + 3 * i);
            origins[3 * i] = cam->c2w[9]; origins[3 * i + 1] = cam->c2w[10]; origins[3 * i + 2] = cam->c2w[11];
        }
}

static void render_one_ray(const orc_tree* tree, const orc_options* opt, const float* o, const float* d, float tl,
                           float* out, orc_counters* cnt) {
    float dir[3] = {d[0], d[1], d[2]}, cen[3] = {o[0], o[1], o[2]};
    out[0] = out[1] = out[2] = out[3] = 0.f;
    const float len = norm3(dir);
    int ok = isfinite(len) && len > 0.f;
    for (int i = 0; i < 3; ++i) ok = ok && isfinite(cen[i]) && isfinite(dir[i]);
    if (!ok) {
        if (opt->render_depth) out[3] = 1.f;
    } else if (tree->N > 0) {
        normalize3(dir);
        float vdir[3] = {dir[0], dir[1], dir[2]};
        maybe_world2ndc(tree, dir, cen);
        for (int i = 0; i < 3; ++i) cen[i] = fmaf(tree->scale[i], cen[i], tree->offset[i]);
        rodrigues(opt->rot_dirs, vdir);
        trace_ray(tree, dir, vdir, cen, opt, tl, out, cnt);
    }
    const float remain = (1.f - out[3]) * opt->background_brightness;
    out[0] = remain + out[0]; out[1] = remain + out[1]; out[2] = remain + out[2];
}

typedef struct {
    const orc_tree* tree; const orc_options* opt;
    const float *o, *d, *tmax; int n;
    float* out; orc_counters cnt; int want_cnt;
    volatile int* next;
} ray_job_t;

static void* ray_worker(void* arg) {
    ray_job_t* j = (ray_job_t*)arg;
    for (;;) {
        const int b = __sync_fetch_and_add(j->next, 256);
        if (b >= j->n) break;
        for (int i = b; i < j->n && i < b + 256; ++i)
            render_one_ray(j->tree, j->opt, j->o + 3 * (size_t)i, j->d + 3 * (size_t)i, j->tmax ? j->tmax[i] : 1e9f,
                           j->out + 4 * (size_t)i, j->want_cnt ? &j->cnt : NULL);
    }
    return NULL;
}

int orc_render_rays(const orc_tree* tree, const orc_options* opt, const float* origins, const float* dirs,
                    const float* t_max, int n, float* rgba_f32, orc_counters* counters, int nthreads) {
    if (!tree || !opt || n < 0 || (n > 0 && (!origins || !dirs || !rgba_f32))) return -1;
    if (tree->N != 0 && tree->N != 2) return -2;
    pthread_once(&g_h2f_once, init_h2f);
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 256) nthreads = 256;
    volatile int next = 0;
    ray_job_t* jobs = (ray_job_t*)calloc((size_t)nthreads, sizeof(ray_job_t));
    pthread_t* th = (pthread_t*)calloc((size_t)nthreads, sizeof(pthread_t));
    for (int i = 0; i < nthreads; ++i) {
        ray_job_t* j = &jobs[i];
        j->tree = tree; j->opt = opt; j->o = origins; j->d = dirs; j->tmax = t_max; j->n = n;
        j->out = rgba_f32; j->want_cnt = counters != NULL; j->next = &next;
        if (i > 0) pthread_create(&th[i], NULL, ray_worker, j);
    }
    ray_worker(&jobs[0]);
    for (int i = 1; i < nthreads; ++i) pthread_join(th[i], NULL);
    if (counters) {
        memset(counters, 0, sizeof(*counters));
        for (int i = 0; i < nthreads; ++i) {
            counters->samples += jobs[i].cnt.samples;
            counters->child_loads += jobs[i].cnt.child_loads;
            counters->shaded += jobs[i].cnt.shaded;
            counters->rays_hit += jobs[i].cnt.rays_hit;
        }
    }
    free(jobs); free(th);
    return 0;
}
