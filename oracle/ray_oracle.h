/* ray_oracle.h -- ray-batch entry points of the CPU restatement (test infrastructure only; see ray_oracle.c). */
#ifndef RAY_ORACLE_H_
#define RAY_ORACLE_H_
#include "march_oracle.h"

#ifdef __cplusplus
extern "C" {
#endif

/* Rays of the pixels of tile (x0, y0, w, h) of cam, row-major: origin c2w[9..11], direction before normalisation. */
void orc_camera_rays(const orc_camera* cam, int x0, int y0, int w, int h, float* origins, float* dirs);

/* n rays (origins/dirs [n][3], t_max [n] or NULL = 1e9) -> rgba_f32 [n][4]; counters accumulated if non-NULL. */
int orc_render_rays(const orc_tree* tree, const orc_options* opt, const float* origins, const float* dirs,
                    const float* t_max, int n, float* rgba_f32, orc_counters* counters, int nthreads);

#ifdef __cplusplus
}
#endif
#endif
