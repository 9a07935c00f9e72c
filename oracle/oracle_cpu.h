/* oracle/oracle_cpu.h -- TEST INFRASTRUCTURE: C restatement of the reference's depthmap path (see oracle_cpu.c). */
#ifndef ORACLE_CPU_H
#define ORACLE_CPU_H
#include <stdint.h>

#include "../include/tsar_b200.h" /* plain structs tsar_camera / tsar_params only */

typedef struct oc_ctx oc_ctx;
oc_ctx *oc_create(int W, int H, int n_images, const float *const *images, const tsar_camera *cams, float cam_f,
                  const int *subset, int V, const tsar_params *p);
void oc_destroy(oc_ctx *c);
float *oc_planes(oc_ctx *c);
float *oc_costs(oc_ctx *c);
int *oc_beview(oc_ctx *c);
long long oc_evals(oc_ctx *c);
void oc_xorwow_row(uint64_t seed, int y, int n, uint32_t *out);
float oc_tex(const float *img, int W, int H, float x, float y);
float oc_multiview(oc_ctx *c, int x, int y, const float *pl, int hrad, int vrad, int pxf, int *beview, float *ratio);
void oc_eval_planes(oc_ctx *c, int n, const int *xy, const float *planes, int pxf, float *cost, int *beview, float *ratio);
void oc_eval_views(oc_ctx *c, int n, const int *xy, const float *planes, int pxf, float *cost, double *src_rel);
void oc_init(oc_ctx *c, uint64_t seed);
void oc_init_planes_only(oc_ctx *c, uint64_t seed);
void oc_spatial(oc_ctx *c, int colour);
void oc_refine(oc_ctx *c, int colour, uint64_t seed);
void oc_iterate(oc_ctx *c, int iters, uint64_t seed0);
void oc_output(oc_ctx *c, float *out);
int oc_fit_region_plane(int W, int H, const tsar_camera *cam0, float cam_f, const float *depth, const float *scale,
                        const float *canny, int region, float region_size, const uint32_t *rnd, float *plane_io);
#endif
