/* oracle_filtered.c - the oracle (oracle/pt_oracle.c, included whole and unchanged) with the product's pixel filter in front.
 *
 * TEST INFRASTRUCTURE ONLY. The reference has no pixel filter: every sample goes through the pixel corner. What follows restates
 * THE PRODUCT'S DEFINITION (csrc/rt_filter.cuh, DESIGN.md 5), not the reference's, so that the anti-aliased renders can be checked
 * against the oracle's own radiance(): words (x, y) of Philox (pixel, sample, 0, 1) with the key (seed_lo, seed_hi),
 * u = (w >> 8) * 2^-24, box (2u - 1) r, tent v = 2u, (v < 1 ? sqrt(v) - 1 : 1 - sqrt(2 - v)) r, and GetRayDirection with px + jx,
 * py + jy in place of px, py. Built like the oracle (gcc -std=c11 -O2 -ffp-contract=off -fno-fast-math) by tests/oracle_filtered.py.
 */
#include "../oracle/pt_oracle.c"

enum { ORC_FILTER_NONE = 0, ORC_FILTER_BOX = 1, ORC_FILTER_TENT = 2 };

static float filter_offset(int type, float r, uint32_t w) {
    if (type == ORC_FILTER_NONE) return 0.f;
    float u = (float)(w >> 8) * 0x1p-24f;
    if (type == ORC_FILTER_BOX) return (u * 2.f - 1.f) * r;
    float v = u * 2.f;
    return (v < 1.f ? sqrtf(v) - 1.f : 1.f - sqrtf(2.f - v)) * r;
}

static v3 filtered_ray_dir(const raygen* g, const uint32_t key[2], int type, float r, int px, int py, uint32_t sample) {
    uint32_t ctr[4] = {(uint32_t)px + (uint32_t)py * (uint32_t)g->w, sample, 0u, 1u}, w[4];
    philox4x32_10(ctr, key, w);
    float nX = (((float)px + filter_offset(type, r, w[0])) / (float)g->w) * 2 - 1;
    float nY = (((float)py + filter_offset(type, r, w[1])) / (float)g->h) * 2 - 1;
    return vnormalized(vadd(vadd(vscale(g->u_axis, nX), vscale(g->v_axis, nY)), g->fwd));
}

/* The primary direction of global sample `sample` of every pixel (w*h*3 floats, y-up). */
void orc_sample_dirs(const orc_camera* cam, int w, int h, uint32_t seed_lo, uint32_t seed_hi, int filter_type, float filter_radius,
                     uint32_t sample, float* out_xyz) {
    raygen g = make_raygen(cam, w, h);
    const uint32_t key[2] = {seed_lo, seed_hi};
    for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
            v3 d = filtered_ray_dir(&g, key, filter_type, filter_radius, x, y, sample);
            float* o = out_xyz + 3 * ((size_t)x + (size_t)y * w);
            o[0] = d.x; o[1] = d.y; o[2] = d.z;
        }
}

/* orc_render (Philox streams: rng_mode 1) with every sample's primary ray taken from filtered_ray_dir; rows split over threads. */
typedef struct {
    const orc_object* objs; int n; const orc_camera* cam; const orc_params* p;
    int s0, nspp, y0, y1, filter_type; float filter_radius;
    float* out_sum; float* out_samples; long long segs;
} filtered_job;

static void* filtered_band(void* arg) {
    filtered_job* j = (filtered_job*)arg;
    const orc_params* p = j->p;
    int w = p->width, h = p->height;
    raygen g = make_raygen(j->cam, w, h);
    rng_t rng; memset(&rng, 0, sizeof rng);
    rng.mode = 1; rng.key[0] = p->seed_lo; rng.key[1] = p->seed_hi;
    long long segs = 0;
    for (int y = j->y0; y < j->y1; ++y)
        for (int x = 0; x < w; ++x) {
            size_t px = (size_t)x + (size_t)y * w;
            float sr = 0.f, sg = 0.f, sb = 0.f;
            for (int s = 0; s < j->nspp; ++s) {
                v3 d = filtered_ray_dir(&g, rng.key, j->filter_type, j->filter_radius, x, y, (uint32_t)(j->s0 + s));
                rng_begin(&rng, (uint32_t)px, (uint32_t)(j->s0 + s));
                col c = radiance(j->objs, j->n, p, g.pos, d, &rng, &segs);
                sr += c.r; sg += c.g; sb += c.b;
                if (j->out_samples) {
                    float* o = j->out_samples + 3 * ((size_t)s * w * h + px);
                    o[0] = c.r; o[1] = c.g; o[2] = c.b;
                }
            }
            if (j->out_sum) { j->out_sum[3*px] = sr; j->out_sum[3*px+1] = sg; j->out_sum[3*px+2] = sb; }
        }
    j->segs = segs;
    return NULL;
}

long long orc_render_filtered(const orc_object* objs, int n, const orc_camera* cam, const orc_params* p, int s0, int nspp,
                              int filter_type, float filter_radius, int threads, float* out_sum_rgb, float* out_per_sample_rgb) {
    if (threads < 1) threads = 1;
    if (threads > 256) threads = 256;
    if (threads > p->height) threads = p->height;
    filtered_job jobs[256]; pthread_t tid[256];
    for (int i = 0; i < threads; ++i) {
        filtered_job* j = &jobs[i];
        j->objs = objs; j->n = n; j->cam = cam; j->p = p; j->s0 = s0; j->nspp = nspp;
        j->filter_type = filter_type; j->filter_radius = filter_radius;
        j->out_sum = out_sum_rgb; j->out_samples = out_per_sample_rgb; j->segs = 0;
        j->y0 = (int)((long long)p->height * i / threads);
        j->y1 = (int)((long long)p->height * (i + 1) / threads);
    }
    for (int i = 0; i < threads; ++i) pthread_create(&tid[i], NULL, filtered_band, &jobs[i]);
    for (int i = 0; i < threads; ++i) pthread_join(tid[i], NULL);
    long long segs = 0;
    for (int i = 0; i < threads; ++i) segs += jobs[i].segs;
    return segs;
}
