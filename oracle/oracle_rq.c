/* oracle/oracle_rq.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE. See oracle_rq.h.
 *
 * Plain-C restatement of the reference ray query. Build with
 *   gcc -std=c11 -O2 -ffp-contract=off -fno-fast-math
 * so that every fp32 operation below is a single IEEE-754 round-to-nearest operation in the
 * order written (x86-64 SSE: FLT_EVAL_METHOD == 0). All literals carry an `f` suffix: MSL
 * literals are float-typed, and the verbatim build uses -fsingle-precision-constant.
 *
 * Arithmetic-order conventions (fixed by oracle/shim/metal_stdlib, SURVEY.md appendix B):
 *   dot(a,b) = (a.x*b.x + a.y*b.y) + a.z*b.z;   cross as written in v3_cross;
 *   normalize(v) = v / sqrtf(dot(v,v));   min/max = fminf/fmaxf;   max3(a,b,c)=max(max(a,b),c).
 */
#include "oracle_rq.h"

#include <float.h>
#include <math.h>
#include <pthread.h>
#include <stdlib.h>
#include <string.h>

#define ORQ_PI_F   3.14159265358979323846264338327950288f
#define ORQ_PI_2_F 1.57079632679489661923132169163975144f

typedef struct { float x, y, z; } v3;

static inline v3 v3_make(float x, float y, float z) { v3 r = {x, y, z}; return r; }
static inline v3 v3_ld(const float* p) { return v3_make(p[0], p[1], p[2]); }
static inline void v3_st(float* p, v3 a) { p[0] = a.x; p[1] = a.y; p[2] = a.z; }
static inline v3 v3_add(v3 a, v3 b) { return v3_make(a.x + b.x, a.y + b.y, a.z + b.z); }
static inline v3 v3_sub(v3 a, v3 b) { return v3_make(a.x - b.x, a.y - b.y, a.z - b.z); }
static inline v3 v3_mul(v3 a, v3 b) { return v3_make(a.x * b.x, a.y * b.y, a.z * b.z); }
static inline v3 v3_scale(v3 a, float s) { return v3_make(a.x * s, a.y * s, a.z * s); }
static inline v3 v3_divs(v3 a, float s) { return v3_make(a.x / s, a.y / s, a.z / s); }
static inline v3 v3_neg(v3 a) { return v3_make(-a.x, -a.y, -a.z); }
static inline float v3_dot(v3 a, v3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
static inline v3 v3_cross(v3 a, v3 b) {
    return v3_make(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
static inline v3 v3_normalize(v3 a) { return v3_divs(a, sqrtf(v3_dot(a, a))); }
static inline float v3_get(v3 a, unsigned i) { return i == 0 ? a.x : (i == 1 ? a.y : a.z); }
static inline void v3_set(v3* a, unsigned i, float v) { if (i == 0) a->x = v; else if (i == 1) a->y = v; else a->z = v; }

/* HitRecord::checkFace  HitRecord.hh:26-29 */
static inline void check_face(v3 dir, v3 gn, uint32_t* front, v3* sn) {
    int f = v3_dot(dir, gn) <= 0.0f;
    *front = (uint32_t)f;
    *sn = f ? gn : v3_neg(gn);
}

/* ---------------------------------------------------------------- AABB  (AABB.hh:73-112) */
static inline int slab(const orq_aabb* b, v3 o, v3 d, const float range[2], float* tmin_out, float* tmax_out) {
    v3 inv = v3_make(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);                 /* AABB.hh:75,94 */
    v3 ts = v3_mul(v3_sub(v3_ld(b->mini), o), inv);                       /* :77,96 */
    v3 te = v3_mul(v3_sub(v3_ld(b->maxi), o), inv);                       /* :78,97 */
    v3 a = v3_make(fminf(ts.x, te.x), fminf(ts.y, te.y), fminf(ts.z, te.z));
    v3 c = v3_make(fmaxf(ts.x, te.x), fmaxf(ts.y, te.y), fmaxf(ts.z, te.z));
    float tmin = fmaxf(fmaxf(a.x, a.y), a.z);                             /* max3 :83,102 */
    float tmax = fminf(fminf(c.x, c.y), c.z);                             /* min3 :84,103 */
    tmin = fmaxf(tmin, range[0]);                                          /* :86,105 */
    tmax = fminf(tmax, range[1]);                                          /* :87,106 */
    *tmin_out = tmin; *tmax_out = tmax;
    return !(tmax < tmin || tmax < 0.0f);                                  /* :89,108 */
}

int orq_aabb_hit(const orq_aabb* box, const float o[3], const float d[3], const float range[2]) {
    float tmin, tmax;
    return slab(box, v3_ld(o), v3_ld(d), range, &tmin, &tmax);
}

int orq_aabb_hit_t(const orq_aabb* box, const float o[3], const float d[3], const float range[2], float* t) {
    float tmin, tmax;
    if (!slab(box, v3_ld(o), v3_ld(d), range, &tmin, &tmax)) return 0;
    *t = (tmin < 0.0f) ? tmax : tmin;                                      /* :109 */
    return 1;
}

/* AABB::hit(ray, range, record)  AABB.hh:114-209 -- used by Cube::hit_test only */
static int aabb_hit_record(const orq_aabb* b, v3 o, v3 d, const float range[2],
                           float* t_out, v3* p_out, v3* gn_out, float uv_out[2]) {
    /* gamma(3) = (3*MachineEpsilon)/(1-3*MachineEpsilon), MachineEpsilon = FLT_EPSILON*0.5  Math.hh:51-55 */
    const float g3 = (3 * FLT_EPSILON * 0.5f) / (1 - 3 * FLT_EPSILON * 0.5f);
    const float widen = 1 + 2 * g3;
    float tmin = -FLT_MAX, tmax = range[1];
    unsigned axis = 0;
    v3 mini = v3_ld(b->mini), maxi = v3_ld(b->maxi);
    v3 ddd = v3_sub(o, mini), bbb = v3_sub(o, maxi);
    int inside = (ddd.x > 0.0f && ddd.y > 0.0f && ddd.z > 0.0f) && (bbb.x < 0.0f && bbb.y < 0.0f && bbb.z < 0.0f);
    v3 gn = v3_make(0.0f, 0.0f, 0.0f), hp, p;
    if (inside) {                                                          /* :124-166 */
        for (unsigned i = 0; i < 3; ++i) {
            float lo = (v3_get(mini, i) - v3_get(o, i)) / v3_get(d, i);
            float hi = (v3_get(maxi, i) - v3_get(o, i)) / v3_get(d, i);
            float ts = fminf(hi, lo), te = fmaxf(hi, lo);
            te *= widen;
            tmin = fmaxf(ts, tmin);
            if (te < tmax) { tmax = te; axis = i; }
            if (tmax < tmin || tmax < 0.0f) return 0;
        }
        *t_out = tmax;
        v3_set(&gn, axis, v3_get(d, axis) > 0.0f ? 1.0f : -1.0f);
        hp = v3_add(o, v3_scale(d, tmax));
        p = hp;
        v3_set(&p, axis, v3_get(d, axis) > 0.0f ? v3_get(maxi, axis) : v3_get(mini, axis));
    } else {                                                               /* :168-208 */
        for (unsigned i = 0; i < 3; ++i) {
            float lo = (v3_get(mini, i) - v3_get(o, i)) / v3_get(d, i);
            float hi = (v3_get(maxi, i) - v3_get(o, i)) / v3_get(d, i);
            float ts = fminf(hi, lo), te = fmaxf(hi, lo);
            te *= widen;
            tmax = fminf(te, tmax);
            if (ts > tmin) { tmin = ts; axis = i; }
            if (tmax < tmin || tmax < 0.0f) return 0;
        }
        *t_out = tmin;
        v3_set(&gn, axis, v3_get(d, axis) > 0.0f ? -1.0f : 1.0f);
        hp = v3_add(o, v3_scale(d, tmin));
        p = hp;
        v3_set(&p, axis, v3_get(d, axis) > 0.0f ? v3_get(mini, axis) : v3_get(maxi, axis));
    }
    *p_out = p; *gn_out = gn;
    uv_out[0] = v3_get(hp, (1 + axis) % 3);                                /* :162-163, :205-206 */
    uv_out[1] = v3_get(hp, (2 + axis) % 3);
    return 1;
}

/* ---------------------------------------------------------------- Triangle  (Triangle.hh:31-85) */
int orq_triangle_hit(const orq_vertex* triList, const uint32_t abc[3], const float o_[3], const float d_[3],
                     float range[2], orq_record* rec, float bary[2]) {
    const orq_vertex* A = &triList[abc[0]];
    const orq_vertex* B = &triList[abc[1]];
    const orq_vertex* C = &triList[abc[2]];
    v3 ori = v3_ld(o_), dir = v3_ld(d_);
    v3 v0 = v3_ld(A->v), v1 = v3_ld(B->v), v2 = v3_ld(C->v);
    v3 e1 = v3_sub(v1, v0);                                                /* :43 */
    v3 e2 = v3_sub(v2, v0);                                                /* :44 */
    v3 pvec = v3_cross(dir, e2);                                           /* :46 */
    float det = v3_dot(e1, pvec);                                          /* :47 */
    if (fabsf(det) < FLT_EPSILON) return 0;                                /* :55 (CULLING undefined) */
    float invDet = 1.0f / det;                                             /* :58 */
    v3 tvec = v3_sub(ori, v0);                                             /* :60 */
    float u = v3_dot(tvec, pvec) * invDet;                                 /* :61 */
    if (u < 0.0f || u > 1.0f) return 0;                                    /* :62 */
    v3 qvec = v3_cross(tvec, e1);                                          /* :64 */
    float v = v3_dot(dir, qvec) * invDet;                                  /* :65 */
    if (v < 0.0f || (u + v) > 1.0f) return 0;                              /* :66 */
    float w = 1.0f - u - v;                                                /* :68 */
    float t = v3_dot(e2, qvec) * invDet;                                   /* :69 */
    if (t > range[1] || t < range[0]) return 0;                            /* :71  (t == range.y passes) */
    range[1] = t;                                                          /* :75 */
    if (bary) { bary[0] = u; bary[1] = v; }
    if (rec) {
        v3 p = v3_add(v3_add(v3_scale(v1, u), v3_scale(v2, v)), v3_scale(v0, w));      /* :73 */
        v3 gn = v3_add(v3_add(v3_scale(v3_ld(B->n), u), v3_scale(v3_ld(C->n), v)), v3_scale(v3_ld(A->n), w)); /* :78 */
        rec->uv[0] = (u * B->uv[0] + v * C->uv[0]) + w * A->uv[0];         /* :79 */
        rec->uv[1] = (u * B->uv[1] + v * C->uv[1]) + w * A->uv[1];
        v3 sn; uint32_t f;
        check_face(dir, gn, &f, &sn);                                      /* :81 */
        rec->hit = 1; rec->t = t; rec->front = f; rec->material = 19;      /* :82 */
        v3_st(rec->p, p); v3_st(rec->gn, gn); v3_st(rec->sn, sn);
    }
    return 1;
}

/* ---------------------------------------------------------------- Sphere  (Sphere.hh:19-78) */
int orq_sphere_hit(const orq_sphere* s, const float o_[3], const float d_[3], float range[2], orq_record* rec) {
    v3 o = v3_ld(o_), d = v3_ld(d_), c = v3_ld(s->center);
    v3 oc = v3_sub(o, c);                                                  /* :35 */
    float a = v3_dot(d, d);                                                /* :37 */
    float half_b = v3_dot(oc, d);                                          /* :38 */
    float cc = v3_dot(oc, oc) - s->radius * s->radius;                     /* :39 */
    float disc = half_b * half_b - a * cc;                                 /* :41 */
    if (disc <= 0.0f) return 0;                                            /* :42 */
    float t_min = range[0], t_max = range[1];
    float root = sqrtf(disc);                                              /* :47 */
    float temp = (-half_b - root) / a;                                     /* :49 */
    if (!(temp < t_max && temp > t_min)) {                                 /* :50 (strict) */
        temp = (-half_b + root) / a;                                       /* :63 */
        if (!(temp < t_max && temp > t_min)) return 0;                     /* :64 */
    }
    range[1] = temp;                                                       /* :58,72 */
    if (rec) {
        v3 p = v3_add(o, v3_scale(d, temp));                               /* Ray::pointAt  Ray.hh:30-32 */
        v3 gn = v3_divs(v3_sub(p, c), s->radius);                          /* :53,67 */
        v3 sn; uint32_t f;
        check_face(d, gn, &f, &sn);
        float phi = atan2f(gn.z, gn.x);                                    /* sphereUV :19-24 */
        float theta = asinf(gn.y);
        rec->uv[0] = 1 - (phi + ORQ_PI_F) / (2 * ORQ_PI_F);
        rec->uv[1] = (theta + ORQ_PI_2_F) / ORQ_PI_F;
        rec->hit = 1; rec->t = temp; rec->front = f; rec->material = s->material;
        v3_st(rec->p, p); v3_st(rec->gn, gn); v3_st(rec->sn, sn);
    }
    return 1;
}

/* ---------------------------------------------------------------- Square  (Square.hh:60-113) */
int orq_square_hit(const orq_square* s, const float o_[3], const float d_[3], float range[2], orq_record* rec) {
    v3 o = v3_ld(o_), d = v3_ld(d_);
    unsigned ai = s->axis_i, aj = s->axis_j, ak = s->axis_k;
    float t = (s->value_k - v3_get(o, ak)) / v3_get(d, ak);                /* :82 */
    if (isinf(t) || isnan(t)) return 0;                                    /* :84 */
    if (t < range[0] || t > range[1]) return 0;                            /* :85 */
    float a = v3_get(o, ai) + t * v3_get(d, ai);                           /* :87 */
    if (a < s->range_i[0] || a > s->range_i[1]) return 0;
    float b = v3_get(o, aj) + t * v3_get(d, aj);                           /* :90 */
    if (b < s->range_j[0] || b > s->range_j[1]) return 0;
    range[1] = t;                                                          /* :108 */
    if (rec) {
        rec->uv[0] = (a - s->range_i[0]) / (s->range_i[1] - s->range_i[0]); /* :93 */
        rec->uv[1] = (b - s->range_j[0]) / (s->range_j[1] - s->range_j[0]);
        v3 gn = v3_make(0.0f, 0.0f, 0.0f), sn, p = v3_make(0.0f, 0.0f, 0.0f);
        v3_set(&gn, ak, 1.0f);
        uint32_t f;
        check_face(d, gn, &f, &sn);                                        /* :100 */
        gn = sn;                                                           /* :101 */
        v3_set(&p, ak, s->value_k); v3_set(&p, ai, a); v3_set(&p, aj, b);  /* :104-106 */
        rec->hit = 1; rec->t = t; rec->front = f; rec->material = s->material;
        v3_st(rec->p, p); v3_st(rec->gn, gn); v3_st(rec->sn, sn);
    }
    return 1;
}

/* ---------------------------------------------------------------- Cube  (Cube.hh:17-47) */
/* float4x4 * float4 as the shim defines it: ((c0*x + c1*y) + c2*z) + c3*w, per component */
static inline void m4_mul(const float m[16], float x, float y, float z, float w, float out[4]) {
    for (int r = 0; r < 4; ++r)
        out[r] = ((m[0 + r] * x + m[4 + r] * y) + m[8 + r] * z) + m[12 + r] * w;
}

int orq_cube_hit(const orq_cube* c, const float o_[3], const float d_[3], float range[2], orq_record* rec) {
    v3 o = v3_ld(o_), d = v3_ld(d_);
    float lo4[4], ld4[4];
    m4_mul(c->inverse, o.x, o.y, o.z, 1.0f, lo4);                          /* :19 */
    m4_mul(c->inverse, d.x, d.y, d.z, 0.0f, ld4);                          /* :20 */
    v3 lo = v3_make(lo4[0], lo4[1], lo4[2]);
    v3 ld = v3_normalize(v3_make(ld4[0], ld4[1], ld4[2]));                 /* Ray ctor normalises :23 */
    float lt, luv[2]; v3 lp, lgn;
    if (!aabb_hit_record(&c->box, lo, ld, range, &lt, &lp, &lgn, luv)) return 0;   /* :24 */
    float wp4[4];
    m4_mul(c->model, lp.x, lp.y, lp.z, 1.0f, wp4);                         /* :26-27 */
    v3 wp = v3_make(wp4[0], wp4[1], wp4[2]);
    v3 dv = v3_sub(o, wp);
    float t = sqrtf(v3_dot(dv, dv));                                       /* distance :32 */
    if (t >= range[1]) return 0;                                           /* :34 */
    range[1] = t;                                                          /* :36 */
    if (rec) {
        float n4[4];
        m4_mul(c->normal, lgn.x, lgn.y, lgn.z, 0.0f, n4);                  /* :41-42 */
        v3 gn = v3_normalize(v3_make(n4[0], n4[1], n4[2])), sn;
        uint32_t f;
        check_face(d, gn, &f, &sn);                                        /* :43 */
        rec->hit = 1; rec->t = t; rec->front = f; rec->material = c->material;
        rec->uv[0] = luv[0]; rec->uv[1] = luv[1];
        v3_st(rec->p, wp); v3_st(rec->gn, gn); v3_st(rec->sn, sn);
    }
    return 1;
}

/* ---------------------------------------------------------------- offset_ray  (Math.hh:57-74) */
static inline uint32_t f2u(float f) { uint32_t i; memcpy(&i, &f, 4); return i; }
static inline float u2f(uint32_t i) { float f; memcpy(&f, &i, 4); return f; }
/* (int32_t)v as x86 computes it (cvttss2si): truncation, INT32_MIN for NaN and outside [-2^31, 2^31). The cast itself is
 * undefined there in C, so the rule is spelled out. */
static inline int32_t x86_f2i(float v) { return (v != v || v >= 0x1p31f || v < -0x1p31f) ? INT32_MIN : (int32_t)v; }

void orq_offset_ray(const float p[3], const float n[3], float out[3]) {
    const float origin = 1.0f / 32.0f, float_scale = 1.0f / 65536.0f, int_scale = 256.0f;
    for (int k = 0; k < 3; ++k) {
        uint32_t of_i = (uint32_t)x86_f2i(int_scale * n[k]);                /* :64 (truncation) */
        float p_i = u2f(f2u(p[k]) + ((p[k] < 0.0f) ? 0u - of_i : of_i));    /* :66-69, modulo 2^32 */
        out[k] = fabsf(p[k]) < origin ? p[k] + float_scale * n[k] : p_i;   /* :71-73 */
    }
}

void orq_normalize(const float d[3], float out[3]) { v3_st(out, v3_normalize(v3_ld(d))); }   /* Ray.hh:21-23 */

/* ---------------------------------------------------------------- Scene::hit  (Render.hh:135-252) */
int orq_scene_hit(const orq_prims* P, const orq_ray* ray, int any,
                  orq_hit* hit, orq_record* rec_out, orq_counters* cnt_out) {
    const orq_bvh* N = P->bvhList;
    const float o[3] = {ray->ox, ray->oy, ray->oz};
    const float d[3] = {ray->dx, ray->dy, ray->dz};
    const float test_t = ray->tmax;

    uint32_t the_index = 0, tested_index = UINT32_MAX;                     /* :137-138 */
    uint32_t stack_mark = 0, stack_level = 0;                              /* :140-141 */
    float range[2] = {FLT_MIN, test_t};                                    /* :143 */

    orq_counters cnt; memset(&cnt, 0, sizeof cnt);
    orq_record rec; memset(&rec, 0, sizeof rec);
    uint32_t best = UINT32_MAX; float bu = 0.0f, bv = 0.0f;
    int result = 0, early = 0;

    if (orq_aabb_hit(&N[0].bBOX, o, d, range)) {                           /* :145 */
        do {
            uint32_t sel = UINT32_MAX;
            uint32_t l = N[the_index].left, r = N[the_index].right, p = N[the_index].parent;   /* :151-153 */
            if (tested_index != l && tested_index != r) {                  /* :155 came from parent */
                cnt.n_fp++;
                if ((stack_level & 31u) > cnt.max_level) cnt.max_level = stack_level & 31u;
                float tl = range[1], tr = range[1];                        /* :157 */
                int lt = orq_aabb_hit_t(&N[l].bBOX, o, d, range, &tl);     /* :159 */
                int rt = orq_aabb_hit_t(&N[r].bBOX, o, d, range, &tr);     /* :160 */
                if (!lt && !rt) {                                          /* :162-169 */
                    tested_index = the_index; the_index = p; stack_level -= 1;
                    continue;
                }
                if (lt && rt) stack_mark |= 1u << (stack_level & 31u);     /* :171-172 */
                sel = (tl < tr) ? l : r;                                   /* :174 ties -> right */
                if ((sel == l && !lt) || (sel == r && !rt)) cnt.n_quirk++;
            } else {                                                       /* :189 came from child */
                cnt.n_fc++;
                uint32_t need = (stack_mark >> (stack_level & 31u)) & 1u;  /* :191 */
                stack_mark &= ~(1u << (stack_level & 31u));                /* :193 */
                if (need == 0) {                                           /* :195-202 */
                    tested_index = the_index; the_index = p; stack_level -= 1;
                    continue;
                }
                sel = (tested_index == l) ? r : l;                         /* :204-208 */
            }
            cnt.n_disp++;
            uint32_t pIndex = N[sel].pIndex;                               /* :211 */
            float prev = range[1];
            int h = 0;
            switch (N[sel].pType) {                                        /* :213 */
                case ORQ_BVH:
                    the_index = sel; stack_level += 1;                     /* :217-219 */
                    continue;
                case ORQ_SPHERE:
                    cnt.n_sph++;
                    h = orq_sphere_hit(&P->sphereList[pIndex], o, d, range, &rec);
                    if (h) { bu = rec.uv[0]; bv = rec.uv[1]; }
                    break;
                case ORQ_SQUARE:
                    cnt.n_sq++;
                    h = orq_square_hit(&P->squareList[pIndex], o, d, range, &rec);
                    if (h) { bu = rec.uv[0]; bv = rec.uv[1]; }
                    break;
                case ORQ_CUBE:
                    cnt.n_cube++;
                    h = orq_cube_hit(&P->cubeList[pIndex], o, d, range, &rec);
                    if (h) { bu = rec.uv[0]; bv = rec.uv[1]; }
                    break;
                case ORQ_TRIANGLE: {
                    cnt.n_tri++;
                    uint32_t abc[3] = {P->idxList[pIndex * 3], P->idxList[pIndex * 3 + 1], P->idxList[pIndex * 3 + 2]};  /* :232-235 */
                    float bary[2];
                    h = orq_triangle_hit(P->triList, abc, o, d, range, &rec, bary);
                    if (h) { bu = bary[0]; bv = bary[1]; }
                    break;
                }
                default: break;
            }
            if (h) {
                if (best != UINT32_MAX && range[1] == prev) cnt.n_tie++;
                best = sel;
            }
            if (any && range[1] < test_t) { early = 1; break; }            /* :244 */
            tested_index = sel;                                            /* :246 */
        } while (tested_index != 0);                                       /* :248 */
    }
    result = early ? 1 : (range[1] < test_t);                              /* :251 */

    if (hit) {
        memset(hit, 0, sizeof *hit);
        if (result && best != UINT32_MAX) {
            hit->t = rec.t;
            hit->pType = (uint32_t)N[best].pType;
            hit->pIndex = N[best].pIndex;
            hit->leafNode = best;
            hit->u = bu; hit->v = bv;
            hit->material = rec.material;
            hit->flags = 1u | (rec.front ? 2u : 0u);
        }
    }
    if (rec_out) {
        if (result) { *rec_out = rec; rec_out->hit = 1; }
        else memset(rec_out, 0, sizeof *rec_out);
    }
    if (cnt_out) *cnt_out = cnt;
    return result;
}

/* ---------------------------------------------------------------- batch driver */
typedef struct {
    const orq_prims* prims; const orq_ray* rays; uint64_t lo, hi; int any;
    orq_hit* hits; orq_record* recs; orq_counters* cnts; orq_totals tot;
} job_t;

static void* job_main(void* arg) {
    job_t* j = (job_t*)arg;
    memset(&j->tot, 0, sizeof j->tot);
    for (uint64_t i = j->lo; i < j->hi; ++i) {
        orq_counters c;
        orq_scene_hit(j->prims, &j->rays[i], j->any, &j->hits[i], j->recs ? &j->recs[i] : NULL, &c);
        if (j->cnts) j->cnts[i] = c;
        const uint32_t* cv = (const uint32_t*)&c;
        for (int k = 0; k < 9; ++k) j->tot.v[k] += cv[k];
        if (c.max_level > j->tot.v[9]) j->tot.v[9] = c.max_level;
    }
    return NULL;
}

void orq_trace(const orq_prims* prims, const orq_ray* rays, uint64_t n, int any, int nthreads,
               orq_hit* hits, orq_record* recs, orq_counters* cnts, orq_totals* totals) {
    if (nthreads < 1) nthreads = 1;
    if (n < 1024) nthreads = 1;
    job_t* jobs = (job_t*)calloc((size_t)nthreads, sizeof(job_t));
    pthread_t* th = (pthread_t*)calloc((size_t)nthreads, sizeof(pthread_t));
    for (int k = 0; k < nthreads; ++k) {
        jobs[k].prims = prims; jobs[k].rays = rays; jobs[k].any = any;
        jobs[k].lo = n * (uint64_t)k / (uint64_t)nthreads;
        jobs[k].hi = n * (uint64_t)(k + 1) / (uint64_t)nthreads;
        jobs[k].hits = hits; jobs[k].recs = recs; jobs[k].cnts = cnts;
        if (nthreads == 1) job_main(&jobs[k]);
        else pthread_create(&th[k], NULL, job_main, &jobs[k]);
    }
    if (totals) memset(totals, 0, sizeof *totals);
    for (int k = 0; k < nthreads; ++k) {
        if (nthreads > 1) pthread_join(th[k], NULL);
        if (totals) {
            for (int q = 0; q < 9; ++q) totals->v[q] += jobs[k].tot.v[q];
            if (jobs[k].tot.v[9] > totals->v[9]) totals->v[9] = jobs[k].tot.v[9];
        }
    }
    free(jobs); free(th);
}

uint64_t orq_algorithmic_bytes(const orq_totals* t, uint64_t n_rays) {
    /* SURVEY.md section 8(d): 60*N_fp + 12*N_fc + 8*N_disp + 48*N_tri + 16*N_sph + 28 + 20 per ray.
     * Square test reads axes/ranges/value_k/material = 32 B; cube test reads inverse+model matrices
     * and the local box = 160 B (extension for the two leaf types the formula does not list). */
    return 60 * t->v[0] + 12 * t->v[1] + 8 * t->v[2] + 48 * t->v[3] + 16 * t->v[4]
         + 32 * t->v[5] + 160 * t->v[6] + 48 * n_rays;
}
