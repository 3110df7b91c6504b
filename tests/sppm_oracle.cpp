// sppm_oracle.cpp — CPU reference of stochastic progressive photon mapping (include/cgrt.h cgrt_set_sppm) for tests/test_sppm.py.
// TEST INFRASTRUCTURE ONLY. It drives the unchanged PPM oracle (oracle/ppm_oracle.hpp: scene classes, trace(), Hashtable, photon()) and
// adds what SPPM changes: per-pixel statistics, a new Hashtable and eye pass every round with the SPPM camera stream, every visible point
// at its pixel's radius, the per-pixel fold of the round's accumulators, and the image from the pixels. tests/sppm_oracle.py compiles it.
#include "../oracle/ppm_oracle.hpp"

#include <memory>
#ifdef _OPENMP
#include <omp.h>
#endif

using namespace orc;

namespace {

const uint32_t PASS_SPPM_EYE = 3;  // Philox pass of the SPPM camera: (seed, 3, path, dim = round)

struct Sppm {
    Renderer R;
    std::vector<std::unique_ptr<Object>> owned;
    std::vector<Texture> textures;
    int mode = 1;  // 1 jitter, 2 corner
    uint32_t round = 0;
    std::vector<Vec3> tau;
    std::vector<double> r2;
    std::vector<int> n;

    size_t npix() const { return (size_t)R.cfg.width * R.cfg.height; }

    // Camera of eye path `path` in round `round`: jitter ux, uy first (jitter mode), then the lens sample; (w + ux, h + uy) in place of
    // (w, h) in the expressions of main.cpp:188-198.
    static void camera(Renderer &W, int mode, uint32_t round, int w, int h, uint64_t path, Rng &rng) {
        const Config &cfg = W.cfg;
        Rng g = Rng::philox(cfg.seed, PASS_SPPM_EYE, path, round);
        double xs = (double)w, ys = (double)h;
        if (mode == 1) {
            xs = (double)w + g.u01();
            ys = (double)h + g.u01();
        }
        double x = (2.0 * (xs / cfg.width) - 1) * 10.0;
        double y = (2.0 * (ys / cfg.height) - 1) * 10.0 * cfg.height / cfg.width;
        Vec3 dir = (Vec3(x, y, 0) - cfg.camorg).normalize();
        Vec3 org = cfg.camorg;
        if (cfg.use_dof) {
            Vec3 point_on_focus = dir * ((cfg.focus_plane - cfg.camorg.z) / dir.z) + cfg.camorg;
            org = cfg.camorg + uniform_sampling_circle(g, cfg.lens_radius);
            dir = (point_on_focus - org).normalize();
        }
        W.trace(org, dir, Vec3(), Vec3(1, 1, 1), true, 0, w, h, rng, path, 0);
    }

    // A new table and the eye pass of `r`: row blocks traced on `nthreads` threads into sinks, inserted in the reference's creation order
    // (h outer, w inner, samples, DFS), then every visible point takes its pixel's radius.
    void begin_round(uint32_t r, int nthreads) {
        round = r;
        if (R.htable && R.owns_htable) delete R.htable;
        R.htable = new Hashtable(R.cfg.hashsize, 200.0 / R.cfg.height);
        R.owns_htable = true;
        R.next_seq = 0;
        const int H = R.cfg.height, block = 8, nblocks = (H + block - 1) / block;
        std::vector<std::vector<Hitpoint>> sinks((size_t)nblocks);
#ifdef _OPENMP
#pragma omp parallel for schedule(dynamic, 1) num_threads(nthreads > 0 ? nthreads : 1)
#endif
        for (int b = 0; b < nblocks; b++) {
            Renderer w = R.worker();
            w.sink = &sinks[(size_t)b];
            Rng rng = Rng::philox(R.cfg.seed, 0, 0, 0);
            for (int h = b * block; h < H && h < (b + 1) * block; h++)
                for (int x = 0; x < R.cfg.width; x++)
                    for (int j = 0; j < R.cfg.num_of_samples; j++)
                        camera(w, mode, round, x, h, ((uint64_t)h * R.cfg.width + x) * (uint64_t)R.cfg.num_of_samples + j, rng);
        }
        for (auto &sk : sinks)
            for (auto &hp : sk) {
                hp.seq = R.next_seq++;
                hp.r2 = r2[(size_t)hp.h * R.cfg.width + hp.w];
                R.htable->insert(hp);
            }
    }

    // The U2 rule per pixel: the round's accumulators summed per pixel in canonical order (buckets ascending, insertion order inside a
    // bucket), then g = (n a + a M) / (n a + M); tau = (tau + dflux) g; R2 *= g; n += M.
    void fold() {
        std::vector<Vec3> d(npix());
        std::vector<long long> m(npix(), 0);
        for (auto &b : R.htable->hashtable)
            for (auto &hp : b) {
                const size_t p = (size_t)hp.h * R.cfg.width + hp.w;
                d[p] = d[p] + hp.dflux;
                m[p] += hp.m;
                hp.dflux = Vec3();
                hp.m = 0;
            }
        for (size_t p = 0; p < npix(); p++)
            if (m[p] > 0) {
                double na = n[p] * R.cfg.alpha;
                double mm = (double)m[p];
                double g = (na + R.cfg.alpha * mm) / (na + mm);
                tau[p] = (tau[p] + d[p]) * g;
                r2[p] *= g;
                n[p] += (int)m[p];
            }
    }
};

Vec3 v3(const double *p) { return Vec3(p[0], p[1], p[2]); }
void st3(double *p, const Vec3 &v) { p[0] = v.x; p[1] = v.y; p[2] = v.z; }

}  // namespace

extern "C" {

struct sppm_config {  // the fields of oracle.binding.OrcConfig
    int32_t width, height, max_depth, num_of_samples, use_dof, consume_dof_rng, hashsize, update_mode, into_rule, pad;
    double alpha, focus_plane, lens_radius;
    double lightorg[3], camorg[3];
    uint64_t seed;
};

// Pixel statistics start at n = 0, tau = 0, R2 = (200/height)^2.
void *sppm_create(const sppm_config *k, int mode) {
    if (mode != 1 && mode != 2) return nullptr;
    Sppm *s = new Sppm();
    Config &g = s->R.cfg;
    g.width = k->width; g.height = k->height; g.max_depth = k->max_depth; g.num_of_samples = k->num_of_samples;
    g.use_dof = k->use_dof; g.consume_dof_rng = k->consume_dof_rng; g.hashsize = k->hashsize;
    g.update = UPDATE_U2_PER_ROUND; g.into_rule = (IntoRule)k->into_rule;
    g.alpha = k->alpha; g.focus_plane = k->focus_plane; g.lens_radius = k->lens_radius;
    g.lightorg = v3(k->lightorg); g.camorg = v3(k->camorg); g.seed = k->seed;
    s->mode = mode;
    const double r = 200.0 / g.height;
    s->tau.assign(s->npix(), Vec3());
    s->r2.assign(s->npix(), r * r);
    s->n.assign(s->npix(), 0);
    return s;
}
void sppm_destroy(void *s) { delete (Sppm *)s; }

int sppm_add_texture(void *s_, const uint8_t *rgb, int w, int h, const double *n, const double *p, double lenx, double leny, int isbump) {
    Sppm *s = (Sppm *)s_;
    std::vector<Vec3> d((size_t)w * h);
    for (size_t i = 0; i < d.size(); i++)  // main.cpp:303-316
        d[i] = Vec3((double)rgb[3 * i] / (double)256, (double)rgb[3 * i + 1] / (double)256, (double)rgb[3 * i + 2] / (double)256);
    s->textures.push_back(Texture(d, h, w, v3(n), v3(p), lenx, leny, isbump != 0));
    return (int)s->textures.size() - 1;
}
int sppm_add_sphere(void *s_, const double *c, double r, const double *col, double refl, double transp) {
    Sppm *s = (Sppm *)s_;
    s->owned.emplace_back(new Sphere(v3(c), r, v3(col), refl, transp));
    s->R.objs.push_back(s->owned.back().get());
    return (int)s->R.objs.size() - 1;
}
int sppm_add_plane(void *s_, const double *p, const double *n, const double *col, double refl, double transp, int tex) {
    Sppm *s = (Sppm *)s_;
    s->owned.emplace_back(new Plane(v3(p), v3(n), v3(col), refl, transp, tex >= 0 ? s->textures[tex] : Texture()));
    s->R.objs.push_back(s->owned.back().get());
    return (int)s->R.objs.size() - 1;
}
int sppm_add_mesh(void *s_, const double *tri9, int ntri, const double *col, double refl, double transp, int objtype) {
    Sppm *s = (Sppm *)s_;
    std::vector<Triangle> t((size_t)ntri);
    for (int i = 0; i < ntri; i++) t[i] = Triangle(v3(tri9 + 9 * i), v3(tri9 + 9 * i + 3), v3(tri9 + 9 * i + 6));
    s->owned.emplace_back(new TriangleMesh(t, v3(col), refl, transp, objtype));
    s->R.objs.push_back(s->owned.back().get());
    return (int)s->R.objs.size() - 1;
}
int sppm_add_bezier(void *s_, const double *cp3, int ncp, const double *pos, const double *col, double refl, double transp) {
    Sppm *s = (Sppm *)s_;
    std::vector<Vec3> cp;
    for (int i = 0; i < ncp; i++) cp.push_back(v3(cp3 + 3 * i));
    s->owned.emplace_back(new Bezier(cp, v3(pos), v3(col), refl, transp));
    s->R.objs.push_back(s->owned.back().get());
    return (int)s->R.objs.size() - 1;
}

int sppm_begin_round(void *s_, uint32_t round, int nthreads) {
    ((Sppm *)s_)->begin_round(round, nthreads);
    return 0;
}

// Photons with global indices [first, first+count) into the round's accumulators (the oracle's photon(), atomics under OpenMP).
int sppm_photon_pass(void *s_, uint64_t first, uint64_t count, int nthreads) {
    Sppm *s = (Sppm *)s_;
    if (!s->R.htable) return -1;
#ifdef _OPENMP
#pragma omp parallel num_threads(nthreads > 0 ? nthreads : 1)
    {
        Renderer w = s->R.worker();
        Rng rng = Rng::philox(s->R.cfg.seed, PASS_PHOTON, 0, 0);
#pragma omp for schedule(dynamic, 4096)
        for (int64_t i = 0; i < (int64_t)count; i++) w.photon(rng, first + (uint64_t)i);
    }
#else
    (void)nthreads;
    Rng rng = Rng::philox(s->R.cfg.seed, PASS_PHOTON, 0, 0);
    for (uint64_t i = 0; i < count; i++) s->R.photon(rng, first + i);
#endif
    return 0;
}

int sppm_fold(void *s_) {
    Sppm *s = (Sppm *)s_;
    if (!s->R.htable) return -1;
    s->fold();
    return 0;
}

int64_t sppm_num_visible(void *s_) {
    Sppm *s = (Sppm *)s_;
    int64_t k = 0;
    if (s->R.htable)
        for (auto &b : s->R.htable->hashtable) k += (int64_t)b.size();
    return k;
}
// The round's visible points in canonical order (buckets ascending, insertion order inside a bucket). Any pointer may be NULL.
int sppm_download_visible(void *s_, double *pos, double *r2, int32_t *hw, uint32_t *key, double *dflux, int32_t *m) {
    Sppm *s = (Sppm *)s_;
    if (!s->R.htable) return 0;
    size_t i = 0;
    for (size_t b = 0; b < s->R.htable->hashtable.size(); b++)
        for (const Hitpoint &hp : s->R.htable->hashtable[b]) {
            if (pos) st3(pos + 3 * i, hp.pos);
            if (r2) r2[i] = hp.r2;
            if (hw) { hw[2 * i] = hp.h; hw[2 * i + 1] = hp.w; }
            if (key) key[i] = (uint32_t)b;
            if (dflux) st3(dflux + 3 * i, hp.dflux);
            if (m) m[i] = hp.m;
            i++;
        }
    return 0;
}
int sppm_download_pixels(void *s_, double *tau, double *r2, int32_t *n) {
    Sppm *s = (Sppm *)s_;
    for (size_t p = 0; p < s->npix(); p++) {
        if (tau) st3(tau + 3 * p, s->tau[p]);
        if (r2) r2[p] = s->r2[p];
        if (n) n[p] = s->n[p];
    }
    return 0;
}
// main.cpp:252-258 with the pixel's statistics; n_emitted = photons traced so far, the num_of_samples factor comes from the config.
int sppm_gather_image(void *s_, double n_emitted, double *rgb) {
    Sppm *s = (Sppm *)s_;
    const double ne = n_emitted * (double)s->R.cfg.num_of_samples;
    for (size_t p = 0; p < s->npix(); p++) st3(rgb + 3 * p, Vec3() + s->tau[p] * (1.0 / (PI * s->r2[p] * ne)));
    return 0;
}

}  // extern "C"
