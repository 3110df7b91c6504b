// oracle_capi.cpp — C API over the CPU oracle (oracle/ppm_oracle.hpp) for ctypes.
// TEST INFRASTRUCTURE ONLY: used by tests/, __graft_entry__.smoke() and bench.py's CPU-baseline legs.
// The scene-building entry points mirror include/cgrt.h one for one (orc_ prefix instead of cgrt_) so
// the parity tests feed the same description to both sides.
#include "ppm_oracle.hpp"

#include <chrono>
#include <memory>
#ifdef _OPENMP
#include <omp.h>
#endif

using namespace orc;

namespace {

// The deterministic 31-bit stream shared with oracle/ref_driver.cpp (there it replaces rand()).
struct SplitMix {
    uint64_t s;
    int next31() {
        uint64_t z = (s += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        z = z ^ (z >> 31);
        return (int)(z >> 33);
    }
};
int splitmix_cb(void *st) { return ((SplitMix *)st)->next31(); }

const uint32_t PASS_SPPM_EYE = 3;  // Philox pass of the SPPM camera: (seed, 3, path, dim = round)

struct Ctx {
    Renderer R;
    std::vector<std::unique_ptr<Object>> owned;
    std::vector<Texture> textures;
    SplitMix libc_stream{1};
    bool libc_mode = false;
    Rng make_rng() { return libc_mode ? Rng::external(splitmix_cb, &libc_stream) : Rng::philox(R.cfg.seed, 0, 0, 0); }
    std::vector<const Hitpoint *> canon;  // hitpoints in canonical (bucket-major, insertion) order
    void index() {
        canon.clear();
        if (!R.htable) return;
        for (auto &b : R.htable->hashtable)
            for (auto &hp : b) canon.push_back(&hp);
    }

    // Stochastic PPM (orc_set_sppm): the camera mode (0 off, 1 jitter, 2 corner), the statistics per pixel, and the visible points of a
    // split round's eye pass, which wait in `pending` (open from orc_sppm_eye_pass until orc_build_grid inserts them).
    int sppm = 0;
    std::vector<Vec3> tau;
    std::vector<double> r2;
    std::vector<int> n;
    std::vector<Hitpoint> pending;
    bool pending_open = false;
    size_t npix() const { return (size_t)R.cfg.width * R.cfg.height; }
    size_t pixel(const Hitpoint &hp) const { return (size_t)hp.h * R.cfg.width + hp.w; }

    // The U2 rule per pixel: the round's accumulators summed per pixel in canonical order (buckets ascending, insertion order inside a
    // bucket), then g = (n a + a M) / (n a + M); tau = (tau + dflux) g; R2 *= g; n += M.
    void fold() {
        std::vector<Vec3> d(npix());
        std::vector<long long> m(npix(), 0);
        for (auto &b : R.htable->hashtable)
            for (auto &hp : b) {
                const size_t p = pixel(hp);
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

void new_table(Renderer &R) {
    if (R.htable && R.owns_htable) delete R.htable;
    R.htable = new Hashtable(R.cfg.hashsize, 200.0 / R.cfg.height);
    R.owns_htable = true;
}

// Rows [y0, y1) of an eye pass in blocks of 8 rows on `nthreads` OpenMP threads: trace_rows(worker, rng, r0, r1) appends a block's
// hitpoints to its own sink in creation order. Philox mode only: every path re-keys its own stream, so the result does not depend on
// who traces a block. Returns the sinks in row order; the workers' eye counters are added to R's.
template <class TraceRows>
std::vector<std::vector<Hitpoint>> eye_blocks(Renderer &R, int y0, int y1, int nthreads, TraceRows trace_rows) {
    const int block = 8, nblocks = y1 > y0 ? (y1 - y0 + block - 1) / block : 0;
    std::vector<std::vector<Hitpoint>> sinks((size_t)nblocks);
    std::vector<Counters> part((size_t)nblocks);
    std::vector<KDCounters> kpart((size_t)nblocks);
#ifdef _OPENMP
#pragma omp parallel for schedule(dynamic, 1) num_threads(nthreads > 0 ? nthreads : 1)
#endif
    for (int b = 0; b < nblocks; b++) {
        Renderer w = R.worker();
        w.sink = &sinks[(size_t)b];
        Rng rng = Rng::philox(R.cfg.seed, 0, 0, 0);
        const int r0 = y0 + b * block;
        trace_rows(w, rng, r0, std::min(r0 + block, y1));
        part[(size_t)b] = w.ctr;
        kpart[(size_t)b] = w.kdc;
    }
    for (auto &kp : kpart) { R.kdc.node_visits += kp.node_visits; R.kdc.tri_tests += kp.tri_tests; }
    for (auto &p : part) { R.ctr.eye_segments += p.eye_segments; R.ctr.misses += p.misses; }
    return sinks;
}

// The SPPM camera of eye path `path` in round `round`: jitter ux, uy first (jitter mode), then the lens sample; (w + ux, h + uy) in place of
// (w, h) in the expressions of main.cpp:188-198.
void sppm_camera(Renderer &W, int mode, uint32_t round, int w, int h, uint64_t path, Rng &rng) {
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

// A new, empty table and SPPM round `round`'s eye pass over rows [y0, y1); returns the row blocks' visible points (eye_blocks).
std::vector<std::vector<Hitpoint>> sppm_trace(Ctx *c, uint32_t round, int y0, int y1, int nthreads) {
    new_table(c->R);
    c->R.next_seq = 0;
    c->pending.clear();
    c->pending_open = false;
    const int mode = c->sppm;
    return eye_blocks(c->R, y0, y1, nthreads, [mode, round](Renderer &w, Rng &rng, int r0, int r1) {
        const Config &g = w.cfg;
        for (int h = r0; h < r1; h++)
            for (int x = 0; x < g.width; x++)
                for (int j = 0; j < g.num_of_samples; j++)
                    sppm_camera(w, mode, round, x, h, ((uint64_t)h * g.width + x) * (uint64_t)g.num_of_samples + j, rng);
    });
}

// The exchange record of the GPU path (cgrt_export_hitpoints_dev, include/cgrt.h), 12 doubles: pos, normal, f, bits(sort key),
// bits(h << 32 | w), 0. The sort key key << 32 | path*16 + code orders a hitpoint set canonically (buckets ascending, then creation order).
uint64_t sort_key(const Hashtable &ht, const Hitpoint &hp) {
    int ix, iy, iz;
    ht.compute_coord(hp.pos.x, hp.pos.y, hp.pos.z, ix, iy, iz);
    return ((uint64_t)ht.hash(ix, iy, iz) << 32) | (uint64_t)(uint32_t)(hp.path * 16u + (hp.code & 15u));
}
void put_record(const Hashtable &ht, const Hitpoint &hp, double *r) {
    st3(r, hp.pos); st3(r + 3, hp.normal); st3(r + 6, hp.f);
    uint64_t sk = sort_key(ht, hp);
    uint64_t hw = ((uint64_t)(uint32_t)hp.h << 32) | (uint64_t)(uint32_t)hp.w;
    memcpy(r + 9, &sk, 8); memcpy(r + 10, &hw, 8); r[11] = 0.0;
}
// -> the hitpoint of record q (pos, normal, f, pixel, path, code; every other field as constructed) and its sort key.
Hitpoint get_record(const double *q, uint64_t &sk) {
    uint64_t hw;
    memcpy(&sk, q + 9, 8); memcpy(&hw, q + 10, 8);
    Hitpoint hp;
    hp.pos = v3(q); hp.normal = v3(q + 3); hp.f = v3(q + 6);
    hp.h = (int)(hw >> 32); hp.w = (int)(uint32_t)hw;
    uint32_t lo = (uint32_t)sk;
    hp.code = lo & 15u; hp.path = lo >> 4;
    return hp;
}

// Inserts hitpoints with sort keys `sk` into R's table in canonical order: stable sort on the key, seq = sorted position.
void insert_sorted(Renderer &R, std::vector<Hitpoint> &hps, const std::vector<uint64_t> &sk) {
    std::vector<size_t> order(hps.size());
    for (size_t i = 0; i < order.size(); i++) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&sk](size_t a, size_t b) { return sk[a] < sk[b]; });
    uint32_t seq = 0;
    for (size_t i : order) {
        hps[i].seq = seq++;
        R.htable->insert(hps[i]);
    }
}

}  // namespace

extern "C" {

struct orc_config {  // keep in sync with OrcConfig in oracle/binding.py
    int32_t width, height, max_depth, num_of_samples, use_dof, consume_dof_rng, hashsize, update_mode, into_rule, pad;
    double alpha, focus_plane, lens_radius;
    double lightorg[3], camorg[3];
    uint64_t seed;
};

struct orc_counters {
    uint64_t eye_segments, photon_segments, diffuse_hits, bucket_probes, nonempty_probes, candidates, deposits, misses;
    uint64_t node_visits, tri_tests;
};

void *orc_create() { return new Ctx(); }
void orc_destroy(void *c) { delete (Ctx *)c; }

int orc_set_config(void *c_, const orc_config *k) {
    Ctx *c = (Ctx *)c_;
    Config &g = c->R.cfg;
    g.width = k->width; g.height = k->height; g.max_depth = k->max_depth; g.num_of_samples = k->num_of_samples;
    g.use_dof = k->use_dof; g.consume_dof_rng = k->consume_dof_rng; g.hashsize = k->hashsize;
    g.update = (UpdateMode)k->update_mode; g.into_rule = (IntoRule)k->into_rule;
    g.alpha = k->alpha; g.focus_plane = k->focus_plane; g.lens_radius = k->lens_radius;
    g.lightorg = v3(k->lightorg); g.camorg = v3(k->camorg); g.seed = k->seed;
    return 0;
}

// libc-compat random stream (pins the oracle against oracle/_ref): mode=1 on, seed selects the stream.
int orc_set_libc_rng(void *c_, int on, uint64_t seed) {
    Ctx *c = (Ctx *)c_;
    c->libc_mode = on != 0;
    c->libc_stream.s = seed;
    return 0;
}

int orc_add_texture(void *c_, const uint8_t *rgb, int w, int h, const double *n, const double *p, double lenx, double leny, int isbump) {
    Ctx *c = (Ctx *)c_;
    std::vector<Vec3> d((size_t)w * h);
    for (size_t i = 0; i < d.size(); i++)  // main.cpp:303-316
        d[i] = Vec3((double)rgb[3 * i] / (double)256, (double)rgb[3 * i + 1] / (double)256, (double)rgb[3 * i + 2] / (double)256);
    c->textures.push_back(Texture(d, h, w, v3(n), v3(p), lenx, leny, isbump != 0));
    return (int)c->textures.size() - 1;
}
int orc_add_sphere(void *c_, const double *ctr, double r, const double *col, double refl, double transp) {
    Ctx *c = (Ctx *)c_;
    c->owned.emplace_back(new Sphere(v3(ctr), r, v3(col), refl, transp));
    c->R.objs.push_back(c->owned.back().get());
    return (int)c->R.objs.size() - 1;
}
int orc_add_plane(void *c_, const double *p, const double *n, const double *col, double refl, double transp, int tex_id) {
    Ctx *c = (Ctx *)c_;
    c->owned.emplace_back(new Plane(v3(p), v3(n), v3(col), refl, transp, tex_id >= 0 ? c->textures[tex_id] : Texture()));
    c->R.objs.push_back(c->owned.back().get());
    return (int)c->R.objs.size() - 1;
}
int orc_add_mesh(void *c_, const double *tri9, int ntri, const double *col, double refl, double transp, int objtype) {
    Ctx *c = (Ctx *)c_;
    std::vector<Triangle> t((size_t)ntri);
    for (int i = 0; i < ntri; i++) t[i] = Triangle(v3(tri9 + 9 * i), v3(tri9 + 9 * i + 3), v3(tri9 + 9 * i + 6));
    c->owned.emplace_back(new TriangleMesh(t, v3(col), refl, transp, objtype));
    c->R.objs.push_back(c->owned.back().get());
    return (int)c->R.objs.size() - 1;
}
int orc_add_bezier(void *c_, const double *cp3, int ncp, const double *pos, const double *col, double refl, double transp) {
    Ctx *c = (Ctx *)c_;
    std::vector<Vec3> cp;
    for (int i = 0; i < ncp; i++) cp.push_back(v3(cp3 + 3 * i));
    c->owned.emplace_back(new Bezier(cp, v3(pos), v3(col), refl, transp));
    c->R.objs.push_back(c->owned.back().get());
    return (int)c->R.objs.size() - 1;
}

// objects.h:338-403 loaders: returns the triangle count; tri9 may be NULL to query the size.
int orc_load_mesh_text(const char *filename, int typeofdata, double a, const double *b, double *tri9, int cap) {
    std::vector<Triangle> t;
    if (!load_mesh_text(filename, typeofdata, a, v3(b), t)) return -1;
    if (tri9) {
        int n = std::min((int)t.size(), cap);
        for (int i = 0; i < n; i++) { st3(tri9 + 9 * i, t[i].pa); st3(tri9 + 9 * i + 3, t[i].pb); st3(tri9 + 9 * i + 6, t[i].pc); }
    }
    return (int)t.size();
}

// Number of triangles in the displaced height-field of plane `obj` (0 if none), and its triangles.
int orc_bump_triangles(void *c_, int obj, double *tri9, int cap) {
    Ctx *c = (Ctx *)c_;
    Plane *p = dynamic_cast<Plane *>(c->R.objs[obj]);
    if (!p) return -1;
    const auto &t = p->bumpmapping.tris;
    if (tri9) {
        int n = std::min((int)t.size(), cap);
        for (int i = 0; i < n; i++) { st3(tri9 + 9 * i, t[i].pa); st3(tri9 + 9 * i + 3, t[i].pb); st3(tri9 + 9 * i + 6, t[i].pc); }
    }
    return (int)t.size();
}

// ---- unit-level parity hooks -------------------------------------------------------------------------------------

// hash.h:22-42 on free-standing positions. celllength_in is the ctor argument (e.g. 200/height).
int orc_hash_keys(int64_t n, const double *pos, int hashsize, double celllength_in, uint32_t *key, int32_t *ixyz) {
    Hashtable ht(hashsize, celllength_in, false);
    for (int64_t i = 0; i < n; i++) {
        int ix, iy, iz;
        ht.compute_coord(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2], ix, iy, iz);
        if (ixyz) { ixyz[3 * i] = ix; ixyz[3 * i + 1] = iy; ixyz[3 * i + 2] = iz; }
        key[i] = ht.hash(ix, iy, iz);
    }
    return 0;
}
uint32_t orc_hash(int ix, int iy, int iz, int hashsize) { Hashtable ht(hashsize, 1.0, false); return ht.hash(ix, iy, iz); }
int orc_grid_params(int hashsize, double celllength_in, int *cells, double *celllength) {
    Hashtable ht(hashsize, celllength_in, false);
    *cells = ht.num_of_cell_per_dim; *celllength = ht.celllength;
    return 0;
}

// main.cpp:50-76 closest hit over the whole scene for a batch of rays. obj=-1 on miss.
// nrm = face-forwarded normal, nrm_raw = what Object::intersect returned. Bezier draws come from a per-ray stream.
int orc_intersect_batch(void *c_, int64_t n, const double *org, const double *dir, double *t, double *nrm, double *nrm_raw,
                        int32_t *obj, int32_t *into, int32_t *prim) {
    Ctx *c = (Ctx *)c_;
    Rng rng = c->make_rng();
    for (int64_t i = 0; i < n; i++) {
        TraceCtx tc;
        tc.into_rule = c->R.cfg.into_rule;
        Rng brng = rng;
        if (!c->libc_mode) brng.reseed(c->R.cfg.seed, PASS_BEZIER, (uint64_t)i, 0);
        tc.rng = c->libc_mode ? &rng : &brng;
        HitRecord hr;
        bool hit = c->R.closest_hit(v3(org + 3 * i), v3(dir + 3 * i), hr, tc);
        obj[i] = hit ? hr.id : -1;
        if (t) t[i] = hit ? hr.t : 0.0;
        if (nrm) st3(nrm + 3 * i, hit ? hr.n_ff : Vec3());
        if (nrm_raw) st3(nrm_raw + 3 * i, hit ? hr.n_raw : Vec3());
        if (into) into[i] = hit ? hr.into : 0;
        if (prim) prim[i] = hit ? hr.prim : -1;
    }
    return 0;
}

// Per-object Object::intersect (raw normal), for pinning each primitive against the reference classes.
int orc_object_intersect(void *c_, int objid, int64_t n, const double *org, const double *dir, int32_t *hit, double *len, double *nrm) {
    Ctx *c = (Ctx *)c_;
    Rng rng = c->make_rng();
    TraceCtx tc;
    tc.into_rule = c->R.cfg.into_rule;
    tc.rng = &rng;
    for (int64_t i = 0; i < n; i++) {
        double l = 0; Vec3 nv;
        bool h = c->R.objs[objid]->intersect(v3(org + 3 * i), v3(dir + 3 * i), l, nv, &tc);
        hit[i] = h; len[i] = h ? l : 0.0; st3(nrm + 3 * i, h ? nv : Vec3());
    }
    return 0;
}

// Brute-force closest triangle of a mesh object / bump plane (property test: tree == brute force).
int orc_mesh_brute(void *c_, int objid, int64_t n, const double *org, const double *dir, int32_t *hit, double *len, int32_t *tri) {
    Ctx *c = (Ctx *)c_;
    const KDTree *kd = nullptr;
    if (auto *m = dynamic_cast<TriangleMesh *>(c->R.objs[objid])) kd = &m->kdtree;
    else if (auto *p = dynamic_cast<Plane *>(c->R.objs[objid])) kd = &p->bumpmapping;
    if (!kd) return -1;
    for (int64_t i = 0; i < n; i++) {
        double l = 0; Vec3 nv; int id = -1;
        bool h = kd->intersect_brute(v3(org + 3 * i), v3(dir + 3 * i), l, nv, &id);
        hit[i] = h; len[i] = h ? l : 0.0; tri[i] = h ? id : -1;
    }
    return 0;
}

int orc_surface_color(void *c_, int objid, int64_t n, const double *pos, double *col) {
    Ctx *c = (Ctx *)c_;
    for (int64_t i = 0; i < n; i++) st3(col + 3 * i, c->R.objs[objid]->getSurfaceColor(v3(pos + 3 * i)));
    return 0;
}
int orc_texture_color(void *c_, int tex, int64_t n, const double *pos, int32_t *hit, double *col, int32_t *rowcol) {
    Ctx *c = (Ctx *)c_;
    for (int64_t i = 0; i < n; i++) {
        Vec3 cl; int r = -1, cc = -1;
        bool h = c->textures[tex].color(v3(pos + 3 * i), cl, &r, &cc);
        hit[i] = h; st3(col + 3 * i, h ? cl : Vec3());
        if (rowcol) { rowcol[2 * i] = r; rowcol[2 * i + 1] = cc; }
    }
    return 0;
}
double orc_texture_height(void *c_, int tex, int i, int j) {
    Ctx *c = (Ctx *)c_;
    return c->textures[tex].height[(size_t)i * c->textures[tex].W + j];
}

// Bezier known-answer hooks (bezier.h:127-162, 215-224): what = 0 valueP(u), 1 gradP(u), 2 funcValue, 3 normalvec(paras),
// 4..6 gradValue columns.
int orc_bezier_eval(void *c_, int objid, int what, const double *paras, const double *org, const double *dir, double *out) {
    Ctx *c = (Ctx *)c_;
    Bezier *b = dynamic_cast<Bezier *>(c->R.objs[objid]);
    if (!b) return -1;
    Vec3 ra, rb, rc;
    switch (what) {
        case 0: st3(out, b->valueP(paras[1])); break;
        case 1: st3(out, b->gradP(paras[1])); break;
        case 2: st3(out, b->funcValue(v3(paras), v3(org), v3(dir))); break;
        case 3: st3(out, b->normalvec(v3(paras))); break;
        default:
            b->gradValue(v3(paras), v3(org), v3(dir), ra, rb, rc);
            st3(out, what == 4 ? ra : what == 5 ? rb : rc);
    }
    return 0;
}

int orc_gamma_corr(int64_t n, const double *x, int32_t *out) {
    for (int64_t i = 0; i < n; i++) out[i] = gammaCorr(x[i]);
    return 0;
}
int orc_det_inv(const double *a, const double *b, const double *c, double *d, double *inv9) {
    Vec3 ra, rb, rc;
    *d = det(v3(a), v3(b), v3(c));
    bool ok = inv(v3(a), v3(b), v3(c), ra, rb, rc);
    if (ok) { st3(inv9, ra); st3(inv9 + 3, rb); st3(inv9 + 6, rc); }
    return ok;
}
int orc_philox(const uint32_t *ctr, const uint32_t *key, uint32_t *out) { philox4x32_10(ctr, key, out); return 0; }

// The Philox sampling definitions shared with the GPU: what = 0 sphere, 1 halfsphere(about aux), 2 circle(radius aux[0]), 3 u01 x3.
int orc_sample(uint64_t seed, uint32_t pass, uint64_t path, uint32_t dim, int what, const double *aux, double *out) {
    Rng r = Rng::philox(seed, pass, path, dim);
    switch (what) {
        case 0: st3(out, uniform_sampling_sphere(r)); break;
        case 1: st3(out, uniform_sampling_halfsphere(r, v3(aux))); break;
        case 2: st3(out, uniform_sampling_circle(r, aux[0])); break;
        default: out[0] = r.u01(); out[1] = r.u01(); out[2] = r.u01();
    }
    return 0;
}

// ---- passes --------------------------------------------------------------------------------------------------------

// main.cpp:42 — one top-level trace() call (depth 0) on the context's hash table; creates the table on first use.
int orc_trace(void *c_, const double *org, const double *dir, const double *flux, const double *adj, int flag, int x, int y, uint64_t path) {
    Ctx *c = (Ctx *)c_;
    if (!c->R.htable) c->R.htable = new Hashtable(c->R.cfg.hashsize, 200.0 / c->R.cfg.height);
    Rng rng = c->make_rng();
    c->R.trace(v3(org), v3(dir), v3(flux), v3(adj), flag != 0, 0, x, y, rng, path, 0);
    return 0;
}

int orc_eye_pass(void *c_, int y0, int y1) {
    Ctx *c = (Ctx *)c_;
    Rng rng = c->make_rng();
    c->R.eye_pass(rng, y0, y1);
    c->index();
    return 0;
}
// The same eye pass with the rows traced by `nthreads` threads (eye_blocks, Philox mode only). The blocks are inserted in row order with
// consecutive sequence numbers — exactly the table the sequential loop of main.cpp:185-219 builds.
int orc_eye_pass_mt(void *c_, int y0, int y1, int nthreads) {
    Ctx *c = (Ctx *)c_;
    if (c->libc_mode || nthreads <= 1) return orc_eye_pass(c_, y0, y1);
    Renderer &R = c->R;
    if (y1 < 0) y1 = R.cfg.height;
    if (!R.htable) R.htable = new Hashtable(R.cfg.hashsize, 200.0 / R.cfg.height);
    for (auto &sk : eye_blocks(R, y0, y1, nthreads, [](Renderer &w, Rng &rng, int r0, int r1) { w.eye_pass(rng, r0, r1); })) {
        for (auto &hp : sk) { hp.seq = R.next_seq++; R.htable->insert(hp); }
        std::vector<Hitpoint>().swap(sk);
    }
    c->index();
    return 0;
}

// ---- stochastic PPM (include/cgrt.h cgrt_set_sppm): a new eye pass every round, statistics per pixel -------------------------------
// A round is orc_sppm_begin_round, or the split round of several ranks: orc_sppm_eye_pass (a row tile) -> orc_export_hitpoints /
// orc_import_hitpoints (the union of the tiles) -> orc_build_grid; then orc_photon_pass -> orc_round_update (the per-pixel fold).

// mode 0 off, 1 jitter, 2 corner; after orc_set_config. Resets the pixel statistics to tau = 0, R2 = (200/height)^2, n = 0.
// Returns -1 for a bad mode, -2 when the config's update is not per round (U2).
int orc_set_sppm(void *c_, int mode) {
    Ctx *c = (Ctx *)c_;
    if (mode < 0 || mode > 2) return -1;
    if (mode && c->R.cfg.update != UPDATE_U2_PER_ROUND) return -2;
    c->sppm = mode;
    const double r = 200.0 / c->R.cfg.height;
    c->tau.assign(c->npix(), Vec3());
    c->r2.assign(c->npix(), r * r);
    c->n.assign(c->npix(), 0);
    c->pending.clear();
    c->pending_open = false;
    return 0;
}
// A new table and round `round`'s eye pass; the visible points inserted in the reference's creation order (h outer, w inner, samples,
// DFS), every one at its pixel's R2.
int orc_sppm_begin_round(void *c_, uint32_t round, int nthreads) {
    Ctx *c = (Ctx *)c_;
    if (!c->sppm) return -1;
    Renderer &R = c->R;
    for (auto &sk : sppm_trace(c, round, 0, R.cfg.height, nthreads))
        for (auto &hp : sk) {
            hp.seq = R.next_seq++;
            hp.r2 = c->r2[c->pixel(hp)];
            R.htable->insert(hp);
        }
    c->index();
    return 0;
}
// A new, empty table and round `round`'s eye pass over rows [y0, y1) (y1 < 0: to the last row) into the pending visible points, in
// creation order. Nothing is inserted until orc_build_grid.
int orc_sppm_eye_pass(void *c_, uint32_t round, int y0, int y1, int nthreads) {
    Ctx *c = (Ctx *)c_;
    if (y1 < 0) y1 = c->R.cfg.height;
    if (!c->sppm || y0 < 0 || y1 > c->R.cfg.height || y0 > y1) return -1;
    for (auto &sk : sppm_trace(c, round, y0, y1, nthreads)) c->pending.insert(c->pending.end(), sk.begin(), sk.end());
    c->pending_open = true;
    c->index();
    return 0;
}
// SPPM: the pending visible points into the round's table in canonical order, every one at its pixel's R2. PPM: nothing to do, the eye
// pass filled the table.
int orc_build_grid(void *c_) {
    Ctx *c = (Ctx *)c_;
    if (!c->sppm) return 0;
    if (!c->pending_open) return -1;
    std::vector<uint64_t> sk(c->pending.size());
    for (size_t i = 0; i < sk.size(); i++) {
        c->pending[i].r2 = c->r2[c->pixel(c->pending[i])];
        sk[i] = sort_key(*c->R.htable, c->pending[i]);
    }
    insert_sorted(c->R, c->pending, sk);
    c->pending.clear();
    c->pending_open = false;
    c->index();
    return 0;
}
int orc_sppm_download_pixels(void *c_, double *tau, double *r2, int32_t *n) {
    Ctx *c = (Ctx *)c_;
    for (size_t p = 0; p < c->npix(); p++) {
        if (tau) st3(tau + 3 * p, c->tau[p]);
        if (r2) r2[p] = c->r2[p];
        if (n) n[p] = c->n[p];
    }
    return 0;
}

int64_t orc_num_hitpoints(void *c_) { Ctx *c = (Ctx *)c_; c->index(); return (int64_t)c->canon.size(); }

// Canonical order (buckets ascending, insertion order inside a bucket; main.cpp:252-254). Any pointer may be NULL.
int orc_download_hitpoints(void *c_, double *pos, double *normal, double *f, double *flux, double *r2, int32_t *n, int32_t *hw,
                           uint32_t *key, uint32_t *seq, uint32_t *code, uint64_t *path) {
    Ctx *c = (Ctx *)c_;
    c->index();
    for (size_t i = 0; i < c->canon.size(); i++) {
        const Hitpoint &hp = *c->canon[i];
        if (pos) st3(pos + 3 * i, hp.pos);
        if (normal) st3(normal + 3 * i, hp.normal);
        if (f) st3(f + 3 * i, hp.f);
        if (flux) st3(flux + 3 * i, hp.flux);
        if (r2) r2[i] = hp.r2;
        if (n) n[i] = hp.n;
        if (hw) { hw[2 * i] = hp.h; hw[2 * i + 1] = hp.w; }
        if (key) {
            int ix, iy, iz;
            c->R.htable->compute_coord(hp.pos.x, hp.pos.y, hp.pos.z, ix, iy, iz);
            key[i] = c->R.htable->hash(ix, iy, iz);
        }
        if (seq) seq[i] = hp.seq;
        if (code) code[i] = hp.code;
        if (path) path[i] = hp.path;
    }
    return 0;
}
// Per-round accumulators (U2) in canonical order, before orc_round_update clears them.
int orc_download_accum(void *c_, double *dflux, int32_t *m) {
    Ctx *c = (Ctx *)c_;
    c->index();
    for (size_t i = 0; i < c->canon.size(); i++) {
        if (dflux) st3(dflux + 3 * i, c->canon[i]->dflux);
        if (m) m[i] = c->canon[i]->m;
    }
    return 0;
}

// Test plumbing for the 2-rank (gloo) sharding tests: write back all-reduced accumulators, and move hitpoint sets
// between oracle instances in the GPU path's record format (put_record / get_record).
int orc_upload_accum(void *c_, const double *dflux, const int32_t *m) {
    Ctx *c = (Ctx *)c_;
    c->index();
    for (size_t i = 0; i < c->canon.size(); i++) {
        Hitpoint *hp = const_cast<Hitpoint *>(c->canon[i]);
        if (dflux) hp->dflux = v3(dflux + 3 * i);
        if (m) hp->m = m[i];
    }
    return 0;
}
// The table in canonical order; under SPPM, while a split round's eye pass is open, its pending visible points. rec12 NULL: count only.
int64_t orc_export_hitpoints(void *c_, double *rec12) {
    Ctx *c = (Ctx *)c_;
    if (c->pending_open) {
        for (size_t i = 0; rec12 && i < c->pending.size(); i++) put_record(*c->R.htable, c->pending[i], rec12 + 12 * i);
        return (int64_t)c->pending.size();
    }
    c->index();
    for (size_t i = 0; rec12 && i < c->canon.size(); i++) put_record(*c->R.htable, *c->canon[i], rec12 + 12 * i);
    return (int64_t)c->canon.size();
}
// Replaces the hitpoint set: records in any order are inserted in canonical order (stable sort on the 64-bit sort key). Under SPPM
// they replace the pending visible points of the open eye pass (-1 when none is open), which orc_build_grid inserts.
int orc_import_hitpoints(void *c_, int64_t n, const double *rec12) {
    Ctx *c = (Ctx *)c_;
    std::vector<Hitpoint> hps((size_t)n);
    std::vector<uint64_t> sk((size_t)n);
    for (int64_t i = 0; i < n; i++) hps[(size_t)i] = get_record(rec12 + 12 * i, sk[(size_t)i]);
    if (c->sppm) {
        if (!c->pending_open) return -1;
        c->pending.swap(hps);
        return 0;
    }
    const double r = 200.0 / c->R.cfg.height;
    new_table(c->R);
    for (auto &hp : hps) hp.r2 = r * r;
    insert_sorted(c->R, hps, sk);
    c->index();
    return 0;
}

// Photons with global indices [first, first+count). nthreads>1 requires U2 (atomic accumulators) + Philox.
// Returns wall seconds through *seconds.
int orc_photon_pass(void *c_, uint64_t first, uint64_t count, int nthreads, double *seconds) {
    Ctx *c = (Ctx *)c_;
    if (!c->R.htable) return -1;
    auto t0 = std::chrono::steady_clock::now();
    if (nthreads <= 1 || c->libc_mode || c->R.cfg.update != UPDATE_U2_PER_ROUND) {
        Rng rng = c->make_rng();
        for (uint64_t i = 0; i < count; i++) c->R.photon(rng, first + i);
    } else {
#ifdef _OPENMP
        std::vector<Counters> part((size_t)nthreads);
        std::vector<KDCounters> kpart((size_t)nthreads);
#pragma omp parallel num_threads(nthreads)
        {
            Renderer w = c->R.worker();
            Rng rng = Rng::philox(c->R.cfg.seed, PASS_PHOTON, 0, 0);
#pragma omp for schedule(dynamic, 4096)
            for (int64_t i = 0; i < (int64_t)count; i++) w.photon(rng, first + (uint64_t)i);
            part[omp_get_thread_num()] = w.ctr;
            kpart[omp_get_thread_num()] = w.kdc;
        }
        for (auto &kp : kpart) { c->R.kdc.node_visits += kp.node_visits; c->R.kdc.tri_tests += kp.tri_tests; }
        for (auto &p : part) {
            Counters &k = c->R.ctr;
            k.photon_segments += p.photon_segments; k.diffuse_hits += p.diffuse_hits; k.bucket_probes += p.bucket_probes;
            k.nonempty_probes += p.nonempty_probes; k.candidates += p.candidates; k.deposits += p.deposits; k.misses += p.misses;
        }
#else
        return -2;
#endif
    }
    if (seconds) *seconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    return 0;
}
// U2 per hitpoint; under SPPM the per-pixel fold (Ctx::fold).
int orc_round_update(void *c_) {
    Ctx *c = (Ctx *)c_;
    if (!c->sppm) c->R.round_update();
    else if (c->R.htable) c->fold();
    else return -1;
    return 0;
}

int orc_gather_image(void *c_, double n_emitted, double *rgb) {
    Ctx *c = (Ctx *)c_;
    std::vector<Vec3> img;
    // n_emitted = num_photon*num_threads; the num_of_samples factor of main.cpp:256 comes from the config (same convention as cgrt_gather_image)
    const double ne = n_emitted * (double)c->R.cfg.num_of_samples;
    if (!c->sppm) c->R.gather_image(ne, img);
    else  // main.cpp:252-258 with the pixel's statistics
        for (size_t p = 0; p < c->npix(); p++) img.push_back(Vec3() + c->tau[p] * (1.0 / (PI * c->r2[p] * ne)));
    for (size_t i = 0; i < img.size(); i++) st3(rgb + 3 * i, img[i]);
    return 0;
}
// main.cpp:403-411: tone map + gamma + vertical flip into 8-bit RGB.
int orc_tonemap_flip(int width, int height, const double *rgb, uint8_t *out) {
    size_t counter = 0;
    for (int i = 0; i < height; i++)
        for (int j = 0; j < width; j++) {
            const double *px = rgb + 3 * ((size_t)(height - i - 1) * width + j);
            out[3 * counter] = (uint8_t)(char)gammaCorr(px[0]);
            out[3 * counter + 1] = (uint8_t)(char)gammaCorr(px[1]);
            out[3 * counter + 2] = (uint8_t)(char)gammaCorr(px[2]);
            counter++;
        }
    return 0;
}

// average.cpp:19-65: imgdata[i] = sum over the n images of img_k[i] / n (unsigned char arithmetic, division before the sum).
int orc_average_u8(int n, const uint8_t *const *imgs, int64_t nbytes, uint8_t *out) {
    for (int64_t i = 0; i < nbytes; i++) {
        unsigned char acc = 0;
        for (int k = 0; k < n; k++) {
            if (k == 0) acc = (unsigned char)(imgs[k][i] / n);
            else acc += (unsigned char)(imgs[k][i] / n);
        }
        out[i] = acc;
    }
    return 0;
}

int orc_get_counters(void *c_, orc_counters *o) {
    Ctx *c = (Ctx *)c_;
    const Counters &k = c->R.ctr;
    o->eye_segments = k.eye_segments; o->photon_segments = k.photon_segments; o->diffuse_hits = k.diffuse_hits;
    o->bucket_probes = k.bucket_probes; o->nonempty_probes = k.nonempty_probes; o->candidates = k.candidates;
    o->deposits = k.deposits; o->misses = k.misses;
    o->node_visits = c->R.kdc.node_visits; o->tri_tests = c->R.kdc.tri_tests;
    return 0;
}
int orc_max_threads() {
#ifdef _OPENMP
    return omp_get_max_threads();
#else
    return 1;
#endif
}

}  // extern "C"
