// fixed_capi.cpp — the CPU oracle with fixed-point U2 accumulators (accum_mode 2). TEST INFRASTRUCTURE ONLY.
//
// The whole oracle C API (oracle/oracle_capi.cpp, every orc_* entry point) is compiled into this library unchanged; the fxo_* entry
// points below add the fixed-point mode on top of it. A context made by fxo_create is an ordinary oracle context (pass it to any orc_*
// function) that also carries int64 accumulators {sum q_x, sum q_y, sum q_z, M} per hitpoint, indexed by the hitpoint's sequence number.
//
// The definition restated here is the device code's (cgraytracing_b200/csrc/cgrt_passes.cuh, deposit_value_f32 / deposit_fixed /
// fixed_to_update): an accepted pair adds q = round-half-even(cf * 2^22) per channel, cf = ((float)f * (float)flux) * (float)(1/pi) in
// IEEE float (no contraction: built with -ffp-contract=off); the update reads dflux = (double)sum q * 2^-22 and M. A value cf > 2^16
// (or NaN) or a round's M > 2^24 per hitpoint (SPPM: per pixel) raises the error word.
#include "../oracle/oracle_capi.cpp"

#include <cmath>

namespace {

const float FIX_SCALE = 4194304.0f;  // 2^22
const double FIX_INV_SCALE = 1.0 / 4194304.0;
const float FIX_MAX_VALUE = 65536.0f;  // 2^16
const int64_t FIX_MAX_COUNT = 16777216;  // 2^24
enum { FIX_ERR_VALUE = 1, FIX_ERR_COUNT = 2 };

struct FxCtx : Ctx {
    std::vector<int64_t> acc;  // 4 per hitpoint sequence number
    int err = 0;
};

inline float deposit_value_f32(double f, double flux) { return ((float)f * (float)flux) * (float)(1.0 / PI); }
inline int64_t fixed_q(float cf) { return (int64_t)std::llrintf(cf * FIX_SCALE); }  // round-half-even in the default rounding mode

void fx_deposit(FxCtx &X, const Hitpoint &hp, const Vec3 &flux) {
    const float cx = deposit_value_f32(hp.f.x, flux.x), cy = deposit_value_f32(hp.f.y, flux.y), cz = deposit_value_f32(hp.f.z, flux.z);
    if (!(cx <= FIX_MAX_VALUE) || !(cy <= FIX_MAX_VALUE) || !(cz <= FIX_MAX_VALUE)) {
#pragma omp atomic
        X.err |= FIX_ERR_VALUE;
        return;
    }
    int64_t *a = X.acc.data() + 4 * (size_t)hp.seq;
    const int64_t qx = fixed_q(cx), qy = fixed_q(cy), qz = fixed_q(cz);
#pragma omp atomic
    a[0] += qx;
#pragma omp atomic
    a[1] += qy;
#pragma omp atomic
    a[2] += qz;
#pragma omp atomic
    a[3] += 1;
}

// Renderer::trace (oracle/ppm_oracle.hpp) for a photon (flag false), with the fixed-point deposit in place of the U2 fp64 one.
void fx_trace(Renderer &R, FxCtx &X, const Vec3 &org, const Vec3 &dir, Vec3 flux, int depth, Rng &rng, uint64_t path) {
    const Config &cfg = R.cfg;
    if (depth >= cfg.max_depth) return;
    rng.reseed(cfg.seed, PASS_PHOTON, path, (uint32_t)depth + 1);
    Rng bez_rng = rng;
    TraceCtx tc;
    tc.into_rule = cfg.into_rule;
    tc.kdc = &R.kdc;
    if (rng.mode == 1) {
        bez_rng.reseed(cfg.seed, PASS_BEZIER, path, (uint32_t)depth * 2 + 1);
        tc.rng = &bez_rng;
    } else {
        tc.rng = &rng;
    }
    R.ctr.photon_segments++;
    HitRecord hr;
    if (!R.closest_hit(org, dir, hr, tc)) { R.ctr.misses++; return; }
    const Object *obj = R.objs[hr.id];
    Vec3 intersection = org + dir * hr.t;
    bool into = hr.into != 0;
    Vec3 normalvec_old = hr.n_raw;
    Vec3 normalvec = hr.n_ff;
    Vec3 f = obj->getSurfaceColor(intersection);
    double p = max3(f.x, f.y, f.z);
    if (obj->getReflection() < EPS && obj->getTransparency() < EPS) {
        R.ctr.diffuse_hits++;
        Hashtable *ht = R.htable;
        int ix, iy, iz;
        ht->compute_coord(intersection.x, intersection.y, intersection.z, ix, iy, iz);
        ix -= 1; iy -= 1; iz -= 1;
        for (int idx = 0; idx < 3; idx++)
            for (int idy = 0; idy < 3; idy++)
                for (int idz = 0; idz < 3; idz++) {
                    std::vector<Hitpoint> &bucket = ht->hashtable[ht->hash(ix + idx, iy + idy, iz + idz)];
                    R.ctr.bucket_probes++;
                    if (!bucket.empty()) R.ctr.nonempty_probes++;
                    for (size_t i = 0; i < bucket.size(); i++) {
                        const Hitpoint &hp = bucket[i];
                        R.ctr.candidates++;
                        Vec3 d = hp.pos - intersection;
                        if ((hp.normal.dot(normalvec) > EPS) && (d.dot(d) <= hp.r2)) {
                            R.ctr.deposits++;
                            fx_deposit(X, hp, flux);
                        }
                    }
                }
        Vec3 newdir = uniform_sampling_halfsphere(rng, normalvec);
        fx_trace(R, X, intersection, newdir, f * flux * (1.0 / p), depth + 1, rng, path);
    } else if (obj->getTransparency() < EPS) {
        Vec3 newdir = dir - normalvec * 2.0 * normalvec.dot(dir);
        fx_trace(R, X, intersection + normalvec * EPS, newdir, f * flux * obj->getReflection(), depth + 1, rng, path);
    } else {
        double nc = 1.0, nt = 1.33, nnt = into ? nc / nt : nt / nc, ddn = dir.dot(normalvec), cos2t;
        Vec3 refl_dir = dir - normalvec_old * 2.0 * normalvec_old.dot(dir);
        if ((cos2t = 1 - nnt * nnt * (1 - ddn * ddn)) < 0) {
            fx_trace(R, X, intersection + normalvec * EPS, refl_dir, flux, depth + 1, rng, path);
            return;
        }
        Vec3 refr_dir = (dir * nnt - normalvec_old * ((into ? 1 : -1) * (ddn * nnt + std::sqrt(cos2t)))).normalize();
        if (uniform_sampling_zeroone(rng) < 0.5) fx_trace(R, X, intersection + normalvec * EPS, refl_dir, flux, depth + 1, rng, path);
        else fx_trace(R, X, intersection - normalvec * EPS, refr_dir, flux, depth + 1, rng, path);
    }
}

// Renderer::photon with fx_trace.
void fx_photon(Renderer &R, FxCtx &X, Rng &rng, uint64_t index) {
    rng.reseed(R.cfg.seed, PASS_PHOTON, index, 0);
    double a = uniform_sampling_zeroone(rng) * 4 - 2;
    double b = uniform_sampling_zeroone(rng) * 4 - 2;
    Vec3 disturbance = Vec3(a, 0, b);
    Vec3 dir = uniform_sampling_sphere(rng);
    fx_trace(R, X, R.cfg.lightorg + disturbance, dir, Vec3(700, 700, 700) * (PI * 4.0), 0, rng, index);
}

// Accumulators for every hitpoint of the current table (sequence numbers are dense per table); new slots are zero.
void fx_size(FxCtx &X) {
    X.index();
    size_t need = 0;
    for (const Hitpoint *hp : X.canon) need = std::max(need, 4 * ((size_t)hp->seq + 1));
    if (X.acc.size() < need) X.acc.resize(need, 0);
}

void add_counters(Counters &k, const Counters &p) {
    k.photon_segments += p.photon_segments; k.diffuse_hits += p.diffuse_hits; k.bucket_probes += p.bucket_probes;
    k.nonempty_probes += p.nonempty_probes; k.candidates += p.candidates; k.deposits += p.deposits; k.misses += p.misses;
}

}  // namespace

extern "C" {

void *fxo_create() { return static_cast<Ctx *>(new FxCtx()); }
void fxo_destroy(void *c) { delete static_cast<FxCtx *>(static_cast<Ctx *>(c)); }
static FxCtx *fx(void *c) { return static_cast<FxCtx *>(static_cast<Ctx *>(c)); }

// Photons [first, first+count) with fixed-point deposits, on nthreads OpenMP threads; reverse != 0 traces them last to first.
int fxo_photon_pass(void *c_, uint64_t first, uint64_t count, int nthreads, int reverse) {
    FxCtx &X = *fx(c_);
    if (!X.R.htable || X.libc_mode || X.R.cfg.update != UPDATE_U2_PER_ROUND) return -1;
    fx_size(X);
    const int nt = nthreads > 0 ? nthreads : 1;
    std::vector<Counters> part((size_t)nt);
    std::vector<KDCounters> kpart((size_t)nt);
#ifdef _OPENMP
#pragma omp parallel num_threads(nt)
#endif
    {
#ifdef _OPENMP
        const int t = omp_get_thread_num();
#else
        const int t = 0;
#endif
        Renderer w = X.R.worker();
        Rng rng = Rng::philox(X.R.cfg.seed, PASS_PHOTON, 0, 0);
#ifdef _OPENMP
#pragma omp for schedule(dynamic, 1024)
#endif
        for (int64_t i = 0; i < (int64_t)count; i++) fx_photon(w, X, rng, first + (uint64_t)(reverse ? (int64_t)count - 1 - i : i));
        part[(size_t)t] = w.ctr;
        kpart[(size_t)t] = w.kdc;
    }
    for (auto &kp : kpart) { X.R.kdc.node_visits += kp.node_visits; X.R.kdc.tri_tests += kp.tri_tests; }
    for (auto &p : part) add_counters(X.R.ctr, p);
    return 0;
}

// One caller-made photon (orc_trace with flag 0) with fixed-point deposits: path = its photon index.
int fxo_trace(void *c_, const double *org, const double *dir, const double *flux, uint64_t path) {
    FxCtx &X = *fx(c_);
    if (!X.R.htable || X.libc_mode) return -1;
    fx_size(X);
    Rng rng = X.make_rng();
    fx_trace(X.R, X, v3(org), v3(dir), v3(flux), 0, rng, path);
    return 0;
}

// The round update of the fixed-point mode: per hitpoint (PPM) dflux = sum q * 2^-22 and M into Renderer::round_update; under SPPM the
// integer sums per pixel, converted once, into the fold of Ctx::fold's rule. Clears the accumulators.
int fxo_round_update(void *c_) {
    FxCtx &X = *fx(c_);
    if (!X.R.htable) return -1;
    fx_size(X);
    if (!X.sppm) {
        for (const Hitpoint *cp : X.canon) {
            Hitpoint *hp = const_cast<Hitpoint *>(cp);
            int64_t *a = X.acc.data() + 4 * (size_t)hp->seq;
            if (a[3] > FIX_MAX_COUNT) X.err |= FIX_ERR_COUNT;
            hp->dflux = Vec3((double)a[0] * FIX_INV_SCALE, (double)a[1] * FIX_INV_SCALE, (double)a[2] * FIX_INV_SCALE);
            hp->m = (int)a[3];
        }
        X.R.round_update();
    } else {
        std::vector<int64_t> s(4 * X.npix(), 0);
        for (const Hitpoint *hp : X.canon) {
            const int64_t *a = X.acc.data() + 4 * (size_t)hp->seq;
            int64_t *t = s.data() + 4 * X.pixel(*hp);
            for (int k = 0; k < 4; k++) t[k] += a[k];
        }
        for (size_t p = 0; p < X.npix(); p++) {
            const int64_t *t = s.data() + 4 * p;
            if (t[3] > FIX_MAX_COUNT) X.err |= FIX_ERR_COUNT;
            if (t[3] > 0) {
                Vec3 d((double)t[0] * FIX_INV_SCALE, (double)t[1] * FIX_INV_SCALE, (double)t[2] * FIX_INV_SCALE);
                double na = X.n[p] * X.R.cfg.alpha;
                double mm = (double)t[3];
                double g = (na + X.R.cfg.alpha * mm) / (na + mm);
                X.tau[p] = (X.tau[p] + d) * g;
                X.r2[p] *= g;
                X.n[p] += (int)t[3];
            }
        }
    }
    std::fill(X.acc.begin(), X.acc.end(), 0);
    return 0;
}

// The round's accumulators in canonical order: acc4 = {sum q_x, sum q_y, sum q_z, M} (int64), and/or dflux = sum q * 2^-22 and m = M
// as the update reads them. Any pointer may be NULL.
int fxo_download_accum(void *c_, int64_t *acc4, double *dflux, double *m) {
    FxCtx &X = *fx(c_);
    fx_size(X);
    for (size_t i = 0; i < X.canon.size(); i++) {
        const int64_t *a = X.acc.data() + 4 * (size_t)X.canon[i]->seq;
        for (int k = 0; k < 4; k++) {
            if (acc4) acc4[4 * i + k] = a[k];
            if (dflux && k < 3) dflux[3 * i + k] = (double)a[k] * FIX_INV_SCALE;
        }
        if (m) m[i] = (double)a[3];
    }
    return 0;
}
// Writes back all-reduced int64 accumulators (canonical order), for the sharding tests.
int fxo_upload_accum(void *c_, const int64_t *acc4) {
    FxCtx &X = *fx(c_);
    fx_size(X);
    for (size_t i = 0; i < X.canon.size(); i++)
        for (int k = 0; k < 4; k++) X.acc[4 * (size_t)X.canon[i]->seq + k] = acc4[4 * i + k];
    return 0;
}
// FIX_ERR_* bits raised so far (they stay raised).
int fxo_error(void *c_) { return fx(c_)->err; }
// The definition itself on free-standing inputs: cf and q of n (f, flux) pairs per channel.
int fxo_deposit_value(int64_t n, const double *f, const double *flux, float *cf, int64_t *q) {
    for (int64_t i = 0; i < n; i++) {
        const float v = deposit_value_f32(f[i], flux[i]);
        if (cf) cf[i] = v;
        if (q) q[i] = fixed_q(v);
    }
    return 0;
}

}  // extern "C"
