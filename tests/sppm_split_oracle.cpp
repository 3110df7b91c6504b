// sppm_split_oracle.cpp — the SPPM CPU reference (tests/sppm_oracle.cpp, included unchanged) with the round split the way ranks of several
// GPUs run it (include/cgrt.h: cgrt_sppm_eye_pass -> record exchange -> cgrt_build_grid), for tests/test_sppm_multi_gpu.py.
// TEST INFRASTRUCTURE ONLY. tests/sppm_split_oracle.py compiles it.
//
// A round here is: sppm_eye_rows (a new, empty table and the eye pass of round r over rows [y0, y1) into a pending set, creation order;
// nothing is inserted) -> optionally export the pending records and import the union of every rank's tile -> sppm_build_table (the pending
// visible points inserted in canonical order: stable sort on key << 32 | path*16 + code, the sort key of the GPU grid, every one at its
// pixel's radius). The pending set lives in its own handle (sppm_pending_create) next to the reference's.
#include "sppm_oracle.cpp"

#include <algorithm>
#include <cstring>

namespace {

struct Pending {
    std::vector<Hitpoint> hp;
};

uint64_t sort_key(const Sppm &s, const Hitpoint &hp) {
    int ix, iy, iz;
    s.R.htable->compute_coord(hp.pos.x, hp.pos.y, hp.pos.z, ix, iy, iz);
    return ((uint64_t)s.R.htable->hash(ix, iy, iz) << 32) | (uint64_t)(uint32_t)(hp.path * 16u + (hp.code & 15u));
}

// Sppm::begin_round's eye pass over rows [y0, y1), without the table inserts.
void trace_rows(Sppm &s, Pending &p, uint32_t r, int y0, int y1, int nthreads) {
    Renderer &R = s.R;
    s.round = r;
    if (R.htable && R.owns_htable) delete R.htable;
    R.htable = new Hashtable(R.cfg.hashsize, 200.0 / R.cfg.height);
    R.owns_htable = true;
    R.next_seq = 0;
    p.hp.clear();
    const int block = 8, nblocks = y1 > y0 ? (y1 - y0 + block - 1) / block : 0;
    std::vector<std::vector<Hitpoint>> sinks((size_t)nblocks);
#ifdef _OPENMP
#pragma omp parallel for schedule(dynamic, 1) num_threads(nthreads > 0 ? nthreads : 1)
#endif
    for (int b = 0; b < nblocks; b++) {
        Renderer w = R.worker();
        w.sink = &sinks[(size_t)b];
        Rng rng = Rng::philox(R.cfg.seed, 0, 0, 0);
        for (int h = y0 + b * block; h < y1 && h < y0 + (b + 1) * block; h++)
            for (int x = 0; x < R.cfg.width; x++)
                for (int j = 0; j < R.cfg.num_of_samples; j++)
                    Sppm::camera(w, s.mode, s.round, x, h, ((uint64_t)h * R.cfg.width + x) * (uint64_t)R.cfg.num_of_samples + j, rng);
    }
    for (auto &sk : sinks)
        for (auto &hp : sk) p.hp.push_back(hp);
}

void build_table(Sppm &s, Pending &p) {
    std::vector<std::pair<uint64_t, size_t>> order(p.hp.size());
    for (size_t i = 0; i < p.hp.size(); i++) order[i] = {sort_key(s, p.hp[i]), i};
    std::stable_sort(order.begin(), order.end(),
                     [](const std::pair<uint64_t, size_t> &a, const std::pair<uint64_t, size_t> &b) { return a.first < b.first; });
    uint32_t seq = 0;
    for (auto &o : order) {
        Hitpoint hp = p.hp[o.second];
        hp.seq = seq++;
        hp.r2 = s.r2[(size_t)hp.h * s.R.cfg.width + hp.w];
        s.R.htable->insert(hp);
    }
    p.hp.clear();
}

}  // namespace

extern "C" {

void *sppm_pending_create() { return new Pending(); }
void sppm_pending_destroy(void *p) { delete (Pending *)p; }

int sppm_eye_rows(void *s_, void *p_, uint32_t round, int y0, int y1, int nthreads) {
    Sppm *s = (Sppm *)s_;
    if (y1 < 0) y1 = s->R.cfg.height;
    if (y0 < 0 || y1 > s->R.cfg.height || y0 > y1) return -1;
    trace_rows(*s, *(Pending *)p_, round, y0, y1, nthreads);
    return 0;
}
// The pending visible points as 12-double records (pos, normal, f, bits(key << 32 | path*16 + code), bits(h << 32 | w), 0: the format of
// cgrt_export_hitpoints_dev and oracle.binding.Oracle.export_hitpoints). rec12 NULL: count only.
int64_t sppm_export_pending(void *s_, void *p_, double *rec12) {
    const Sppm *s = (const Sppm *)s_;
    const Pending *p = (const Pending *)p_;
    for (size_t i = 0; rec12 && i < p->hp.size(); i++) {
        const Hitpoint &hp = p->hp[i];
        double *r = rec12 + 12 * i;
        st3(r, hp.pos); st3(r + 3, hp.normal); st3(r + 6, hp.f);
        uint64_t sk = sort_key(*s, hp);
        uint64_t hw = ((uint64_t)(uint32_t)hp.h << 32) | (uint64_t)(uint32_t)hp.w;
        memcpy(r + 9, &sk, 8); memcpy(r + 10, &hw, 8); r[11] = 0.0;
    }
    return (int64_t)p->hp.size();
}
// Replaces the pending visible points with n records (any order).
int sppm_import_pending(void *s_, void *p_, int64_t n, const double *rec12) {
    if (!((Sppm *)s_)->R.htable) return -1;
    Pending *p = (Pending *)p_;
    p->hp.assign((size_t)n, Hitpoint());
    for (int64_t i = 0; i < n; i++) {
        const double *q = rec12 + 12 * i;
        uint64_t sk, hw;
        memcpy(&sk, q + 9, 8); memcpy(&hw, q + 10, 8);
        Hitpoint &hp = p->hp[(size_t)i];
        hp.pos = v3(q); hp.normal = v3(q + 3); hp.f = v3(q + 6);
        hp.h = (int)(hw >> 32); hp.w = (int)(uint32_t)hw;
        uint32_t lo = (uint32_t)sk;
        hp.code = lo & 15u; hp.path = lo >> 4;
    }
    return 0;
}
int sppm_build_table(void *s_, void *p_) {
    Sppm *s = (Sppm *)s_;
    if (!s->R.htable) return -1;
    build_table(*s, *(Pending *)p_);
    return 0;
}
// Writes the round's accumulators back in canonical order (after an all-reduce of what sppm_download_visible returned).
int sppm_upload_accum(void *s_, const double *dflux, const int32_t *m) {
    Sppm *s = (Sppm *)s_;
    if (!s->R.htable) return -1;
    size_t i = 0;
    for (auto &b : s->R.htable->hashtable)
        for (Hitpoint &hp : b) {
            if (dflux) hp.dflux = v3(dflux + 3 * i);
            if (m) hp.m = m[i];
            i++;
        }
    return 0;
}

}  // extern "C"
