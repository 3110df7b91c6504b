// cgrt_passes.cuh — the wavefront passes: eye pass, hash grid, photon trace + deposit, round update, image gather.
// Replaces trace()/render() (main.cpp:42-266). Recursion becomes per-depth kernels over ray queues that are
// compacted with warp ballots (one atomic per warp); the hash table of vectors becomes a sorted array + cell-start
// table; photon deposits are atomics into per-round accumulators.
#pragma once
#include "../../include/cgrt.h"
#include "cgrt_build.cuh"

namespace cgrt {

// Ray queue, structure of arrays. w = path weight: adj for eye rays (main.cpp:42 `adj`), flux for photons (`flux`).
struct RayQueue {
    double *ox, *oy, *oz, *dx, *dy, *dz, *wx, *wy, *wz;
    uint32_t *id;    // eye: path = (h*W + w)*samples + s ; photon: offset from the call's first photon index
    uint32_t *aux;   // eye: DFS split code (nsplit << 4 | bits, SURVEY Q19)
};

// Hitpoint hot record read per candidate in the gather: 64 bytes (two sectors).
struct __align__(16) HpHot {
    double px, py, pz, r2;
    double nx, ny, nz, pad;
};

// fp32 prefilter record of one hitpoint (see photon_deposit_kernel). E bounds |fl(hp) - fl(X)| - |hp - X| for any photon
// position X within the radius: two float roundings per axis at magnitude <= m + r, sqrt(3) axes, with 2x headroom.
__device__ __forceinline__ float4 make_prefilter(double px, double py, double pz, double r2) {
    double r = sqrt(r2);
    double m = fmax(fmax(fabs(px), fabs(py)), fabs(pz)) + r + 1.0;
    double E = 4.5e-7 * m;
    double b = (r + E) * (r + E) * (1.0 + 4e-6);
    return make_float4((float)px, (float)py, (float)pz, __double2float_ru(b));
}
// The same bound read the other way: a float squared distance <= (r - E)^2 (rounded down, negative when r <= E so that nothing
// qualifies) proves the fp64 test dot(dd, dd) <= r2 of main.cpp:116 true. Stored next to the fp32 normal: {nx, ny, nz, (r - E)^2}.
__device__ __forceinline__ float prefilter_inner(double px, double py, double pz, double r2) {
    double r = sqrt(r2);
    double m = fmax(fmax(fabs(px), fabs(py)), fabs(pz)) + r + 1.0;
    double E = 4.5e-7 * m;
    if (r <= E) return -1.0f;
    double b = (r - E) * (r - E) * (1.0 - 4e-6);
    return __double2float_rd(b);
}

struct PassParams {
    int width, height, max_depth, samples, use_dof;
    uint32_t hashsize;
    uint32_t bin_mask;     // counting-sort bins of the deposit table - 1 (2^22 or 2^23 bins)
    double celllength;     // Hashtable ctor result, hash.h:25-26
    double inv_celllength; // 1 / celllength (cell_floor_div)
    double r2_init;        // (200/height)^2, main.cpp:84,94
    double alpha, focus_plane, lens_radius;
    double cam[3], light[3];
    uint64_t seed;
};

// One slot per active lane of the warp, claimed with a single atomic (ballot + popc prefix).
__device__ __forceinline__ unsigned int warp_claim(bool want, unsigned int *counter, unsigned int n = 1) {
    unsigned int active = __activemask();
    unsigned int mask = __ballot_sync(active, want);
    if (!want) return 0xffffffffu;
    int lane = threadIdx.x & 31;
    int leader = __ffs(mask) - 1;
    unsigned int base = 0;
    // all wanting lanes request the same n here (n is uniform across the call sites)
    if (lane == leader) base = atomicAdd(counter, n * __popc(mask));
    base = __shfl_sync(mask, base, leader);
    return base + n * __popc(mask & ((1u << lane) - 1u));
}

__device__ __forceinline__ void push_ray(const RayQueue &q, unsigned int s, d3 o, d3 d, d3 w, uint32_t id, uint32_t aux) {
    q.ox[s] = o.x; q.oy[s] = o.y; q.oz[s] = o.z;
    q.dx[s] = d.x; q.dy[s] = d.y; q.dz[s] = d.z;
    q.wx[s] = w.x; q.wy[s] = w.y; q.wz[s] = w.z;
    q.id[s] = id;
    if (q.aux) q.aux[s] = aux;
}

struct Counters {
    unsigned long long eye_segments, photon_segments, diffuse_hits, candidates, deposits, gathered_hits, exact_tests;
    unsigned long long cell_groups, staged_candidates;  // deposit kernel: groups of same-cell hits, bucket entries read for them
};

// =================================================================================================================
// Eye pass, one kernel per depth level. Level 0 generates the camera rays (main.cpp:188-209) in registers.
// Hitpoint records (CGRT_HP_RECORD_DOUBLES doubles): pos, normal, f*adj, bits(sortkey), bits(h<<32|w), 0.
// sortkey = bucket key << 32 | (path*16 + dfs bits): sorting by it gives the reference's bucket order (hash.h:52,
// main.cpp:252-254) whatever order the wavefront produced the hitpoints in.
// =================================================================================================================
enum { HP_POS = 0, HP_NRM = 3, HP_F = 6, HP_KEY = 9, HP_PIX = 10 };  // offsets into a hitpoint record
static_assert(HP_PIX + 2 == CGRT_HP_RECORD_DOUBLES, "hitpoint record layout");
#define CGRT_TRACE_BLOCK 128
#ifndef CGRT_PHOTON_BLOCK
#define CGRT_PHOTON_BLOCK 128   /* threads per block of photon_trace_kernel */
#endif
#ifndef CGRT_FETCH
#define CGRT_FETCH 256         /* indices a warp of photon_trace_kernel draws from the global cursor at a time (64-256: 4.95 ms, 1024: 5.07 ms) */
#endif
// minimum resident blocks per SM asked of ptxas for the photon kernels (register caps; tuned with A/B builds)
#ifndef CGRT_TRACE_MINB
#define CGRT_TRACE_MINB 1   /* 6 (80 registers) and 8 (64 registers, spills) were measured: no gain / slower */
#endif
#ifndef CGRT_TRAV_MINB
#define CGRT_TRAV_MINB 8   /* 64 registers: 13.7 vs 15.1 ms of trace time per round; 6 (80 registers) gained nothing */
#endif

// F32: every tree lies within CGRT_F32_BOUND (all BASELINE scenes) — the traversal instantiation without fp64 box arithmetic, as in the photon pass
// (c4: 3.58 -> 3.86 G eye rays/s). Register caps of 167 / 161 / 96 were measured: c3 within 1.78-1.94 ms either way.
// SPPM (FIRST only): 0 = the PPM camera; CGRT_SPPM_JITTER / CGRT_SPPM_CORNER = the camera of round `sppm_round`, drawn from
// (seed, PASS_SPPM_EYE, path, round): jitter ux, uy (jitter mode only), then the lens sample; the pixel position w + ux, h + uy enters
// the expressions of main.cpp:188-198 in place of w, h. A template parameter and a trailing argument, so that the PPM instantiations
// compile as before (the argument moves no other parameter; PassParams, which every photon kernel reads, is left as it is).
template <bool FIRST, bool F32, int SPPM = 0>
__global__ void __launch_bounds__(CGRT_TRACE_BLOCK) eye_bounce_kernel(const __grid_constant__ SceneDev S, const __grid_constant__ PassParams P, int depth,
                                                         RayQueue qin, unsigned int n_in, int y0, RayQueue qout, unsigned int *n_out,
                                                         double *hp_rec, unsigned int *hp_count, unsigned int hp_cap, Counters *ctr,
                                                         uint32_t sppm_round) {
    __shared__ TraceShared<CGRT_TRACE_BLOCK> sm;
    unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = i < n_in;
    d3 o = mk(0, 0, 0), d = mk(0, 0, 1), adj = mk(0, 0, 0);
    uint32_t path = 0, code = 0;
    if (!active) {
    } else if (FIRST && SPPM == 0) {
        uint32_t s = i % (uint32_t)P.samples;
        uint32_t pix = i / (uint32_t)P.samples;
        int w = (int)(pix % (uint32_t)P.width), h = y0 + (int)(pix / (uint32_t)P.width);
        path = ((uint32_t)h * (uint32_t)P.width + (uint32_t)w) * (uint32_t)P.samples + s;
        code = 0;
        d3 cam = mk(P.cam[0], P.cam[1], P.cam[2]);
        double x = (2.0 * ((double)w / P.width) - 1) * 10.0;
        double y = (2.0 * ((double)h / P.height) - 1) * 10.0 * P.height / P.width;
        d = normalize(mk(x, y, 0) - cam);
        o = cam;
        if (P.use_dof) {  // main.cpp:203-207
            d3 pof = d * ((P.focus_plane - cam.z) / d.z) + cam;
            Philox g;
            g.init(P.seed, PASS_EYE, (uint64_t)path, 0);
            o = cam + sample_circle(g, P.lens_radius);
            d = normalize(pof - o);
        }
        adj = mk(1, 1, 1);
    } else if (FIRST) {
        uint32_t s = i % (uint32_t)P.samples;
        uint32_t pix = i / (uint32_t)P.samples;
        int w = (int)(pix % (uint32_t)P.width), h = y0 + (int)(pix / (uint32_t)P.width);
        path = ((uint32_t)h * (uint32_t)P.width + (uint32_t)w) * (uint32_t)P.samples + s;
        code = 0;
        Philox g;
        g.init(P.seed, PASS_SPPM_EYE, (uint64_t)path, sppm_round);
        double xs = (double)w, ys = (double)h;
        if (SPPM == CGRT_SPPM_JITTER) {
            xs = (double)w + g.u01();
            ys = (double)h + g.u01();
        }
        d3 cam = mk(P.cam[0], P.cam[1], P.cam[2]);
        double x = (2.0 * (xs / P.width) - 1) * 10.0;
        double y = (2.0 * (ys / P.height) - 1) * 10.0 * P.height / P.width;
        d = normalize(mk(x, y, 0) - cam);
        o = cam;
        if (P.use_dof) {
            d3 pof = d * ((P.focus_plane - cam.z) / d.z) + cam;
            o = cam + sample_circle(g, P.lens_radius);
            d = normalize(pof - o);
        }
        adj = mk(1, 1, 1);
    } else {
        o = mk(qin.ox[i], qin.oy[i], qin.oz[i]);
        d = mk(qin.dx[i], qin.dy[i], qin.dz[i]);
        adj = mk(qin.wx[i], qin.wy[i], qin.wz[i]);
        path = qin.id[i];
        code = qin.aux[i];
    }
    Hit hit;
    bool found = closest_hit_block<CGRT_TRACE_BLOCK, false, F32>(S, active, o, d, hit, sm, nullptr);
    {   // segments counter: one atomic per warp
        unsigned int act = __ballot_sync(0xffffffffu, active);
        if ((threadIdx.x & 31) == 0 && act) atomicAdd(&ctr->eye_segments, (unsigned long long)__popc(act));
    }
    int mat = -1;
    d3 X = mk(0, 0, 0), n_ff = mk(0, 0, 0), n_old = mk(0, 0, 0), f = mk(0, 0, 0);
    bool into = true;
    if (found) {
        const ObjDev &O = S.obj[hit.obj];
        X = o + d * hit.t;  // main.cpp:68
        n_old = hit.n;
        n_ff = hit.n;
        if (dot(n_ff, d) > 0) { n_ff = -n_ff; into = false; }  // main.cpp:73-76
        f = surface_color(S, hit.obj, X);
        mat = O.material;
    }
    bool cont = (depth + 1 < P.max_depth);

    // ---- diffuse: create the hitpoint (main.cpp:85-99)
    bool mk_hp = (mat == MAT_DIFFUSE);
    unsigned int hs = warp_claim(mk_hp, hp_count);
    if (mk_hp && hs < hp_cap) {
        int ix, iy, iz;
        cell_coord(X, P.celllength, P.inv_celllength, ix, iy, iz);
        uint32_t key = cell_hash(ix, iy, iz, P.hashsize);
        uint64_t sortkey = ((uint64_t)key << 32) | (uint64_t)(path * 16u + (code & 15u));
        uint32_t pix = path / (uint32_t)P.samples;
        uint64_t hw = ((uint64_t)(pix / (uint32_t)P.width) << 32) | (uint64_t)(pix % (uint32_t)P.width);
        d3 fa = f * adj;
        double *r = hp_rec + (size_t)hs * CGRT_HP_RECORD_DOUBLES;
        r[HP_POS] = X.x; r[HP_POS + 1] = X.y; r[HP_POS + 2] = X.z;
        r[HP_NRM] = n_ff.x; r[HP_NRM + 1] = n_ff.y; r[HP_NRM + 2] = n_ff.z;
        r[HP_F] = fa.x; r[HP_F + 1] = fa.y; r[HP_F + 2] = fa.z;
        r[HP_KEY] = __longlong_as_double((long long)sortkey);
        r[HP_PIX] = __longlong_as_double((long long)hw);
        r[HP_PIX + 1] = 0.0;
    }

    // ---- mirror / glass: children (main.cpp:129-157)
    int nchild = 0;
    d3 co[2], cd[2], cw[2];
    uint32_t ccode[2] = {code, code};
    if (cont && mat == MAT_MIRROR) {
        const ObjDev &O = S.obj[hit.obj];
        cd[0] = d - n_ff * 2.0 * dot(n_ff, d);
        co[0] = X + n_ff * CGRT_EPS;
        cw[0] = f * adj * O.refl;
        nchild = 1;
    } else if (cont && mat == MAT_GLASS) {
        double nc = 1.0, nt = 1.33, nnt = into ? nc / nt : nt / nc, ddn = dot(d, n_ff), cos2t;
        d3 refl_dir = d - n_old * 2.0 * dot(n_old, d);
        if ((cos2t = 1 - nnt * nnt * (1 - ddn * ddn)) < 0) {  // total internal reflection, main.cpp:144
            co[0] = X + n_ff * CGRT_EPS; cd[0] = refl_dir; cw[0] = adj;
            nchild = 1;
        } else {
            d3 refr_dir = normalize(d * nnt - n_old * ((into ? 1 : -1) * (ddn * nnt + sqrt(cos2t))));
            double a = nt - nc, b = nt + nc, R0 = a * a / (b * b), c = 1 - (into ? -ddn : dot(refr_dir, n_old));
            double Re = R0 + (1 - R0) * c * c * c * c * c;
            d3 fa = f * adj;
            int ns = (int)(code >> 4);
            int shift = 3 - ns;
            uint32_t bits = code & 15u;
            co[0] = X + n_ff * CGRT_EPS; cd[0] = refl_dir; cw[0] = fa * Re;
            ccode[0] = ((uint32_t)(ns + 1) << 4) | bits;
            co[1] = X - n_ff * CGRT_EPS; cd[1] = refr_dir; cw[1] = fa * (1 - Re);
            ccode[1] = ((uint32_t)(ns + 1) << 4) | (bits | (shift >= 0 ? (1u << shift) : 0u));
            nchild = 2;
        }
    }
    // mirrors/TIR want 1 slot, splits want 2: claim in two rounds so each claim is uniform
    unsigned int s0 = warp_claim(nchild >= 1, n_out);
    unsigned int s1 = warp_claim(nchild >= 2, n_out);
    if (nchild >= 1) push_ray(qout, s0, co[0], cd[0], cw[0], path, ccode[0]);
    if (nchild >= 2) push_ray(qout, s1, co[1], cd[1], cw[1], path, ccode[1]);
}

// =================================================================================================================
// Grid build helpers
// =================================================================================================================
__global__ void hp_extract_keys_kernel(const double *__restrict__ rec, unsigned int n, uint64_t *__restrict__ keys) {
    unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) keys[i] = (uint64_t)__double_as_longlong(rec[(size_t)i * CGRT_HP_RECORD_DOUBLES + HP_KEY]);
}

// Imported records are checked before build_grid uses their key and pixel as indices (lower_bound_table_kernel,
// sppm_visible_radius_kernel): bit 0 = a key >= hashsize, bit 1 = a key that is not the cell key of the position (the hitpoint would sit
// in a bucket no photon near it gathers), bit 2 = a pixel outside the image.
__global__ void hp_validate_kernel(const double *__restrict__ rec, unsigned int n, double celllength, uint32_t hashsize, int width, int height,
                                   unsigned int *__restrict__ bad) {
    unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double *r = rec + (size_t)i * CGRT_HP_RECORD_DOUBLES;
    const uint32_t key = (uint32_t)((uint64_t)__double_as_longlong(r[HP_KEY]) >> 32);
    const uint64_t hw = (uint64_t)__double_as_longlong(r[HP_PIX]);
    int ix, iy, iz;
    cell_coord(mk(r[HP_POS], r[HP_POS + 1], r[HP_POS + 2]), celllength, 1.0 / celllength, ix, iy, iz);
    unsigned int f = 0;
    if (key >= hashsize) f |= 1u;
    else if (key != cell_hash(ix, iy, iz, hashsize)) f |= 2u;
    if ((uint32_t)(hw >> 32) >= (uint32_t)height || (uint32_t)hw >= (uint32_t)width) f |= 4u;
    if (f) atomicOr(bad, f);
}

struct HpArrays {
    float4 *pre;           // fp32 prefilter {x, y, z, (r+E)^2} read per candidate
    float4 *pre_n;         // fp32 accept filter {nx, ny, nz, (r-E)^2}
    float4 *pre_f;         // fp32 copy of f {fx, fy, fz, 0} (float-accumulator mode deposits from it)
    HpHot *hot;            // pos, r2, normal (exact test)
    double *f;             // [n][4] f*adj (+pad)
    double *flux;          // [n][4] tau (+pad)
    int *cnt;              // accepted photon count n
    int *hw;               // [n][2] pixel (h, w)
    uint32_t *key;         // bucket key
    uint32_t *seq;         // path*16 + dfs bits
};

// A new radius for hitpoint k (hh = its hot record, position read from it): the exact record and both fp32 filter bounds follow it.
// Every radius change after hp_gather_sorted_kernel goes through here, so no filter is ever left at an older radius.
__device__ __forceinline__ void set_radius(const HpArrays &A, unsigned int k, const HpHot &hh, double r2) {
    A.hot[k].r2 = r2;
    A.pre[k] = make_prefilter(hh.px, hh.py, hh.pz, r2);
    A.pre_n[k].w = prefilter_inner(hh.px, hh.py, hh.pz, r2);
}

__global__ void hp_gather_sorted_kernel(const double *__restrict__ rec, const uint32_t *__restrict__ perm, unsigned int n, double r2_init,
                                        HpArrays A, uint64_t *__restrict__ pixkeys, int width) {
    unsigned int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const double *r = rec + (size_t)perm[k] * CGRT_HP_RECORD_DOUBLES;
    HpHot h;
    h.px = r[HP_POS]; h.py = r[HP_POS + 1]; h.pz = r[HP_POS + 2]; h.r2 = r2_init;
    h.nx = r[HP_NRM]; h.ny = r[HP_NRM + 1]; h.nz = r[HP_NRM + 2]; h.pad = 0.0;
    A.hot[k] = h;
    A.pre[k] = make_prefilter(h.px, h.py, h.pz, r2_init);
    A.pre_n[k] = make_float4((float)h.nx, (float)h.ny, (float)h.nz, prefilter_inner(h.px, h.py, h.pz, r2_init));
    A.pre_f[k] = make_float4((float)r[HP_F], (float)r[HP_F + 1], (float)r[HP_F + 2], 0.f);
    A.f[4 * (size_t)k] = r[HP_F]; A.f[4 * (size_t)k + 1] = r[HP_F + 1]; A.f[4 * (size_t)k + 2] = r[HP_F + 2]; A.f[4 * (size_t)k + 3] = 0.0;
    A.flux[4 * (size_t)k] = 0.0; A.flux[4 * (size_t)k + 1] = 0.0; A.flux[4 * (size_t)k + 2] = 0.0; A.flux[4 * (size_t)k + 3] = 0.0;
    A.cnt[k] = 0;
    uint64_t sk = (uint64_t)__double_as_longlong(r[HP_KEY]);
    uint64_t hw = (uint64_t)__double_as_longlong(r[HP_PIX]);
    A.key[k] = (uint32_t)(sk >> 32);
    A.seq[k] = (uint32_t)sk;
    int hh = (int)(hw >> 32), ww = (int)(uint32_t)hw;
    A.hw[2 * (size_t)k] = hh; A.hw[2 * (size_t)k + 1] = ww;
    pixkeys[k] = (uint64_t)hh * (uint64_t)width + (uint64_t)ww;
}

// SPPM: every visible point of a round takes its pixel's current radius (in place of the r2_init hp_gather_sorted_kernel wrote).
__global__ void sppm_visible_radius_kernel(unsigned int n, HpArrays A, const double *__restrict__ pix_r2, int width) {
    unsigned int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const double r2 = pix_r2[(size_t)A.hw[2 * (size_t)k] * (size_t)width + (size_t)A.hw[2 * (size_t)k + 1]];
    const HpHot hh = A.hot[k];  // a local copy: passing A.hot[k] itself compiles to 24 more instructions
    set_radius(A, k, hh, r2);
}

// start[v] = first sorted index whose key is >= v, for v in [0, nvals]; keys ascending.
__global__ void lower_bound_table_kernel(const uint32_t *__restrict__ keys32, const uint64_t *__restrict__ keys64, unsigned int n, unsigned int nvals,
                                         uint32_t *__restrict__ start) {
    unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i > n) return;
    long long prev = (i == 0) ? -1 : (keys32 ? (long long)keys32[i - 1] : (long long)keys64[i - 1]);
    long long cur = (i == n) ? (long long)nvals : (keys32 ? (long long)keys32[i] : (long long)keys64[i]);
    for (long long v = prev + 1; v <= cur; v++) start[v] = i;
}

// =================================================================================================================
// Reach map: a bitmap over (hashed) cell coordinates that is set for every cell within +-2 cells of a hitpoint's cell.
// A photon hit can only ever be accepted by a hitpoint at distance <= r0 = 200/height <= 1.0045 cells (main.cpp:116 with
// r2 <= r0^2; SURVEY Q13), i.e. by a hitpoint at most 2 cells away on every axis — whichever bucket the hash put it in.
// A hit whose cell is not in the map therefore deposits nothing, and the photon kernel drops it before it costs a record,
// a sort slot and a 27-bucket gather (about half of all hits in the reference scenes land on the unobserved front part of
// the room). Hash collisions in the bitmap only add false positives. cull = 0 disables it (counter parity tests).
// =================================================================================================================
#define CGRT_REACH_BITS 26  /* 64 Mi bits = 8 MB */
__device__ __forceinline__ uint32_t reach_hash(int ix, int iy, int iz) {
    uint32_t h = (uint32_t)ix * 0x8DA6B343u ^ (uint32_t)iy * 0xD8163841u ^ (uint32_t)iz * 0xCB1AB31Fu;
    h ^= h >> 13; h *= 0x9E3779B1u; h ^= h >> 16;
    return h & ((1u << CGRT_REACH_BITS) - 1u);
}
__global__ void reach_mark_kernel(const HpHot *__restrict__ hot, unsigned int n, double celllength, uint32_t *__restrict__ bitmap) {
    unsigned int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    int ix, iy, iz;
    cell_coord(mk(hot[k].px, hot[k].py, hot[k].pz), celllength, 1.0 / celllength, ix, iy, iz);
    for (int a = -2; a <= 2; a++)
        for (int b = -2; b <= 2; b++)
            for (int c = -2; c <= 2; c++) {
                uint32_t h = reach_hash(ix + a, iy + b, iz + c);
                uint32_t bit = 1u << (h & 31u);
                if (!(bitmap[h >> 5] & bit)) atomicOr(bitmap + (h >> 5), bit);
            }
}

// =================================================================================================================
// Photon pass (main.cpp:221-249 + the photon half of trace(), :101-128,:158-166).
//
// photon_trace_kernel<FIRST>: one thread owns one photon and keeps its ray in registers from bounce to bounce — there
// are no per-bounce global ray queues for the ~96 % of segments that only meet analytic primitives. A segment whose
// ray reaches the padded root box of a mesh (or of the displaced floor) is NOT traversed in place: the photon is
// suspended into a compacted global queue (warp ballot + one atomic per warp) and the thread retires. The next launch
// (<FIRST = false>) resumes exactly those photons: every lane starts with a BVH traversal, so the warp is dense where the
// single-kernel version ran traversals with 2-5 live lanes; after that segment the photon continues analytically until
// it needs a mesh again and is suspended into the next queue. max_depth launches bound the chain.
// Photon k always draws Philox stream (seed, PASS_PHOTON, k, bounce): any partition of [first, first+count) over
// launches, queues, chunks or GPUs produces the same deposits.
//
// Deposits go to a dense, deterministic table: slot = depth * n + k (k = photon number inside the launch), 64- or 96-byte
// record (DepositRecC / DepositRec) + 32-bit bin; empty slots keep CGRT_KEY_INVALID (pre-filled by a memset). The bin histogram is accumulated by
// the same kernel; bin_scan_* + bin_scatter_kernel then turn it into the cell-grouped order the deposit kernel walks.
// =================================================================================================================
#define CGRT_KEY_INVALID 0xFFFFFFFFu  /* memset pattern of an empty slot */
// Counting-sort bins: 2^22 (16 MB of counters, L2-resident) — 2^23 when the hash table is large (c5, 4096^2: 16x the cells of c3): more bins keep
// the cells apart, so the deposit kernel's groups are larger (c5: 80 -> 67 ms per launch), but the producers' histogram atomics leave the
// L2 (2^24: emission 37 -> 61 ms). PassParams::bin_mask carries the choice.
#define CGRT_BIN_BITS_MIN 22
#define CGRT_BIN_BITS_MAX 23

struct __align__(32) DepositRec {
    double pos[3], nrm[3], flux[3];  // main.cpp:103-122: intersection, face-forwarded normal, photon flux
    int ix, iy, iz, pad0;            // hash.h:38-42 cell of pos
    double pad1;
};
// The record of the float-accumulator mode, 64 bytes = two sectors: the deposit is computed from the float flux there, so the flux travels as
// three floats, and the cell is recomputed from the position by the consumer (four 16-byte loads per record instead of six, a third less of
// the table to write and to read). Position and normal stay fp64: the rare pairs the float filters cannot decide take the reference's test.
struct __align__(32) DepositRecC {
    double pos[3], nrm[3];
    float flux[3];
    uint32_t pad;
};
__host__ __device__ __forceinline__ size_t deposit_rec_bytes(bool compact) { return compact ? sizeof(DepositRecC) : sizeof(DepositRec); }
// Slots of the suspend queue are reserved per warp AHEAD of need (CGRT_QRES at a time, the next range requested while the current one still has
// 32 free slots), so a suspension never waits for its atomic's round trip to the L2 (7 % of the trace kernels' samples before). What a warp
// has reserved and not used when it exits is marked as holes (depth = CGRT_QHOLE), which the consumers skip; the photon queues carry
// CGRT_QHOLE_MARGIN entries beyond the photon count for them.
#define CGRT_QRES 64u
#define CGRT_QHOLE 0xFFFFFFFFu
#define CGRT_QHOLE_MARGIN ((size_t)1 << 19)
struct __align__(16) PhotonState {   // a suspended photon, 128 bytes
    double o[3], d[3], flux[3];      // the ray it was about to trace and the flux it carries
    double nearest, nrm[3];          // closest analytic hit so far (photon_traverse_kernel merges the meshes into it)
    int id, prim;
    uint32_t local, depth;
    double pad;
};

// Bin of a deposit: any well-mixed CGRT_BIN_BITS-bit function of the cell. It only brings the records of one cell next to
// each other (so one warp can reuse the cell's 27 candidate lists); correctness never depends on it, two cells sharing a
// bin are told apart by their coordinates in the deposit kernel.
__device__ __forceinline__ uint32_t cell_bin(int ix, int iy, int iz, uint32_t bin_mask) {
    uint32_t h = (uint32_t)ix * 0x9E3779B1u ^ (uint32_t)iy * 0x85EBCA77u ^ (uint32_t)iz * 0xC2B2AE3Du;
    h ^= h >> 15; h *= 0x2C1B3C6Du; h ^= h >> 12;
    return h & bin_mask;
}

// The BVH part of the closest hit for suspended photons: one thread per queue entry, every lane traverses (dense warps,
// small register footprint). The winner of (analytic hit, mesh hits) is written back into the entry.
// (Measured and rejected: a persistent form in which lanes whose traversal has ended take the next ray of the warp's share as soon as
// 4/8/16 lanes are idle. Live lanes per instruction rose from 6-9 to 11.6, but the instruction count only fell by 14 % (loop and refill
// overhead, 224 bytes of spills at 64 registers) and the issue rate dropped from 61 % to 47 %: 6.8-7.0 ms vs 5.7 ms per round.
// Also rejected: a warp-synchronous traversal that postpones leaves and tests the postponed triangles of 4/8/16 lanes together (the fp64
// triangle test is 27 % of the instructions at 1.7 live lanes): 6.2-6.3 ms — the two ballots per node step cost more than the test saves.)
template <bool COUNT, bool F32>
__global__ void __launch_bounds__(128, CGRT_TRAV_MINB) photon_traverse_kernel(const __grid_constant__ SceneDev S, PhotonState *__restrict__ q,
                                                              const unsigned int *__restrict__ n_in, TravCounters *tcg) {
    const unsigned int total = *n_in;
    TravCounters tcl;
    tcl.node_visits = 0; tcl.tri_tests = 0;
    for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
        // Only (nearest, id) of the running closest hit stay in registers across a traversal; the ray is re-read from the queue entry
        // (L1) for every tree, and a closer hit is written back at once.
        if (q[i].depth == CGRT_QHOLE) continue;  // a reserved slot nobody used
        double nearest = q[i].nearest;
        int id = q[i].id;
        for (int k = 0; k < S.nobj; k++) {
            if (S.obj[k].bvh < 0) continue;  // Bezier objects were resolved by photon_bezier_kernel
            const double2 *p = reinterpret_cast<const double2 *>(q + i);
            double2 q0 = p[0], q1 = p[1], q2 = p[2];
            d3 o = mk(q0.x, q0.y, q1.x), d = mk(q1.y, q2.x, q2.y);
            HitAcc A;
            A.nearest = nearest; A.id = id; A.prim = -1; A.nrm = mk(0, 0, 0);
            double lim;
            if (!deferred_wanted(S, k, o, d, A, lim)) continue;
            if (deferred_resolve<COUNT, false, F32>(S, k, o, d, lim, A, &tcl)) {
                nearest = A.nearest; id = A.id;
                q[i].nearest = A.nearest;
                q[i].nrm[0] = A.nrm.x; q[i].nrm[1] = A.nrm.y; q[i].nrm[2] = A.nrm.z;
                q[i].id = A.id; q[i].prim = A.prim;
            }
        }
    }
    if (COUNT) {
        unsigned int nn = (unsigned int)tcl.node_visits, nt_ = (unsigned int)tcl.tri_tests;
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) { nn += __shfl_xor_sync(0xffffffffu, nn, off); nt_ += __shfl_xor_sync(0xffffffffu, nt_, off); }
        if ((threadIdx.x & 31) == 0) {
            if (nn) atomicAdd(&tcg->node_visits, (unsigned long long)nn);
            if (nt_) atomicAdd(&tcg->tri_tests, (unsigned long long)nt_);
        }
    }
}

// Bezier surfaces of suspended photons: one queue entry per half-warp, one Newton seed per lane (the 16 solves of a ray run side by
// side instead of one after the other in a single thread). Merges with the (len, object index) rule like everything else; the
// traversal kernel that follows skips Bezier objects.
__global__ void __launch_bounds__(128) photon_bezier_kernel(const __grid_constant__ SceneDev S, PhotonState *__restrict__ q, const unsigned int *__restrict__ n_in) {
    const unsigned int total = *n_in;
    const unsigned int half = (blockIdx.x * blockDim.x + threadIdx.x) >> 4, nhalf = (gridDim.x * blockDim.x) >> 4;
    const unsigned int rounds = (total + nhalf - 1) / nhalf;
    for (unsigned int r = 0; r < rounds; r++) {  // both halves of a warp run the same number of rounds: shuffles stay convergent
        const unsigned int i = r * nhalf + half;
        const bool live = i < total && q[i].depth != CGRT_QHOLE;
        d3 o = mk(0, 0, 0), d = mk(0, 0, 1);
        double nearest = CGRT_INF;
        int id = -1;
        if (live) {
            const double2 *p = reinterpret_cast<const double2 *>(q + i);
            double2 q0 = p[0], q1 = p[1], q2 = p[2];
            o = mk(q0.x, q0.y, q1.x); d = mk(q1.y, q2.x, q2.y);
            nearest = q[i].nearest; id = q[i].id;
        }
        for (int k = 0; k < S.nobj; k++) {
            if (S.obj[k].kind != OBJ_BEZIER) continue;
            double len; d3 nv;
            bool hit = live && bezier_intersect_halfwarp(S.bez[S.obj[k].aux], o, d, len, nv);
            if (hit && (len < nearest || (len == nearest && k < id))) {
                nearest = len; id = k;
                if ((threadIdx.x & 15) == 0) {
                    q[i].nearest = len;
                    q[i].nrm[0] = nv.x; q[i].nrm[1] = nv.y; q[i].nrm[2] = nv.z;
                    q[i].id = k; q[i].prim = -1;
                }
            }
        }
    }
}

// trace() of main.cpp:42 called with caller-made rays (cgrt_trace). Photon rays enter the wavefront as queue entries in the state a photon is
// suspended in: the analytic part of the closest hit done, the meshes and Bezier surfaces still to be merged by the kernels that follow.
__global__ void photon_inject_kernel(const __grid_constant__ SceneDev S, unsigned int n, int depth, const double *__restrict__ org,
                                     const double *__restrict__ dir, const double *__restrict__ flux, PhotonState *__restrict__ q, unsigned int *n_out) {
    unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    d3 o = mk(org[3 * i], org[3 * i + 1], org[3 * i + 2]), d = mk(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]);
    HitAcc A;
    analytic_phase(S, o, d, A);
    PhotonState e;
    e.o[0] = o.x; e.o[1] = o.y; e.o[2] = o.z; e.d[0] = d.x; e.d[1] = d.y; e.d[2] = d.z;
    e.flux[0] = flux[3 * i]; e.flux[1] = flux[3 * i + 1]; e.flux[2] = flux[3 * i + 2];
    e.nearest = A.nearest; e.nrm[0] = A.nrm.x; e.nrm[1] = A.nrm.y; e.nrm[2] = A.nrm.z;
    e.id = A.id; e.prim = A.prim; e.local = i; e.depth = (uint32_t)depth; e.pad = 0.0;
    q[i] = e;
    if (i == 0) *n_out = n;
}
// Eye rays: straight into the ray queue of eye_bounce_kernel<false>. path = (y * W + x) * samples + (k mod samples).
__global__ void eye_inject_kernel(unsigned int n, int width, int samples, const double *__restrict__ org, const double *__restrict__ dir,
                                  const double *__restrict__ adj, const int *__restrict__ x, const int *__restrict__ y, RayQueue q) {
    unsigned int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t path = ((uint32_t)y[i] * (uint32_t)width + (uint32_t)x[i]) * (uint32_t)samples + (i % (uint32_t)samples);
    push_ray(q, i, mk(org[3 * i], org[3 * i + 1], org[3 * i + 2]), mk(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]),
             mk(adj[3 * i], adj[3 * i + 1], adj[3 * i + 2]), path, 0u);
}

// Emission (FIRST) or continuation of suspended photons whose pending segment has been resolved by photon_traverse_kernel.
// Persistent threads with refill: a lane whose photon ends (absorbed at the last bounce, missed, or suspended in front of a
// mesh) takes the next photon (FIRST) / queue entry in the same loop iteration, so the warp stays full instead of idling
// until its longest-lived photon finishes (measured before: 19.7 of 32 lanes live in <FIRST>, 8 in the continuation).
// One iteration = [generate a ray] -> [one segment]. The ray of a fresh photon and of a diffuse bounce both come from one
// Philox block through the same code (a fresh photon spends two more draws on its position), so refilling adds no divergence.
enum { PH_NEED = 0, PH_FRESH = 1, PH_DIFFUSE = 2, PH_HAVE_RAY = 3, PH_RESOLVED = 4 };

template <bool FIRST>
__global__ void __launch_bounds__(CGRT_PHOTON_BLOCK, CGRT_TRACE_MINB) photon_trace_kernel(const __grid_constant__ SceneDev S, const __grid_constant__ PassParams P,
                                                                        uint64_t first_index, unsigned int n, const PhotonState *__restrict__ qin,
                                                                        const unsigned int *__restrict__ n_in, PhotonState *__restrict__ qout,
                                                                        unsigned int *n_out, char *__restrict__ rec, int compact, uint32_t *__restrict__ keys,
                                                                        uint32_t *__restrict__ hist, const uint32_t *__restrict__ reach, Counters *ctr,
                                                                        unsigned int *cursor) {
    const unsigned int total = FIRST ? n : *n_in;
    // Work is handed out from the head of the index range: a warp draws CGRT_FETCH consecutive indices at a time from a global cursor
    // (one atomic per CGRT_FETCH photons) and its lanes take them in order. With a static stride per thread the lanes of the grid drift
    // apart (a photon lives 1 to 5 segments) and after ~1000 photons per thread their deposit records, 64- to 96-byte scattered stores, are
    // spread over gigabytes of the table: the emission kernel went from 5.6 to 8.0 ms per 16 Mi photons between 16 Mi and 64 Mi chunks.
    const unsigned int lane_id = threadIdx.x & 31u, lt_mask = (1u << lane_id) - 1u;
    unsigned int wnext = 0, wend = 0;
    bool exhausted = false;
    unsigned int rs = 0, re = 0, nb_reg = 0;  // reserved slots [rs, re) of the output queue (warp-uniform); lane 0 holds the pending next range
    bool res_pending = false;
    const unsigned int qres = total < (1u << 20) ? 32u : CGRT_QRES;  // short queues: fewer holes
    // at most CGRT_FETCH, and small enough that every warp of the grid gets about four turns (the late passes of a round have short queues)
    unsigned int fetch = total / (((gridDim.x * CGRT_PHOTON_BLOCK) >> 5) * 4u);
    fetch = fetch > (unsigned int)CGRT_FETCH ? (unsigned int)CGRT_FETCH : (fetch < 32u ? 32u : (fetch & ~31u));
    unsigned int nseg = 0, nhit = 0;
    int mode = PH_NEED;
    d3 o = mk(0, 0, 0), d = mk(0, 0, 1), flux = mk(0, 0, 0), n_ff = mk(0, 0, 1);
    unsigned int local = 0;
    int depth = 0;
    HitAcc A;
    A.nearest = CGRT_INF; A.id = -1; A.prim = -1; A.nrm = mk(0, 0, 0);
    bool done = false;
    for (;;) {
        // All 32 lanes stay in the loop until the whole warp is out of work and meet here every iteration: without the explicit
        // reconvergence point, lanes that finish a segment early run ahead and the warp falls apart into sub-warps for good.
        __syncwarp();
        // ---- stage 1: a ray for every lane
        {
            bool want = mode == PH_NEED && !done;
            unsigned int need = __ballot_sync(0xffffffffu, want);
            while (need) {  // warp-uniform
                if (wnext >= wend) {
                    if (!exhausted) {
                        unsigned int base = 0;
                        if (lane_id == 0) base = atomicAdd(cursor, fetch);
                        base = __shfl_sync(0xffffffffu, base, 0);
                        if (base >= total) { exhausted = true; }
                        else { wnext = base; wend = (total - base > fetch) ? base + fetch : total; }
                    }
                    if (exhausted) {
                        if (want) done = true;
                        break;
                    }
                }
                const unsigned int avail = wend - wnext, rank = __popc(need & lt_mask), cnt = __popc(need);
                if (want && rank < avail) {
                    const unsigned int next = wnext + rank;
                    want = false;
                    if (FIRST) {
                        local = next; depth = 0;
                        mode = PH_FRESH;
                    } else {
                        const double2 *q = reinterpret_cast<const double2 *>(qin + next);
                        double2 q0 = __ldg(q), q1 = __ldg(q + 1), q2 = __ldg(q + 2), q3 = __ldg(q + 3), q4 = __ldg(q + 4), q5 = __ldg(q + 5), q6 = __ldg(q + 6);
                        o = mk(q0.x, q0.y, q1.x); d = mk(q1.y, q2.x, q2.y); flux = mk(q3.x, q3.y, q4.x);
                        A.nearest = q4.y; A.nrm = mk(q5.x, q5.y, q6.x);
                        long long ip = __double_as_longlong(q6.y);
                        A.id = (int)(uint32_t)ip; A.prim = (int)(uint32_t)(ip >> 32);
                        uint64_t meta = (uint64_t)__double_as_longlong(__ldg(reinterpret_cast<const double *>(q + 7)));
                        local = (uint32_t)meta; depth = (int)(meta >> 32);
                        mode = PH_RESOLVED;  // arrives with the closest hit of its pending segment
                        if ((uint32_t)(meta >> 32) == CGRT_QHOLE) { mode = PH_NEED; want = true; }  // a reserved slot nobody used: take another
                    }
                }
                wnext += cnt < avail ? cnt : avail;
                need = __ballot_sync(0xffffffffu, want);
            }
        }
        if (__all_sync(0xffffffffu, done)) break;
        const uint64_t index = first_index + (uint64_t)local;
        if (!done && (mode == PH_FRESH || mode == PH_DIFFUSE)) {
            // main.cpp:240-246 (fresh: square emitter + uniform sphere) / main.cpp:126 (diffuse bounce: uniform hemisphere)
            Philox g;
            g.init(P.seed, PASS_PHOTON, index, (uint32_t)depth);
            double u0 = g.u01(), u1 = g.u01();
            double a = u0 * 4 - 2, b = u1 * 4 - 2;
            if (mode == PH_FRESH) { u0 = g.u01(); u1 = g.u01(); }
            double z = 1.0 - 2.0 * u0;  // sample_sphere on (u0, u1)
            double sn, cs;
            sincos2pi(u1, sn, cs);
            double r = sqrt(1.0 - z * z);
            d3 s = mk(r * cs, r * sn, z);
            if (mode == PH_FRESH) {
                o = mk(P.light[0], P.light[1], P.light[2]) + mk(a, 0, b);
                d = s;
                flux = mk(700, 700, 700) * (CGRT_PI * 4.0);
            } else {
                if (dot(s, n_ff) < 0) s = -s;  // sample_halfsphere
                d = s;
            }
        }
        // ---- stage 2: one segment
        bool suspended = false;
        if (!done && mode != PH_RESOLVED) {
            analytic_phase(S, o, d, A);
            for (int k = 0; k < S.ndeferred; k++) {
                double lim;
                if (deferred_wanted(S, S.deferred_ix[k], o, d, A, lim)) { suspended = true; break; }
            }
        }
        {   // suspend in front of a mesh: compact into the next queue (warp ballot; slots from the warp's reservation)
            unsigned int m = __ballot_sync(0xffffffffu, suspended);
            unsigned int slot = 0;
            if (m) {  // warp-uniform
                const unsigned int cnt = (unsigned int)__popc(m), avail = re - rs, rank = (unsigned int)__popc(m & lt_mask);
                unsigned int nb = 0;
                if (avail < cnt) {  // the next range is needed: normally requested long ago
                    if (!res_pending && lane_id == 0) nb_reg = atomicAdd(n_out, qres);
                    nb = __shfl_sync(0xffffffffu, nb_reg, 0);
                    res_pending = false;
                }
                slot = rank < avail ? rs + rank : nb + (rank - avail);
                if (avail < cnt) { rs = nb + (cnt - avail); re = nb + qres; }
                else rs += cnt;
                if (!res_pending && re - rs < 32u) {  // ask for the next range now, look at the answer when it is needed
                    if (lane_id == 0) nb_reg = atomicAdd(n_out, qres);
                    res_pending = true;
                }
            }
            if (suspended) {
                double2 *q = reinterpret_cast<double2 *>(qout + slot);
                uint64_t meta = ((uint64_t)(uint32_t)depth << 32) | (uint64_t)local;
                long long ip = ((long long)(uint32_t)A.prim << 32) | (long long)(uint32_t)A.id;
                q[0] = make_double2(o.x, o.y); q[1] = make_double2(o.z, d.x); q[2] = make_double2(d.y, d.z);
                q[3] = make_double2(flux.x, flux.y); q[4] = make_double2(flux.z, A.nearest);
                q[5] = make_double2(A.nrm.x, A.nrm.y); q[6] = make_double2(A.nrm.z, __longlong_as_double(ip));
                q[7] = make_double2(__longlong_as_double((long long)meta), 0.0);
            }
        }
        const bool traced = !done && !suspended;
        nseg += traced ? 1u : 0u;
        if (traced && A.id >= 0) {
            d3 X = o + d * A.nearest;  // main.cpp:68
            // the cell of the hit and its word of the reach map first: the load is in flight while the surface colour (a texel fetch
            // on the floor) and the normal are worked out
            int ix, iy, iz;
            cell_coord(X, P.celllength, P.inv_celllength, ix, iy, iz);
            const uint32_t rh = reach_hash(ix, iy, iz);
            const uint32_t rword = reach ? __ldg(reach + (rh >> 5)) : 0xffffffffu;
            d3 n_old = A.nrm;
            n_ff = A.nrm;
            bool into = true;
            if (dot(n_ff, d) > 0) { n_ff = -n_ff; into = false; }  // main.cpp:73-76
            d3 f = surface_color(S, A.id, X);
            const int mat = S.obj[A.id].material;
            if (mat == MAT_DIFFUSE) {  // the 27-cell gather of main.cpp:103-125 runs in photon_deposit_kernel
                const size_t slot = (size_t)depth * (size_t)n + (size_t)local;
                nhit++;
                const bool reachable = (rword >> (rh & 31u)) & 1u;
                if (reachable) {
                    // streamed: written once, read once by the deposit kernel
                    if (compact) {
                        double2 *r = reinterpret_cast<double2 *>(rec + slot * sizeof(DepositRecC));
                        __stcs(r, make_double2(X.x, X.y)); __stcs(r + 1, make_double2(X.z, n_ff.x)); __stcs(r + 2, make_double2(n_ff.y, n_ff.z));
                        const long long f01 = ((long long)__float_as_uint((float)flux.y) << 32) | (long long)__float_as_uint((float)flux.x);
                        const long long f2 = (long long)__float_as_uint((float)flux.z);
                        __stcs(r + 3, make_double2(__longlong_as_double(f01), __longlong_as_double(f2)));
                    } else {
                        double2 *r = reinterpret_cast<double2 *>(rec + slot * sizeof(DepositRec));
                        __stcs(r, make_double2(X.x, X.y)); __stcs(r + 1, make_double2(X.z, n_ff.x));
                        __stcs(r + 2, make_double2(n_ff.y, n_ff.z)); __stcs(r + 3, make_double2(flux.x, flux.y));
                        __stcs(r + 4, make_double2(flux.z, __longlong_as_double(((long long)(uint32_t)iy << 32) | (uint32_t)ix)));
                        __stcs(r + 5, make_double2(__longlong_as_double((long long)(uint32_t)iz), 0.0));
                    }
                    const uint32_t bin = cell_bin(ix, iy, iz, P.bin_mask);
                    keys[slot] = bin;
                    atomicAdd(hist + bin, 1u);  // histogram of the counting sort, fused into the producer
                }
            }
            if (depth + 1 >= P.max_depth) {
                mode = PH_NEED;
            } else if (mat == MAT_DIFFUSE) {  // main.cpp:126-127: uniform hemisphere (drawn in stage 1), origin NOT offset, flux * f / max(f)
                double p = max3(f.x, f.y, f.z);
                flux = f * flux * (1.0 / p);
                o = X;
                mode = PH_DIFFUSE;
            } else if (mat == MAT_MIRROR) {  // main.cpp:131-134
                d = d - n_ff * 2.0 * dot(n_ff, d);
                o = X + n_ff * CGRT_EPS;
                flux = f * flux * S.obj[A.id].refl;
                mode = PH_HAVE_RAY;
            } else {  // glass, main.cpp:140-164: 50/50 roulette, flux unchanged
                double nc = 1.0, nt = 1.33, nnt = into ? nc / nt : nt / nc, ddn = dot(d, n_ff), cos2t;
                d3 refl_dir = d - n_old * 2.0 * dot(n_old, d);
                if ((cos2t = 1 - nnt * nnt * (1 - ddn * ddn)) < 0) {
                    o = X + n_ff * CGRT_EPS; d = refl_dir;
                } else {
                    d3 refr_dir = normalize(d * nnt - n_old * ((into ? 1 : -1) * (ddn * nnt + sqrt(cos2t))));
                    Philox g;
                    g.init(P.seed, PASS_PHOTON, index, (uint32_t)depth + 1);
                    if (g.u01() < 0.5) { o = X + n_ff * CGRT_EPS; d = refl_dir; }
                    else { o = X - n_ff * CGRT_EPS; d = refr_dir; }
                }
                mode = PH_HAVE_RAY;
            }
            depth++;
        } else if (!done) {
            mode = PH_NEED;  // suspended, or the ray left the scene (main.cpp:64-66)
        }
    }
    {   // what this warp reserved and did not use: holes
        const double2 hole = make_double2(__longlong_as_double((long long)((uint64_t)CGRT_QHOLE << 32)), 0.0);
        for (unsigned int s = rs + lane_id; s < re; s += 32u) reinterpret_cast<double2 *>(qout + s)[7] = hole;
        if (res_pending) {
            const unsigned int nb = __shfl_sync(0xffffffffu, nb_reg, 0);
            for (unsigned int s = nb + lane_id; s < nb + qres; s += 32u) reinterpret_cast<double2 *>(qout + s)[7] = hole;
        }
    }
    // ---- counters: warp reduce, one atomic per warp and counter
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        nseg += __shfl_xor_sync(0xffffffffu, nseg, off);
        nhit += __shfl_xor_sync(0xffffffffu, nhit, off);
    }
    if ((threadIdx.x & 31) == 0) {
        if (nseg) atomicAdd(&ctr->photon_segments, (unsigned long long)nseg);
        if (nhit) atomicAdd(&ctr->diffuse_hits, (unsigned long long)nhit);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// photon_deposit_kernel: the 27-cell gather and deposit of main.cpp:103-125 over deposit records SORTED by cell.
//
// One warp owns a contiguous range of the cell-grouped order. A batch is 32 records, one per lane; the records of the
// batch that lie in one cell form a group and share its candidate list (the hitpoints of the 3x3x3 buckets, read once per
// group instead of once per photon hit): up to 64 candidates at a time are staged in shared memory as 16-byte fp32
// prefilter records {x, y, z, (r + E)^2} (E bounds the float rounding of both positions: the filter can only pass too
// much) and every lane tests its own hit against each of them from a shared-memory broadcast, collecting a 64-bit mask.
// Surviving pairs (~10-15 %) are decided by decide_pair_f32, or by the reference's exact fp64 test (main.cpp:116) where the float
// bounds cannot tell, and deposited with atomics. Two of the 27 cells hashing to one bucket list it twice, like the reference (SURVEY Q13).
//   ACC 0 (fp64 atomics {dflux.xyz, m}) and 2 (per-photon update, deposit_u1): the batch is copied to shared memory (HitShared); the
//         surviving pairs are drained into a per-warp queue and processed 32 at a time by ALL lanes (deposit_pair).
//   ACC 1 (one red.global.add.v4.f32 per deposit): every lane walks its own surviving pairs, its hit in registers.
//   ACC_FIXED (accum_mode 2): the walk of ACC 1 with the fixed-point deposit (deposit_fixed) of every accepted pair.
// ---------------------------------------------------------------------------------------------------------------------
#define CGRT_DEPOSIT_BLOCK 256
#ifndef CGRT_DEPOSIT_MINB
#define CGRT_DEPOSIT_MINB 4   /* resident blocks per SM asked of ptxas (64 registers). Measured with the final kernel: 3 (78 registers) 5.92 ms, 4: 5.45 ms, 5 (48 registers, spills) 5.75 ms, 6: 6.17 ms */
#endif
#ifndef CGRT_DEPOSIT_SPAN
#define CGRT_DEPOSIT_SPAN 256   /* sorted records a warp takes from the cursor at a time. Measured 64 / 128 / 256 / 512 / 1024 / 2048 / 4096: 9.2 / 7.25 / 6.45 / 6.45 / 6.6 / 6.95 / 7.2 ms: consecutive batches of a warp hit the same candidate lists in L1, long spans balance worse */
#endif

__device__ __forceinline__ double4 ldg4(const double4 *p) {  // 32 bytes of a deposit record: streamed (evict-first), two 16-byte loads
    const double2 *q = reinterpret_cast<const double2 *>(p);
    double2 a = __ldcs(q), b = __ldcs(q + 1);
    return make_double4(a.x, a.y, b.x, b.y);
}

// What a warp keeps in shared memory about the 32 records of its batch in the fp64-accumulator modes (ACC 0 and 2; structure of
// arrays, one row per component): the exact fp64 record, because every deposit is computed from the fp64 flux. The float-accumulator
// mode keeps each lane's hit in its registers instead.
struct HitShared {
    double v[9][32];  // pos.xyz, nrm.xyz, flux.xyz
    float f[6][32];   // fp32 pos.xyz, nrm.xyz
};

struct ExactHit {  // the fp64 photon side of one pair
    d3 X, nrm, flux;
};
__device__ __forceinline__ ExactHit exact_hit(const HitShared &H, uint32_t hl) {
    ExactHit e;
    e.X = mk(H.v[0][hl], H.v[1][hl], H.v[2][hl]); e.nrm = mk(H.v[3][hl], H.v[4][hl], H.v[5][hl]); e.flux = mk(H.v[6][hl], H.v[7][hl], H.v[8][hl]);
    return e;
}

__device__ __forceinline__ void red_add_v4(float *ap, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(ap), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

template <int ACC>
__device__ __forceinline__ void deposit_add(void *__restrict__ acc, uint32_t hidx, d3 cc) {
    if (ACC == 0) {
        double *ap = reinterpret_cast<double *>(acc) + 4 * (size_t)hidx;
        atomicAdd(ap, cc.x); atomicAdd(ap + 1, cc.y); atomicAdd(ap + 2, cc.z); atomicAdd(ap + 3, 1.0);
    } else {
        red_add_v4(reinterpret_cast<float *>(acc) + 4 * (size_t)hidx, (float)cc.x, (float)cc.y, (float)cc.z, 1.0f);
    }
}

// The reference's test and deposit in fp64 (main.cpp:116-122) for one pair, from the 64-byte exact record of the hitpoint.
template <int ACC>
__device__ __forceinline__ void deposit_exact(const ExactHit &e, uint32_t hidx, const HpHot *__restrict__ hot, const double *__restrict__ hp_f,
                                              void *__restrict__ acc, unsigned int &ndep) {
    const double2 *hp = reinterpret_cast<const double2 *>(hot + hidx);
    const double2 *fp = reinterpret_cast<const double2 *>(hp_f + 4 * (size_t)hidx);
    double2 a0 = __ldg(hp), a1 = __ldg(hp + 1), b0 = __ldg(hp + 2), b1 = __ldg(hp + 3);
    double2 f0 = __ldg(fp), f1 = __ldg(fp + 1);
    d3 hpos = mk(a0.x, a0.y, a1.x);
    double r2 = a1.y;
    d3 hn = mk(b0.x, b0.y, b1.x);
    d3 dd = hpos - e.X;
    if ((dot(hn, e.nrm) > CGRT_EPS) && (dot(dd, dd) <= r2)) {  // main.cpp:116
        d3 cc = (mk(f0.x, f0.y, f1.x) * e.flux) * (1.0 / CGRT_PI);  // f.mul(flux) * (1/PI), main.cpp:122
        deposit_add<ACC>(acc, hidx, cc);
        ndep++;
    }
}

// The reference's own update rule (main.cpp:116-122, SURVEY Q1 "U1"): an accepted photon shrinks the hitpoint's radius AT ONCE, and the
// next photon is tested against the shrunk radius. r2 is a function of the accepted count alone — r2(n+1) = r2(n) (n a + a) / (n a + 1)
// from the common start (200/height)^2 — so the live state of a hitpoint is one integer: the test reads r2 from a table of the
// reference's recurrence (built on the host in the reference's arithmetic) and an acceptance is a compare-and-swap n -> n+1; a lost race
// re-tests against the newer radius. The reference's flux recurrence flux = (flux + c) g telescopes to flux = r2(n_final) * sum_k c_k /
// r2(n_k): the sums S = sum c / r2_old are accumulated here (fp64 atomics), cgrt_round_update multiplies by the current r2. Photon order
// is arbitrary, as it is between the reference's own racing threads.
struct U1State {
    int *cnt;              // accepted photons per hitpoint (HpArrays::cnt, live)
    const double *r2tab;   // r2 after n accepted photons, n < cap
    int cap;
    int *err;              // fixed-point mode (ACC_FIXED): the context's error word (see deposit_fixed); unused by the other modes
};
__device__ __forceinline__ void deposit_u1(const ExactHit &e, uint32_t hidx, const HpHot *__restrict__ hot, const double *__restrict__ hp_f,
                                           void *__restrict__ acc, const U1State &U, unsigned int &ndep) {
    const double2 *hp = reinterpret_cast<const double2 *>(hot + hidx);
    double2 a0 = __ldg(hp), a1 = __ldg(hp + 1), b0 = __ldg(hp + 2), b1 = __ldg(hp + 3);  // pos and normal never change (r2 in the record is the round-start one)
    d3 hpos = mk(a0.x, a0.y, a1.x), hn = mk(b0.x, b0.y, b1.x);
    if (!(dot(hn, e.nrm) > CGRT_EPS)) return;
    d3 dd = hpos - e.X;
    const double d2 = dot(dd, dd);
    int n_old = *reinterpret_cast<volatile int *>(U.cnt + hidx);
    for (;;) {
        const double r2 = U.r2tab[n_old < U.cap ? n_old : U.cap - 1];
        if (!(d2 <= r2)) return;  // main.cpp:116 against the radius of THIS moment; a later (smaller) radius rejects as well
        const int prev = atomicCAS(U.cnt + hidx, n_old, n_old + 1);
        if (prev == n_old) {
            const double2 *fp = reinterpret_cast<const double2 *>(hp_f + 4 * (size_t)hidx);
            double2 f0 = __ldg(fp), f1 = __ldg(fp + 1);
            d3 cc = (mk(f0.x, f0.y, f1.x) * e.flux) * (1.0 / CGRT_PI);  // f.mul(flux) * (1/PI), main.cpp:122
            double *ap = reinterpret_cast<double *>(acc) + 4 * (size_t)hidx;
            atomicAdd(ap, cc.x / r2); atomicAdd(ap + 1, cc.y / r2); atomicAdd(ap + 2, cc.z / r2);
            ndep++;
            return;
        }
        n_old = prev;
    }
}

// The fp32 decision of one pair that passed the prefilter, from the candidate's filter records q = {x, y, z, (r + E)^2} and
// qn = {nx, ny, nz, (r - E)^2} and the hit's float position h and normal n:
//   distance   s = |fl(hp) - fl(X)|^2 <= (r - E)^2 proves dot(dd, dd) <= r2 (prefilter_inner); the prefilter already had s <= (r + E)^2
//   normals    |fl-dot - dot| <= 5 * 2^-24 * sum |hn_i * nrm_i| (two input roundings and the float evaluation); 1e-6 * sum + 1e-9
//              is the margin used, on either side of CGRT_EPS
// A pair the normal filter rejects is dropped; a pair both filters accept is deposited without touching the hitpoint's exact record.
// Only pairs in the thin shells in between (about 1e-3 of them) take the reference's fp64 test.
enum { PAIR_REJECT, PAIR_ACCEPT, PAIR_EXACT };
__device__ __forceinline__ int decide_pair_f32(float4 q, float4 qn, float hx, float hy, float hz, float nx, float ny, float nz) {
    const float ddx = q.x - hx, ddy = q.y - hy, ddz = q.z - hz;
    const float s = fmaf(ddz, ddz, fmaf(ddy, ddy, ddx * ddx));
    const float dn = fmaf(qn.z, nz, fmaf(qn.y, ny, qn.x * nx));
    const float sn = fmaf(fabsf(qn.z), fabsf(nz), fmaf(fabsf(qn.y), fabsf(ny), fabsf(qn.x * nx)));
    const float mg = fmaf(1e-6f, sn, 1e-9f);
    const float eps = (float)CGRT_EPS;
    if (dn < eps - mg) return PAIR_REJECT;  // the normal test fails whatever the distance
    return (s <= qn.w && dn > eps + mg) ? PAIR_ACCEPT : PAIR_EXACT;
}

// The deposit of an accepted pair in the float walk (accum_mode 1 and 2), per channel: the hitpoint's fp32 f (pre_f) times the photon's
// fp32 flux (the compact record), times fp32 1/pi; round to nearest, never contracted (-fmad=false). The fixed-point mode deposits this
// value for every accepted pair, the thin-shell pairs of the fp64 test included, so that it is a pure function of the pair.
__device__ __forceinline__ float deposit_value_f32(float f, float flux) { return (f * flux) * (float)(1.0 / CGRT_PI); }

// Fixed-point accumulators (accum_mode 2, template id ACC_FIXED): per hitpoint {sum q_x, sum q_y, sum q_z, M} as four int64, where
// q = round-half-even(cf * 2^22) of the value cf above. Integer sums do not depend on the order of the adds, so the round's sums — and
// with them flux, radii, counts and the image — are the same bits whatever the warp order, launch split, rank count or reduction.
// Resolution 2^-22: every cf >= 2 is held exactly, a smaller one to within 2^-23. Range: cf <= 2^16 and M <= 2^24 keep every sum
// <= 2^62; a deposit or a count outside it raises the context's error word (never a silent wrap), which the next synchronising call
// reports. 2^24 is also where the float mode's count lane stops being exact. oracle_fixed/fixed_capi.cpp restates this definition.
#define ACC_FIXED 3
#define CGRT_FIX_SCALE 4194304.0f         /* 2^22 */
#define CGRT_FIX_INV_SCALE (1.0 / 4194304.0)
#define CGRT_FIX_MAX_VALUE 65536.0f       /* 2^16 */
#define CGRT_FIX_MAX_COUNT 16777216ll     /* 2^24 */
enum { FIX_ERR_VALUE = 1, FIX_ERR_COUNT = 2 };

__device__ __forceinline__ long long fixed_q(float cf) { return __float2ll_rn(cf * CGRT_FIX_SCALE); }
// The reds are inline PTX, not atomicAdd / atomicOr: for the builtins the compiler adds its warp-aggregation code around every atomic,
// which took the walk of photon_deposit_kernel<ACC_FIXED> past its 64 registers (148 B of spill stores); with plain reds it has none.
__device__ __forceinline__ void red_add_s64(long long *ap, long long v) {
    asm volatile("red.global.add.u64 [%0], %1;" ::"l"(ap), "l"(v) : "memory");
}
// One accepted pair into hitpoint accumulator ap: three integer reds and the count (PTX has no vector integer red for sm_100a).
__device__ __forceinline__ void deposit_fixed(long long *ap, float cx, float cy, float cz, int *err) {
    if (!(cx <= CGRT_FIX_MAX_VALUE) || !(cy <= CGRT_FIX_MAX_VALUE) || !(cz <= CGRT_FIX_MAX_VALUE)) {  // also catches NaN
        asm volatile("red.global.or.b32 [%0], %1;" ::"l"(err), "r"((int)FIX_ERR_VALUE) : "memory");
        return;
    }
    red_add_s64(ap, fixed_q(cx));
    red_add_s64(ap + 1, fixed_q(cy));
    red_add_s64(ap + 2, fixed_q(cz));
    red_add_s64(ap + 3, 1ll);
}
// The round's fixed-point sums {sq, M} of one hitpoint or pixel as the U2 rule's dflux and M; raises the error word when M > 2^24.
__device__ __forceinline__ void fixed_to_update(long long sx, long long sy, long long sz, long long mc, int *err, double &dx, double &dy, double &dz,
                                                double &m) {
    if (mc > CGRT_FIX_MAX_COUNT) atomicOr(err, FIX_ERR_COUNT);
    dx = (double)sx * CGRT_FIX_INV_SCALE; dy = (double)sy * CGRT_FIX_INV_SCALE; dz = (double)sz * CGRT_FIX_INV_SCALE;
    m = (double)mc;
}
// The reference's fp64 test of one pair (main.cpp:116), from the hitpoint's exact record. It restates the test inside deposit_exact, which
// keeps its own copy so that the kernels of accum_mode 0 and 1 compile to the code that was timed: the two must stay in step.
__device__ __forceinline__ bool accept_exact(const ExactHit &e, uint32_t hidx, const HpHot *__restrict__ hot) {
    const double2 *hp = reinterpret_cast<const double2 *>(hot + hidx);
    double2 a0 = __ldg(hp), a1 = __ldg(hp + 1), b0 = __ldg(hp + 2), b1 = __ldg(hp + 3);
    d3 hpos = mk(a0.x, a0.y, a1.x);
    d3 hn = mk(b0.x, b0.y, b1.x);
    d3 dd = hpos - e.X;
    return (dot(hn, e.nrm) > CGRT_EPS) && (dot(dd, dd) <= a1.y);
}

// One queued pair of the fp64-accumulator modes, its hit in the warp's shared copy. An accepted pair deposits f from global times the
// flux of the shared fp64 record: the deposited value is the reference's.
template <int ACC>
__device__ __forceinline__ void deposit_pair(const HitShared &H, uint32_t hl, uint32_t hidx, float4 q, float4 qn, const HpHot *__restrict__ hot,
                                             const double *__restrict__ hp_f, void *__restrict__ acc, const U1State &U, unsigned int &ndep) {
    static_assert(ACC != 1, "the float-accumulator mode decides its pairs in photon_deposit_kernel's walk");
    if (ACC == 2) {  // per-photon update: the prefilter (round-start radius) only narrows the candidates down
        deposit_u1(exact_hit(H, hl), hidx, hot, hp_f, acc, U, ndep);
        return;
    }
    const int d = decide_pair_f32(q, qn, H.f[0][hl], H.f[1][hl], H.f[2][hl], H.f[3][hl], H.f[4][hl], H.f[5][hl]);
    if (d == PAIR_REJECT) return;
    if (d == PAIR_ACCEPT) {
        const double2 *fp = reinterpret_cast<const double2 *>(hp_f + 4 * (size_t)hidx);
        double2 f0 = __ldg(fp), f1 = __ldg(fp + 1);
        d3 cc = (mk(f0.x, f0.y, f1.x) * mk(H.v[6][hl], H.v[7][hl], H.v[8][hl])) * (1.0 / CGRT_PI);
        deposit_add<0>(acc, hidx, cc);
        ndep++;
        return;
    }
    deposit_exact<0>(exact_hit(H, hl), hidx, hot, hp_f, acc, ndep);
}

template <int ACC>
__global__ void __launch_bounds__(CGRT_DEPOSIT_BLOCK, CGRT_DEPOSIT_MINB) photon_deposit_kernel(const __grid_constant__ PassParams P, const DepositRec *__restrict__ rec,
                                                                            const uint32_t *__restrict__ perm, uint32_t *__restrict__ n_valid,
                                                                            const uint32_t *__restrict__ cell_start,
                                                                            const float4 *__restrict__ pre, const float4 *__restrict__ pre_n,
                                                                            const float4 *__restrict__ pre_f, const HpHot *__restrict__ hot,
                                                                            const double *__restrict__ hp_f, void *__restrict__ acc, Counters *ctr,
                                                                            const U1State U) {
    // per warp: 64 staged candidates (fp32 filter records + hitpoint index) and the queue of (record, candidate) pairs that passed
    // the prefilter
    constexpr int NW = CGRT_DEPOSIT_BLOCK / 32;
    constexpr bool WALK = ACC == 1 || ACC == ACC_FIXED;  // the float walk: compact records, every lane walks its own pairs
    __shared__ float4 cpre_all[NW][64];
    __shared__ float4 cnrm_all[NW][64];
    __shared__ float4 cf_all[WALK ? NW : 1][64];
    __shared__ uint32_t cidx_all[NW][64];
    __shared__ uint32_t queue_all[NW][64];
    __shared__ HitShared hit_all[WALK ? 1 : NW];
    const int lane = threadIdx.x & 31;
    const int wib = threadIdx.x >> 5;
    HitShared &H = hit_all[WALK ? 0 : wib];
    float4 *cpre = cpre_all[wib];
    float4 *cnrm = cnrm_all[wib];
    float4 *cf = cf_all[WALK ? wib : 0];
    uint32_t *cidx = cidx_all[wib];
    uint32_t *queue = queue_all[wib];
    const unsigned int lt = (1u << lane) - 1u;
    unsigned long long cand_total = 0;
    unsigned int ndep = 0, npair = 0, ngroup = 0, nstaged = 0;
    const int idx = lane / 9, idy = (lane / 3) % 3, idz = lane % 3;  // idx outermost, idz innermost (main.cpp:110-112)
    int qn = 0;
    // the candidate list staged last: its cell, its length, the cell's raw candidate count, and whether it is the cell's complete list
    int st_cx = 0, st_cy = 0, st_cz = 0, st_nc = 0;
    uint32_t st_total = 0;
    bool st_ok = false;
    const size_t n_slots = (size_t)__ldg(n_valid);
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&ctr->gathered_hits, (unsigned long long)n_slots);
    // one exact step of the pair queue (ACC 0, 2): 32 queued pairs (fewer at the end of a stage), one per lane. Generic, so that its body is
    // only compiled where it is called.
    auto step = [&](auto first, int count) {
        if (lane < count) {
            const uint32_t e = queue[first + lane];
            const uint32_t hl = e & 31u, b = e >> 8;
            deposit_pair<ACC>(H, hl, cidx[b], cpre[b], cnrm[b], hot, hp_f, acc, U, ndep);
        }
    };
    // spans are handed out from a global cursor (n_valid[1], zeroed by bin_scan_sums_kernel); the next one is requested before the
    // current one is processed, so the atomic's round trip is never waited for
    uint32_t span32 = 0;
    if (lane == 0) span32 = atomicAdd(n_valid + 1, (uint32_t)CGRT_DEPOSIT_SPAN);
    span32 = __shfl_sync(0xffffffffu, span32, 0);
    for (size_t span = span32; span < n_slots;) {
        uint32_t next32 = 0;
        if (lane == 0) next32 = atomicAdd(n_valid + 1, (uint32_t)CGRT_DEPOSIT_SPAN);
        const size_t span_end = span + CGRT_DEPOSIT_SPAN < n_slots ? span + CGRT_DEPOSIT_SPAN : n_slots;
        for (size_t base = span; base < span_end; base += 32) {
            // ---- lane = one deposit record of the batch
            const size_t j = base + lane;
            const bool valid = j < span_end;
            float hx = 0, hy = 0, hz = 0;
            int ix = 0, iy = 0, iz = 0;
            float hown[6] = {0, 0, 0, 0, 0, 0};  // float-accumulator mode: the lane's own hit, normal and flux
            uint32_t src_own = 0;
            if (valid) {
                const uint32_t src = __ldcs(perm + j);
                if (WALK) {
                    // compact record: position and normal fp64, flux as three floats; the cell is recomputed from the position (hash.h:38-42).
                    // The float copy of the hit stays in this lane's registers: in this mode every lane walks its own surviving pairs.
                    const double2 *r = reinterpret_cast<const double2 *>(reinterpret_cast<const DepositRecC *>(rec) + src);
                    const double2 r0 = __ldcs(r), r1 = __ldcs(r + 1), r2 = __ldcs(r + 2), r3 = __ldcs(r + 3);  // streamed once
                    hx = (float)r0.x; hy = (float)r0.y; hz = (float)r1.x;
                    cell_coord(mk(r0.x, r0.y, r1.x), P.celllength, P.inv_celllength, ix, iy, iz);
                    const long long f01 = __double_as_longlong(r3.x), f2 = __double_as_longlong(r3.y);
                    hown[0] = (float)r1.y; hown[1] = (float)r2.x; hown[2] = (float)r2.y;
                    hown[3] = __uint_as_float((uint32_t)f01); hown[4] = __uint_as_float((uint32_t)(f01 >> 32)); hown[5] = __uint_as_float((uint32_t)f2);
                    src_own = src;
                } else {
                    const double4 *r = reinterpret_cast<const double4 *>(rec + src);
                    double4 r0 = ldg4(r), r1 = ldg4(r + 1), r2 = ldg4(r + 2);  // streamed once
                    hx = (float)r0.x; hy = (float)r0.y; hz = (float)r0.z;
                    long long cxy = __double_as_longlong(r2.y);
                    ix = (int)(uint32_t)cxy; iy = (int)(uint32_t)(cxy >> 32); iz = (int)(uint32_t)__double_as_longlong(r2.z);
                    H.f[0][lane] = hx; H.f[1][lane] = hy; H.f[2][lane] = hz;
                    H.f[3][lane] = (float)r0.w; H.f[4][lane] = (float)r1.x; H.f[5][lane] = (float)r1.y;
                    H.v[0][lane] = r0.x; H.v[1][lane] = r0.y; H.v[2][lane] = r0.z;
                    H.v[3][lane] = r0.w; H.v[4][lane] = r1.x; H.v[5][lane] = r1.y;
                    H.v[6][lane] = r1.z; H.v[7][lane] = r1.w; H.v[8][lane] = r2.x;
                }
            }
            __syncwarp();
            unsigned int remaining = __ballot_sync(0xffffffffu, valid);
            while (remaining) {
                // ---- group = the records of the batch that lie in the leader's cell
                const int leader = __ffs(remaining) - 1;
                const int cx = __shfl_sync(0xffffffffu, ix, leader), cy = __shfl_sync(0xffffffffu, iy, leader), cz = __shfl_sync(0xffffffffu, iz, leader);
                const bool in_grp = valid && ix == cx && iy == cy && iz == cz;
                const unsigned int grp = __ballot_sync(0xffffffffu, in_grp) & remaining;
                remaining &= ~grp;
                // A cell's records are consecutive in the sorted order, so the batch that follows usually starts with the cell this one ended
                // with: when the candidates staged last belong to the same cell and were the cell's whole (culled) list, they are used again
                // as they are — the 27 bucket ranges, the filter records and the cull are read and done once per run of a cell, not per batch.
                const bool reuse = st_ok && cx == st_cx && cy == st_cy && cz == st_cz;  // warp-uniform
                uint32_t beg = 0, cnt = 0, excl = 0, total = st_total;
                if (!reuse) {
                    // the 27 bucket ranges of this cell (main.cpp:105-113)
                    if (lane < 27) {
                        uint32_t key = cell_hash(cx - 1 + idx, cy - 1 + idy, cz - 1 + idz, P.hashsize);
                        beg = __ldg(cell_start + key);
                        cnt = __ldg(cell_start + key + 1) - beg;
                    }
                    uint32_t incl = cnt;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
                        if (lane >= o) incl += y;
                    }
                    excl = incl - cnt;
                    total = __shfl_sync(0xffffffffu, incl, 31);
                    if (lane == 0) { ngroup++; nstaged += total; }
                    st_ok = false;  // the staged list is about to be overwritten
                }
                cand_total += (lane == 0) ? (unsigned long long)total * (unsigned int)__popc(grp) : 0ull;
                // the cell of this group as a float box (a hair larger): a candidate whose sphere does not reach the box cannot accept
                // any hit of the group and is dropped once per group instead of being tested against every hit
                const float bx0 = (float)(-35.0 + (double)cx * P.celllength), by0 = (float)(-35.0 + (double)cy * P.celllength),
                            bz0 = (float)(-15.0 + (double)cz * P.celllength), bw = (float)P.celllength;
                const float bm = 1e-5f * (fabsf(bx0) + fabsf(by0) + fabsf(bz0) + bw + 1.0f);
                uint32_t c0 = 0;       // raw candidates consumed so far
                bool first_list = true;
                for (;;) {
                    int nc = st_nc;
                    if (!reuse) {
                        // ---- stage: append the survivors of 32 raw candidates at a time until more than 32 are listed (the list holds 64)
                        nc = 0;
                        while (c0 < total && nc <= 32) {
                            const uint32_t c = c0 + lane;
                            c0 += 32;
                            int lo = 0;  // owner bucket of candidate c = last lane < 27 whose excl <= c (shuffle binary search)
#pragma unroll
                            for (int step_ = 16; step_ >= 1; step_ >>= 1) {
                                int probe = lo + step_;
                                uint32_t e = __shfl_sync(0xffffffffu, excl, probe & 31);
                                if (probe < 27 && e <= c) lo = probe;
                            }
                            const uint32_t e_lo = __shfl_sync(0xffffffffu, excl, lo);
                            const uint32_t b_lo = __shfl_sync(0xffffffffu, beg, lo);
                            bool keep = false;
                            uint32_t hidx = 0;
                            float4 q = make_float4(0.f, 0.f, 0.f, -1.f), q_n = q, q_f = q;
                            if (c < total) {
                                hidx = b_lo + (c - e_lo);
                                q = __ldg(pre + hidx);
                                const float ex = fmaxf(fmaxf(bx0 - bm - q.x, q.x - (bx0 + bw + bm)), 0.f);
                                const float ey = fmaxf(fmaxf(by0 - bm - q.y, q.y - (by0 + bw + bm)), 0.f);
                                const float ez = fmaxf(fmaxf(bz0 - bm - q.z, q.z - (bz0 + bw + bm)), 0.f);
                                keep = fmaf(ez, ez, fmaf(ey, ey, ex * ex)) <= q.w;
                                if (keep) {  // the other two filter records only for candidates that survive the cull (c5: deposit 89 -> 84 ms)
                                    q_n = __ldg(pre_n + hidx);
                                    if (WALK) q_f = __ldg(pre_f + hidx);
                                }
                            }
                            const unsigned int km = __ballot_sync(0xffffffffu, keep);
                            if (keep) {
                                const int at = nc + __popc(km & lt);
                                cpre[at] = q;
                                cnrm[at] = q_n;
                                if (WALK) cf[at] = q_f;
                                cidx[at] = hidx;
                            }
                            nc += __popc(km);
                        }
                        // pad the staged list to a multiple of 8 with records no hit can pass, so that the scan runs in unguarded blocks of 8
                        if (lane < 8 && nc + lane < ((nc + 7) & ~7)) cpre[nc + lane] = make_float4(0.f, 0.f, 0.f, -1.f);
                        __syncwarp();
                        if (c0 >= total && first_list) { st_ok = true; st_cx = cx; st_cy = cy; st_cz = cz; st_nc = nc; st_total = total; }
                        first_list = false;
                    }
                    // ---- prefilter: every lane tests its own hit against the staged candidates (shared-memory broadcast)
                    unsigned int m_lo = 0, m_hi = 0;
                    {
                        const int n_lo = nc < 32 ? nc : 32;
                        for (int k0 = 0; k0 < n_lo; k0 += 8) {
                            unsigned int bits = 0;
#pragma unroll
                            for (int j = 0; j < 8; j++) {
                                const float4 q = cpre[k0 + j];
                                const float ddx = q.x - hx, ddy = q.y - hy, ddz = q.z - hz;
                                bits |= (fmaf(ddz, ddz, fmaf(ddy, ddy, ddx * ddx)) <= q.w) ? (1u << j) : 0u;
                            }
                            m_lo |= bits << k0;
                        }
                        for (int k0 = 32; k0 < nc; k0 += 8) {
                            unsigned int bits = 0;
#pragma unroll
                            for (int j = 0; j < 8; j++) {
                                const float4 q = cpre[k0 + j];
                                const float ddx = q.x - hx, ddy = q.y - hy, ddz = q.z - hz;
                                bits |= (fmaf(ddz, ddz, fmaf(ddy, ddy, ddx * ddx)) <= q.w) ? (1u << j) : 0u;
                            }
                            m_hi |= bits << (k0 - 32);
                        }
                    }
                    if (!((grp >> lane) & 1u)) { m_lo = 0; m_hi = 0; }
                    if constexpr (WALK) {
                        // Float accumulators: every lane walks the candidates that passed its own prefilter, its hit in registers — no pair
                        // queue and no shared-memory copy of the hits. The lanes idle while the busiest one finishes (4.8 pairs per hit
                        // on average, ~10 at most), but the shared-memory traffic of the queue form costs more on the pipe that bounds
                        // this kernel (c3: 5.55 -> 5.42 ms, c2: 1.55 -> 1.44 ms). An accepted pair deposits from the fp32 copy of f.
                        unsigned int mine = 0;
                        while (m_lo | m_hi) {
                            int b;
                            if (m_lo) { b = __ffs(m_lo) - 1; m_lo &= m_lo - 1; }
                            else { b = 32 + __ffs(m_hi) - 1; m_hi &= m_hi - 1; }
                            mine++;
                            const int d = decide_pair_f32(cpre[b], cnrm[b], hx, hy, hz, hown[0], hown[1], hown[2]);
                            if (d == PAIR_REJECT) continue;
                            const uint32_t hidx = cidx[b];
                            if constexpr (ACC == ACC_FIXED) {
                                if (d == PAIR_EXACT) {  // the thin shells: the reference's fp64 test decides, the deposit is the same value
                                    const double2 *r = reinterpret_cast<const double2 *>(reinterpret_cast<const DepositRecC *>(rec) + src_own);
                                    const double2 r0 = __ldcs(r), r1 = __ldcs(r + 1), r2 = __ldcs(r + 2);
                                    ExactHit e;
                                    e.X = mk(r0.x, r0.y, r1.x); e.nrm = mk(r1.y, r2.x, r2.y);
                                    if (!accept_exact(e, hidx, hot)) continue;
                                }
                                const float4 qf = cf[b];
                                deposit_fixed(reinterpret_cast<long long *>(acc) + 4 * (size_t)hidx, deposit_value_f32(qf.x, hown[3]),
                                              deposit_value_f32(qf.y, hown[4]), deposit_value_f32(qf.z, hown[5]), U.err);
                                ndep++;
                            } else if (d == PAIR_ACCEPT) {
                                const float4 qf = cf[b];
                                red_add_v4(reinterpret_cast<float *>(acc) + 4 * (size_t)hidx, deposit_value_f32(qf.x, hown[3]), deposit_value_f32(qf.y, hown[4]),
                                           deposit_value_f32(qf.z, hown[5]), 1.0f);
                                ndep++;
                            } else {
                                // the thin shells the float filters cannot decide: the reference's fp64 test on the record itself
                                const double2 *r = reinterpret_cast<const double2 *>(reinterpret_cast<const DepositRecC *>(rec) + src_own);
                                const double2 r0 = __ldcs(r), r1 = __ldcs(r + 1), r2 = __ldcs(r + 2);
                                ExactHit e;
                                e.X = mk(r0.x, r0.y, r1.x); e.nrm = mk(r1.y, r2.x, r2.y);
                                e.flux = mk((double)hown[3], (double)hown[4], (double)hown[5]);
                                deposit_exact<1>(e, hidx, hot, hp_f, acc, ndep);
                            }
                        }
                        for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
                        npair += (lane == 0) ? mine : 0u;
                        __syncwarp();
                        if (reuse || c0 >= total) break;
                    } else {
                    // ---- drain: one surviving pair per lane and round into the queue; 32 queued pairs = one exact step
                    while (__any_sync(0xffffffffu, (m_lo | m_hi) != 0u)) {
                        const bool has = (m_lo | m_hi) != 0u;
                        int b = 0;
                        if (m_lo) { b = __ffs(m_lo) - 1; m_lo &= m_lo - 1; }
                        else if (m_hi) { b = 32 + __ffs(m_hi) - 1; m_hi &= m_hi - 1; }
                        const unsigned int pm = __ballot_sync(0xffffffffu, has);
                        if (has) queue[qn + __popc(pm & lt)] = (uint32_t)lane | ((uint32_t)b << 8);
                        qn += __popc(pm);
                        npair += (lane == 0) ? (unsigned int)__popc(pm) : 0u;
                        if (qn >= 32) {
                            __syncwarp();
                            qn -= 32;
                            step(qn, 32);
                            __syncwarp();
                        }
                    }
                    // the queue refers to the staged candidates: empty it before they are restaged
                    __syncwarp();
                    step(0, qn);
                    qn = 0;
                    __syncwarp();
                    if (reuse || c0 >= total) break;
                    }
                }
            }
        }
        span = (size_t)__shfl_sync(0xffffffffu, next32, 0);
    }
    // counters: warp-reduce then one atomic per warp
    unsigned long long dep_total = ndep;
    for (int o = 16; o > 0; o >>= 1) {
        cand_total += __shfl_xor_sync(0xffffffffu, cand_total, o);
        dep_total += __shfl_xor_sync(0xffffffffu, dep_total, o);
    }
    if (lane == 0) {
        if (cand_total) atomicAdd(&ctr->candidates, cand_total);
        if (dep_total) atomicAdd(&ctr->deposits, dep_total);
        if (npair) atomicAdd(&ctr->exact_tests, (unsigned long long)npair);
        if (ngroup) atomicAdd(&ctr->cell_groups, (unsigned long long)ngroup);
        if (nstaged) atomicAdd(&ctr->staged_candidates, (unsigned long long)nstaged);
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Counting sort of the deposit slots by bin (not stable: the order inside a bin is irrelevant). The histogram comes from
// photon_trace_kernel; three small kernels scan it exclusively in place, and the scatter turns every valid slot into one
// entry of `perm` with a returning atomic on its bin cursor.
// ---------------------------------------------------------------------------------------------------------------------
#define CGRT_SCAN_BLOCK 1024
#define CGRT_SCAN_ITEMS 4

__device__ __forceinline__ uint32_t block_exclusive_scan_1024(uint32_t v, uint32_t *warp_sums, uint32_t &block_total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
        uint32_t s = warp_sums[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, s, o);
            if (lane >= o) s += y;
        }
        warp_sums[lane] = s;
    }
    __syncthreads();
    block_total = warp_sums[31];
    return (wid > 0 ? warp_sums[wid - 1] : 0u) + x - v;
}
// phase 1: per block of 4096 counters, exclusive scan in place + block total
__global__ void __launch_bounds__(CGRT_SCAN_BLOCK) bin_scan_blocks_kernel(uint32_t *__restrict__ hist, uint32_t *__restrict__ block_sums) {
    __shared__ uint32_t ws[32];
    uint4 *p = reinterpret_cast<uint4 *>(hist) + (size_t)blockIdx.x * CGRT_SCAN_BLOCK + threadIdx.x;
    uint4 v = *p;
    uint32_t total;
    uint32_t ex = block_exclusive_scan_1024(v.x + v.y + v.z + v.w, ws, total);
    *p = make_uint4(ex, ex + v.x, ex + v.x + v.y, ex + v.x + v.y + v.z);
    if (threadIdx.x == 0) block_sums[blockIdx.x] = total;
}
// phase 2: one block scans the (<= 1024) block totals; the grand total is the number of valid deposit slots
__global__ void __launch_bounds__(CGRT_SCAN_BLOCK) bin_scan_sums_kernel(uint32_t *__restrict__ block_sums, int nblocks, uint32_t *__restrict__ n_valid) {
    __shared__ uint32_t ws[32];
    // every thread owns `per` consecutive block totals (1 for up to 2^22 bins)
    const int per = (nblocks + CGRT_SCAN_BLOCK - 1) / CGRT_SCAN_BLOCK, first = (int)threadIdx.x * per;
    uint32_t v = 0;
    for (int j = 0; j < per; j++) v += first + j < nblocks ? block_sums[first + j] : 0u;
    uint32_t total;
    uint32_t ex = block_exclusive_scan_1024(v, ws, total);
    for (int j = 0; j < per; j++)
        if (first + j < nblocks) { const uint32_t c = block_sums[first + j]; block_sums[first + j] = ex; ex += c; }
    if (threadIdx.x == 0) { n_valid[0] = total; n_valid[1] = 0u; }  // [1]: the span cursor of photon_deposit_kernel
}
// phase 3 fused into the scatter: cursor of bin b = hist[b] + block_sums[b / 4096]
__global__ void __launch_bounds__(256) bin_scatter_kernel(const uint32_t *__restrict__ keys, size_t n_slots, uint32_t *__restrict__ hist,
                                                          const uint32_t *__restrict__ block_sums, uint32_t *__restrict__ perm) {
    for (size_t s = (size_t)blockIdx.x * blockDim.x + threadIdx.x; s < n_slots; s += (size_t)gridDim.x * blockDim.x) {
        uint32_t b = __ldg(keys + s);
        if (b == CGRT_KEY_INVALID) continue;
        uint32_t pos = atomicAdd(hist + b, 1u) + __ldg(block_sums + (b >> 12));
        perm[pos] = (uint32_t)s;
    }
}

// =================================================================================================================
// K12: per-round radius / flux update (main.cpp:119-122 batched over a round, SURVEY Q1 "U2"):
//   g = (n a + a M) / (n a + M);  flux = (flux + dflux) g;  r2 *= g;  n += M.   Clears the accumulators.
// =================================================================================================================
__device__ __forceinline__ double u2_gain(int n, double m, double alpha) {
    double na = n * alpha;
    return (na + alpha * m) / (na + m);
}
// The rule for hitpoint k, which accepted m > 0 photons carrying dflux = (dx, dy, dz) this round.
__device__ __forceinline__ void round_update_tail(const HpArrays &A, unsigned int k, double alpha, double dx, double dy, double dz, double m) {
    int cnt = A.cnt[k];
    double g = u2_gain(cnt, m, alpha);
    double *fl = A.flux + 4 * (size_t)k;
    fl[0] = (fl[0] + dx) * g;
    fl[1] = (fl[1] + dy) * g;
    fl[2] = (fl[2] + dz) * g;
    const HpHot hh = A.hot[k];
    set_radius(A, k, hh, hh.r2 * g);
    A.cnt[k] = cnt + (int)m;
}

template <int ACC>
__global__ void round_update_kernel(unsigned int n, double alpha, HpArrays A, void *__restrict__ acc) {
    unsigned int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    double dx, dy, dz, m;
    if (ACC == 0) {
        double4 *ap = reinterpret_cast<double4 *>(acc) + k;
        double4 a = *ap;
        dx = a.x; dy = a.y; dz = a.z; m = a.w;
        *ap = make_double4(0, 0, 0, 0);
    } else {
        float4 *ap = reinterpret_cast<float4 *>(acc) + k;
        float4 a = *ap;
        dx = a.x; dy = a.y; dz = a.z; m = a.w;
        *ap = make_float4(0, 0, 0, 0);
    }
    if (m > 0) round_update_tail(A, k, alpha, dx, dy, dz, m);
}
// The same for the fixed-point accumulators (accum_mode 2).
__global__ void round_update_fixed_kernel(unsigned int n, double alpha, HpArrays A, long long *__restrict__ acc, int *err) {
    unsigned int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    longlong2 *ap = reinterpret_cast<longlong2 *>(acc + 4 * (size_t)k);
    const longlong2 a = ap[0], b = ap[1];
    ap[0] = make_longlong2(0, 0); ap[1] = make_longlong2(0, 0);
    double dx, dy, dz, m;
    fixed_to_update(a.x, a.y, b.x, b.y, err, dx, dy, dz, m);
    if (m > 0) round_update_tail(A, k, alpha, dx, dy, dz, m);
}

// =================================================================================================================
// SPPM fold: the U2 rule above per PIXEL. One thread per pixel walks the round's visible points of that pixel in canonical order
// (pix_perm, as image_gather_kernel does, so the fp64 sums are deterministic), sums their accumulators {dflux, M}, clears them, and
// updates the pixel's statistics:  g = (n a + a M) / (n a + M);  tau = (tau + dflux) g;  R2 *= g;  n += M.
// =================================================================================================================
template <int ACC>
__global__ void sppm_fold_kernel(unsigned int npix, double alpha, const uint32_t *__restrict__ pix_start, const uint32_t *__restrict__ pix_perm,
                                 void *__restrict__ acc, double *__restrict__ tau, double *__restrict__ r2, int *__restrict__ cnt) {
    unsigned int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    double dx = 0, dy = 0, dz = 0, m = 0;
    for (uint32_t j = pix_start[p]; j < pix_start[p + 1]; j++) {
        uint32_t k = pix_perm[j];
        if (ACC == 0) {
            double4 *ap = reinterpret_cast<double4 *>(acc) + k;
            double4 a = *ap;
            dx += a.x; dy += a.y; dz += a.z; m += a.w;
            *ap = make_double4(0, 0, 0, 0);
        } else {
            float4 *ap = reinterpret_cast<float4 *>(acc) + k;
            float4 a = *ap;
            dx += (double)a.x; dy += (double)a.y; dz += (double)a.z; m += (double)a.w;
            *ap = make_float4(0, 0, 0, 0);
        }
    }
    if (m > 0) {
        int c = cnt[p];
        double g = u2_gain(c, m, alpha);
        double *t = tau + 4 * (size_t)p;
        t[0] = (t[0] + dx) * g;
        t[1] = (t[1] + dy) * g;
        t[2] = (t[2] + dz) * g;
        r2[p] *= g;
        cnt[p] = c + (int)m;
    }
}
// The same for the fixed-point accumulators (accum_mode 2): the pixel's integer sums, converted once. M is checked per pixel.
__global__ void sppm_fold_fixed_kernel(unsigned int npix, double alpha, const uint32_t *__restrict__ pix_start, const uint32_t *__restrict__ pix_perm,
                                       long long *__restrict__ acc, double *__restrict__ tau, double *__restrict__ r2, int *__restrict__ cnt, int *err) {
    unsigned int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    long long sx = 0, sy = 0, sz = 0, sm = 0;
    for (uint32_t j = pix_start[p]; j < pix_start[p + 1]; j++) {
        longlong2 *ap = reinterpret_cast<longlong2 *>(acc + 4 * (size_t)pix_perm[j]);
        const longlong2 a = ap[0], b = ap[1];
        sx += a.x; sy += a.y; sz += b.x; sm += b.y;
        ap[0] = make_longlong2(0, 0); ap[1] = make_longlong2(0, 0);
    }
    double dx, dy, dz, m;
    fixed_to_update(sx, sy, sz, sm, err, dx, dy, dz, m);
    if (m > 0) {
        int c = cnt[p];
        double g = u2_gain(c, m, alpha);
        double *t = tau + 4 * (size_t)p;
        t[0] = (t[0] + dx) * g;
        t[1] = (t[1] + dy) * g;
        t[2] = (t[2] + dz) * g;
        r2[p] *= g;
        cnt[p] = c + (int)m;
    }
}

// =================================================================================================================
// The round's exchange over peer memory (one box, NVLink / NVSwitch) fused with the update: no collective library call in the round.
// Every rank keeps its accumulators in a cudaMalloc block that all ranks have mapped (CUDA IPC between processes, peer access inside one
// process). After its deposit kernel a rank publishes "round r deposited" in every peer's flag array; on a side stream a one-block
// kernel waits until all ranks have published r, then ONE kernel reads every rank's accumulators straight out of their memory (P2P
// loads, ranks summed in rank order so that every rank gets the same bits), applies the round update to its own replica of the
// hitpoints and clears its own accumulators of the round after. The accumulators are double-buffered by round parity: a buffer is only
// written again two rounds later, and a rank that has published round r has finished reading round r-1 everywhere (its update r-1
// precedes its deposit r), so no second handshake is needed. Only the NEXT round's deposit kernel waits for this — the next round's
// emission and traversal run underneath, which also absorbs the skew between ranks that a synchronous all-reduce pays every round.
// =================================================================================================================
#define CGRT_MAX_PEERS 16
struct PeerPtrs {
    void *p[CGRT_MAX_PEERS];
};
__device__ __forceinline__ void st_release_sys(int *p, int v) { asm volatile("st.release.sys.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ int ld_acquire_sys(const int *p) {
    int v;
    asm volatile("ld.acquire.sys.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// flags.p[g] = rank g's flag array (world ints); this rank writes its own slot in each of them
__global__ void peer_signal_kernel(PeerPtrs flags, int rank, int world, int value) {
    const int g = threadIdx.x;
    if (g < world) {
        __threadfence_system();
        st_release_sys(reinterpret_cast<int *>(flags.p[g]) + rank, value);
    }
}
// waits until every slot of this rank's own flag array has reached `value`; gives up after `timeout_ns` and raises *err (never hangs the GPU)
__global__ void peer_wait_kernel(const int *my_flags, int world, int value, unsigned long long timeout_ns, int *err) {
    const int g = threadIdx.x;
    if (g >= world) return;
    unsigned long long t0, t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (ld_acquire_sys(my_flags + g) < value) {
        __nanosleep(200);
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if (t - t0 > timeout_ns) { atomicExch(err, 1 + g); return; }
    }
}
// acc.p[g] = rank g's accumulators of this round's parity; clear_next = this rank's accumulators of the other parity.
// The remote loads of one hitpoint are issued together (eight float4 / four double4 in flight per thread) — one after the other they
// cost a NVLink round trip each (measured at 8 GPUs: c2 5.17 ms per round against 4.71 with an in-stream ncclAllReduce). 64-thread
// blocks so that a block fits into the registers the persistent emission kernel of the next round leaves free on an SM.
template <int ACC>
__global__ void __launch_bounds__(64) peer_reduce_update_kernel(unsigned int n, double alpha, HpArrays A, const __grid_constant__ PeerPtrs acc, int world,
                                                                void *__restrict__ clear_next) {
    unsigned int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    // The declaration order reaches ptxas's register assignment of <0>: this one compiles to the code that was timed (other orders
    // compile differently, and re-timing this kernel takes two GPUs).
    double dz = 0, m = 0, dy = 0, dx = 0;
    if (ACC == 0) {
        for (int g0 = 0; g0 < world; g0 += 4) {
            double2 lo[4], hi[4];
#pragma unroll
            for (int j = 0; j < 4; j++) {
                lo[j] = make_double2(0, 0); hi[j] = make_double2(0, 0);
                if (g0 + j < world) {
                    const double2 *ap = reinterpret_cast<const double2 *>(reinterpret_cast<const double4 *>(acc.p[g0 + j]) + k);
                    lo[j] = __ldcg(ap); hi[j] = __ldcg(ap + 1);
                }
            }
#pragma unroll
            for (int j = 0; j < 4; j++) { dx += lo[j].x; dy += lo[j].y; dz += hi[j].x; m += hi[j].y; }  // rank order; an absent rank adds 0
        }
        reinterpret_cast<double4 *>(clear_next)[k] = make_double4(0, 0, 0, 0);
    } else {
        float fx = 0, fy = 0, fz = 0, fm = 0;  // float sums in rank order: what an all-reduce of float accumulators produces, identical on every rank
        for (int g0 = 0; g0 < world; g0 += 8) {
            float4 v[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
                v[j] = make_float4(0, 0, 0, 0);
                if (g0 + j < world) v[j] = __ldcg(reinterpret_cast<const float4 *>(acc.p[g0 + j]) + k);
            }
#pragma unroll
            for (int j = 0; j < 8; j++) { fx += v[j].x; fy += v[j].y; fz += v[j].z; fm += v[j].w; }
        }
        dx = fx; dy = fy; dz = fz; m = fm;
        reinterpret_cast<float4 *>(clear_next)[k] = make_float4(0, 0, 0, 0);
    }
    if (m > 0) round_update_tail(A, k, alpha, dx, dy, dz, m);
}
// The same for the fixed-point accumulators (accum_mode 2): integer sums give the same bits in any rank order; M is checked after the
// exchange.
__global__ void __launch_bounds__(64) peer_reduce_update_fixed_kernel(unsigned int n, double alpha, HpArrays A, const __grid_constant__ PeerPtrs acc,
                                                                      int world, long long *__restrict__ clear_next, int *err) {
    unsigned int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    long long sx = 0, sy = 0, sz = 0, sm = 0;
    for (int g0 = 0; g0 < world; g0 += 4) {
        longlong2 lo[4], hi[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            lo[j] = make_longlong2(0, 0); hi[j] = make_longlong2(0, 0);
            if (g0 + j < world) {
                const longlong2 *ap = reinterpret_cast<const longlong2 *>(reinterpret_cast<const long long *>(acc.p[g0 + j]) + 4 * (size_t)k);
                lo[j] = __ldcg(ap); hi[j] = __ldcg(ap + 1);
            }
        }
#pragma unroll
        for (int j = 0; j < 4; j++) { sx += lo[j].x; sy += lo[j].y; sz += hi[j].x; sm += hi[j].y; }
    }
    longlong2 *cn = reinterpret_cast<longlong2 *>(clear_next + 4 * (size_t)k);
    cn[0] = make_longlong2(0, 0); cn[1] = make_longlong2(0, 0);
    double dx, dy, dz, m;
    fixed_to_update(sx, sy, sz, sm, err, dx, dy, dz, m);
    if (m > 0) round_update_tail(A, k, alpha, dx, dy, dz, m);
}

// Per-photon update mode: the counts are live; a "round update" only folds them into what the next round's filters and the image read:
// r2 = table[n], flux = S * r2 (see deposit_u1), filter radii. The sums S stay in the accumulator buffer for the whole render.
__global__ void round_update_u1_kernel(unsigned int n, HpArrays A, const double *__restrict__ S, const double *__restrict__ r2tab, int cap, int *maxcnt) {
    unsigned int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int cnt = A.cnt[k];
    if (cnt > *maxcnt) atomicMax(maxcnt, cnt);
    const double r2 = r2tab[cnt < cap ? cnt : cap - 1];
    double *fl = A.flux + 4 * (size_t)k;
    fl[0] = S[4 * (size_t)k] * r2; fl[1] = S[4 * (size_t)k + 1] * r2; fl[2] = S[4 * (size_t)k + 2] * r2;
    const HpHot hh = A.hot[k];
    if (hh.r2 != r2) set_radius(A, k, hh, r2);
}

// =================================================================================================================
// K13: image gather (main.cpp:252-258). One thread per pixel walks that pixel's hitpoints in canonical order
// (pix_perm is a stable sort of the canonical order by pixel), so the fp64 sums equal the reference loop's.
// =================================================================================================================
__device__ __forceinline__ int gamma_corr(double x) { return int(pow(1 - exp(-x), 1 / 2.2) * 255 + .5); }  // util.h:45-47

// pixel p's linear value, and (rgb8 != nullptr) its tone-mapped bytes; main.cpp:403-411: row i of the PNG is image[height-1-i]
__device__ __forceinline__ void write_pixel(int width, int height, unsigned int p, d3 acc, double *rgb, uint8_t *rgb8) {
    rgb[3 * (size_t)p] = acc.x; rgb[3 * (size_t)p + 1] = acc.y; rgb[3 * (size_t)p + 2] = acc.z;
    if (rgb8) {
        int h = p / width, w = p % width;
        size_t q = (size_t)(height - 1 - h) * width + w;
        rgb8[3 * q] = (uint8_t)(char)gamma_corr(acc.x);
        rgb8[3 * q + 1] = (uint8_t)(char)gamma_corr(acc.y);
        rgb8[3 * q + 2] = (uint8_t)(char)gamma_corr(acc.z);
    }
}

__global__ void image_gather_kernel(int width, int height, double n_emitted, const uint32_t *__restrict__ pix_start,
                                    const uint32_t *__restrict__ pix_perm, const HpHot *__restrict__ hot, const double *__restrict__ flux,
                                    double *__restrict__ rgb, uint8_t *__restrict__ rgb8) {
    unsigned int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= (unsigned int)(width * height)) return;
    d3 acc = mk(0, 0, 0);
    for (uint32_t j = pix_start[p]; j < pix_start[p + 1]; j++) {
        uint32_t k = pix_perm[j];
        double r2 = hot[k].r2;
        d3 fl = mk(flux[4 * (size_t)k], flux[4 * (size_t)k + 1], flux[4 * (size_t)k + 2]);
        acc = acc + fl * (1.0 / (CGRT_PI * r2 * n_emitted));
    }
    write_pixel(width, height, p, acc, rgb, rgb8);
}

// SPPM image: main.cpp:252-258 with the pixel's statistics in place of its hitpoints' — the expression and the tone map / flip of
// image_gather_kernel, so that a pixel with a single visible point gives PPM's bits.
__global__ void sppm_image_kernel(int width, int height, double n_emitted, const double *__restrict__ tau, const double *__restrict__ r2,
                                  double *__restrict__ rgb, uint8_t *__restrict__ rgb8) {
    unsigned int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= (unsigned int)(width * height)) return;
    d3 acc = mk(0, 0, 0);
    d3 fl = mk(tau[4 * (size_t)p], tau[4 * (size_t)p + 1], tau[4 * (size_t)p + 2]);
    acc = acc + fl * (1.0 / (CGRT_PI * r2[p] * n_emitted));
    write_pixel(width, height, p, acc, rgb, rgb8);
}

// =================================================================================================================
// average.cpp:19-65: out = sum_k (img_k / n) per byte (integer division first, then the sum), and its linear-domain counterpart.
// The n images are stored back to back in `imgs` (n x count).
// =================================================================================================================
__global__ void average_u8_kernel(const uint8_t *__restrict__ imgs, int n, int64_t count, uint8_t *__restrict__ out) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    unsigned int acc = 0;
    for (int k = 0; k < n; k++) acc += (unsigned int)imgs[(size_t)k * count + i] / (unsigned int)n;
    out[i] = (uint8_t)acc;  // imgdata[] is unsigned char: wraps like the reference would (it cannot for n >= 1: n * floor(255 / n) <= 255)
}
__global__ void average_f64_kernel(const double *__restrict__ imgs, int n, int64_t count, double *__restrict__ mean, uint8_t *__restrict__ rgb8) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    double acc = 0.0;
    for (int k = 0; k < n; k++) acc += imgs[(size_t)k * count + i];
    acc = acc / (double)n;
    mean[i] = acc;
    if (rgb8) rgb8[i] = (uint8_t)(char)gamma_corr(acc);
}

// =================================================================================================================
// Parity-hook kernels
// =================================================================================================================
template <bool COUNT>
__global__ void __launch_bounds__(CGRT_TRACE_BLOCK) intersect_batch_kernel(const __grid_constant__ SceneDev S, int64_t n, const double *__restrict__ org,
                                                                           const double *__restrict__ dir, double *t, double *nrm, double *nrm_raw,
                                                                           int *obj, int *into, int *prim, TravCounters *tc_out) {
    __shared__ TraceShared<CGRT_TRACE_BLOCK> sm;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = i < n;
    d3 o = mk(0, 0, 0), d = mk(0, 0, 1);
    if (active) { o = mk(org[3 * i], org[3 * i + 1], org[3 * i + 2]); d = mk(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]); }
    Hit h;
    TravCounters tc;
    tc.node_visits = 0; tc.tri_tests = 0;
    bool found = closest_hit_block<CGRT_TRACE_BLOCK, COUNT>(S, active, o, d, h, sm, &tc);
    if (COUNT) {
        atomicAdd(&tc_out->node_visits, tc.node_visits);
        atomicAdd(&tc_out->tri_tests, tc.tri_tests);
    }
    if (!active) return;
    d3 nf = h.n;
    int in = 1;
    if (found && dot(nf, d) > 0) { nf = -nf; in = 0; }
    if (obj) obj[i] = found ? h.obj : -1;
    if (t) t[i] = found ? h.t : 0.0;
    if (nrm) { nrm[3 * i] = found ? nf.x : 0; nrm[3 * i + 1] = found ? nf.y : 0; nrm[3 * i + 2] = found ? nf.z : 0; }
    if (nrm_raw) { nrm_raw[3 * i] = found ? h.n.x : 0; nrm_raw[3 * i + 1] = found ? h.n.y : 0; nrm_raw[3 * i + 2] = found ? h.n.z : 0; }
    if (into) into[i] = found ? in : 0;
    if (prim) prim[i] = found ? h.prim : -1;
}

__global__ void hash_keys_kernel(int64_t n, const double *__restrict__ pos, uint32_t hashsize, double celllength, uint32_t *key, int *ixyz) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int ix, iy, iz;
    cell_coord(mk(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]), celllength, 1.0 / celllength, ix, iy, iz);
    if (ixyz) { ixyz[3 * i] = ix; ixyz[3 * i + 1] = iy; ixyz[3 * i + 2] = iz; }
    if (key) key[i] = cell_hash(ix, iy, iz, hashsize);
}

__global__ void surface_color_kernel(const __grid_constant__ SceneDev S, int obj, int64_t n, const double *__restrict__ pos, double *col) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    d3 c = surface_color(S, obj, mk(pos[3 * i], pos[3 * i + 1], pos[3 * i + 2]));
    col[3 * i] = c.x; col[3 * i + 1] = c.y; col[3 * i + 2] = c.z;
}

__global__ void sample_kernel(uint64_t seed, uint32_t pass, uint64_t path, uint32_t dim, int what, double a0, double a1, double a2, double *out) {
    Philox g;
    g.init(seed, pass, path, dim);
    d3 r;
    if (what == 0) r = sample_sphere(g);
    else if (what == 1) r = sample_halfsphere(g, mk(a0, a1, a2));
    else if (what == 2) r = sample_circle(g, a0);
    else { r.x = g.u01(); r.y = g.u01(); r.z = g.u01(); }
    out[0] = r.x; out[1] = r.y; out[2] = r.z;
}

}  // namespace cgrt
