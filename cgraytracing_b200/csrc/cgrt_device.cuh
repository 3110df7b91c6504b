// cgrt_device.cuh — device-side building blocks of the photon-mapping hot path (sm_100a).
//
// Arithmetic policy: everything that decides a hit, a position, a cell key or an accept/reject is IEEE fp64 in the
// reference's own operation order (compiled with -fmad=false, so no contraction), which makes the GPU path replay the
// CPU oracle bit for bit. B200 keeps full-rate FP64 vector units (unlike B300), which is what makes this affordable.
// Only the BVH box test is free-form (explicit fma, padded float bounds): it is conservative, never decisive.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cgrt {

// ---------------------------------------------------------------------------------------------------------------
// vec3.h:11-92 as a POD
// ---------------------------------------------------------------------------------------------------------------
struct d3 {
    double x, y, z;
};
__host__ __device__ __forceinline__ d3 mk(double x, double y, double z) { d3 r; r.x = x; r.y = y; r.z = z; return r; }
__host__ __device__ __forceinline__ d3 operator+(d3 a, d3 b) { return mk(a.x + b.x, a.y + b.y, a.z + b.z); }
__host__ __device__ __forceinline__ d3 operator-(d3 a, d3 b) { return mk(a.x - b.x, a.y - b.y, a.z - b.z); }
__host__ __device__ __forceinline__ d3 operator-(d3 a) { return mk(-a.x, -a.y, -a.z); }
__host__ __device__ __forceinline__ d3 operator*(d3 a, double f) { return mk(a.x * f, a.y * f, a.z * f); }   // vec3.h:50
__host__ __device__ __forceinline__ d3 operator*(d3 a, d3 b) { return mk(a.x * b.x, a.y * b.y, a.z * b.z); } // vec3.h:54
__host__ __device__ __forceinline__ double dot(d3 a, d3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }     // vec3.h:61
__host__ __device__ __forceinline__ d3 cross(d3 a, d3 b) {                                                   // vec3.h:81
    return mk(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__host__ __device__ __forceinline__ d3 normalize(d3 a) {  // vec3.h:35-43: multiply by (1/len), three times
    double len = sqrt(a.x * a.x + a.y * a.y + a.z * a.z);
    if (len > 0) {
        a.x *= 1 / len;
        a.y *= 1 / len;
        a.z *= 1 / len;
    }
    return a;
}
// vec3.h:95-97, strictly left to right
__host__ __device__ __forceinline__ double det3(d3 a, d3 b, d3 c) {
    return (a.x * b.y * c.z + b.x * c.y * a.z + c.x * a.y * b.z - a.x * c.y * b.z - b.x * a.y * c.z - c.x * b.y * a.z);
}
// util.h:16-26
__host__ __device__ __forceinline__ double max3(double a, double b, double c) {
    if (a > b && a > c) return a;
    else if (b > c) return b;
    else return c;
}

#define CGRT_EPS 1e-4               /* main.cpp:24 */
#define CGRT_INF 1e10               /* main.cpp:25, objects.h:15 */
#define CGRT_PI 3.14159265358979    /* main.cpp:26 */

// ---------------------------------------------------------------------------------------------------------------
// Philox4x32-10 counter RNG (replaces rand(), sampling.h). key = {seed_lo, seed_hi + pass},
// counter = {path_lo, path_hi, dim, block}; u = (double)(word >> 1) * 2^-31 (a 31-bit lattice like rand()/RAND_MAX).
// ---------------------------------------------------------------------------------------------------------------
// PASS_SPPM_EYE: the camera stream of stochastic progressive photon mapping, one per (eye path, round): dim = round.
enum { PASS_EYE = 0, PASS_PHOTON = 1, PASS_BEZIER = 2, PASS_SPPM_EYE = 3 };

struct Philox {
    uint32_t k0, k1, c0, c1, c2, c3;
    uint32_t buf[4];
    int idx;
    __host__ __device__ __forceinline__ void init(uint64_t seed, uint32_t pass, uint64_t path, uint32_t dim) {
        k0 = (uint32_t)seed;
        k1 = (uint32_t)(seed >> 32) + pass;
        c0 = (uint32_t)path;
        c1 = (uint32_t)(path >> 32);
        c2 = dim;
        c3 = 0;
        idx = 4;
    }
    __host__ __device__ __forceinline__ void block() {
        uint32_t a0 = c0, a1 = c1, a2 = c2, a3 = c3, x0 = k0, x1 = k1;
#pragma unroll
        for (int r = 0; r < 10; r++) {
#ifdef __CUDA_ARCH__
            uint32_t h0 = __umulhi(0xD2511F53u, a0), l0 = 0xD2511F53u * a0;
            uint32_t h1 = __umulhi(0xCD9E8D57u, a2), l1 = 0xCD9E8D57u * a2;
#else
            uint64_t p0 = (uint64_t)0xD2511F53u * a0, p1 = (uint64_t)0xCD9E8D57u * a2;
            uint32_t h0 = (uint32_t)(p0 >> 32), l0 = (uint32_t)p0, h1 = (uint32_t)(p1 >> 32), l1 = (uint32_t)p1;
#endif
            uint32_t n0 = h1 ^ a1 ^ x0, n2 = h0 ^ a3 ^ x1;
            a0 = n0; a1 = l1; a2 = n2; a3 = l0;
            x0 += 0x9E3779B9u;
            x1 += 0xBB67AE85u;
        }
        buf[0] = a0; buf[1] = a1; buf[2] = a2; buf[3] = a3;
        c3++;
        idx = 0;
    }
    __host__ __device__ __forceinline__ double u01() {
        if (idx == 4) block();
        uint32_t w = buf[0];
        // select without dynamic local-memory indexing
        w = idx == 1 ? buf[1] : w;
        w = idx == 2 ? buf[2] : w;
        w = idx == 3 ? buf[3] : w;
        idx++;
        return (double)(w >> 1) * (1.0 / 2147483648.0);
    }
};

#define CGRT_MAX_REJECT 64
// sin and cos of 2*pi*v, v in [0,1), from +,-,* only (the library is built with -fmad=false): bit-identical on any
// IEEE machine. Exact quadrant reduction + minimax kernels on [-pi/4, pi/4].
__host__ __device__ __forceinline__ void sincos2pi(double v, double &s_out, double &c_out) {
    double t = 4.0 * v;
    int k = (int)(t + 0.5);
    double r = t - (double)k;
    double x = r * 1.5707963267948966;
    double z = x * x;
    double ps = -1.66666666666666324348e-01 + z * (8.33333333332248946124e-03 + z * (-1.98412698298579493134e-04 + z * (2.75573137070700676789e-06 +
                z * (-2.50507602534068634195e-08 + z * 1.58969099521155010221e-10))));
    double sn = x + x * z * ps;
    double pc = 4.16666666666666019037e-02 + z * (-1.38888888888741095749e-03 + z * (2.48015872894767294178e-05 + z * (-2.75573143513906633035e-07 +
                z * (2.08757232129817482790e-09 + z * -1.13596475577881948265e-11))));
    double cs = 1.0 - 0.5 * z + z * z * pc;
    int q = k & 3;
    s_out = q == 0 ? sn : (q == 1 ? cs : (q == 2 ? -sn : -cs));
    c_out = q == 0 ? cs : (q == 1 ? -sn : (q == 2 ? -cs : sn));
}
// sampling.h:11-20 as a distribution: uniform on the unit sphere by Archimedes' map (z = 1 - 2 u1, phi = 2 pi u2). The
// reference rejects from the cube; two draws and no loop keep the warp converged (SURVEY Q4).
__host__ __device__ __forceinline__ d3 sample_sphere(Philox &g) {
    double z = 1.0 - 2.0 * g.u01();
    double sn, cs;
    sincos2pi(g.u01(), sn, cs);
    double r = sqrt(1.0 - z * z);
    return mk(r * cs, r * sn, z);
}
// sampling.h:22-29 as a distribution: a sphere sample mirrored into the hemisphere about dir.
__host__ __device__ __forceinline__ d3 sample_halfsphere(Philox &g, d3 dir) {
    d3 s = sample_sphere(g);
    if (dot(s, dir) < 0) s = -s;
    return s;
}
// sampling.h:35-43
__host__ __device__ __forceinline__ d3 sample_circle(Philox &g, double radius) {
    double x = 0, y = 0;
    for (int it = 0; it < CGRT_MAX_REJECT; it++) {
        x = g.u01() * 2.0 - 1;
        y = g.u01() * 2.0 - 1;
        if (x * x + y * y < 1) break;
    }
    return mk(x, y, 0) * radius;
}

// ---------------------------------------------------------------------------------------------------------------
// Device scene (passed to kernels by value as a __grid_constant__ parameter: uniform constant-bank reads)
// ---------------------------------------------------------------------------------------------------------------
enum { OBJ_SPHERE = 0, OBJ_PLANE = 1, OBJ_MESH = 2, OBJ_BEZIER = 3 };
enum { MAT_DIFFUSE = 0, MAT_MIRROR = 1, MAT_GLASS = 2 };  // main.cpp:82,129,135 thresholds (SURVEY Q6)

#define CGRT_MAX_OBJECTS 12
#define CGRT_MAX_BVH 4
#define CGRT_MAX_TEX 4
#define CGRT_MAX_BEZIER 2
#define CGRT_MAX_CP 7

// One 4-wide node, 128 bytes = one cache line: the (float, padded) boxes of up to four children, component by component, and their links.
// child >= 0: 4-wide node index; child < 0: leaf, ~child = index into the Morton-sorted triangle array; CGRT_NO_CHILD: empty slot.
// Built by collapsing the binary LBVH top down (lbvh_collapse_kernel): a traversal reads half as many dependent nodes per ray.
#define CGRT_NO_CHILD ((int)0x80000000)
struct __align__(16) BvhNode4 {
    float lox[4], loy[4], loz[4], hix[4], hiy[4], hiz[4];
    int child[4];
    int pad[4];
};
// One triangle, 96 bytes = three sectors: pa and the edges / normal exactly as Triangle::intersect forms them
// (objects.h:98-99,107): e1 = pa - pb, e2 = pa - pc, n = normalize(e1 x e2).
struct __align__(16) TriRec {
    double pa[3], e1[3], e2[3], n[3];
};

struct ObjDev {
    int kind, material, tex, bvh, objtype, aux;
    double a[3];      // sphere centre | plane position
    double b[3];      // plane normal
    double r, r2;     // sphere radius, radius*radius (objects.h:35)
    double col[3];
    double refl, transp;
};
struct BvhDev {
    const BvhNode4 *nodes4;
    const TriRec *tris;
    const int *tri_id;      // sorted position -> original triangle index
    int ntris;
    int root_is_leaf;
    double orient_sign;     // winding normal * orient_sign points out of the solid (SURVEY Q8)
    float root_lo[3], root_hi[3];  // padded box of the whole tree (the compaction prefilter of closest_hit_block)
    int f32_ok;             // 1: every coordinate is within CGRT_F32_BOUND, the float slab test is conservative
    int pad;
};
struct TexDev {
    const uchar4 *texels;   // row-major [H][W], texel = byte/256 (main.cpp:307-311)
    int W, H, isbump, pad;
    double n[3], p[3], lenx, leny;
};
struct BezDev {
    int ncp, pad;
    double cp[CGRT_MAX_CP][3];
    double pos[3];
    double box[6];          // xmax,xmin,ymax,ymin,zmax,zmin (bezier.h:64-69)
    double umin_r2;         // cap radius^2 = cp[last].z^2 (bezier.h:277)
    double C[CGRT_MAX_CP], Cm[CGRT_MAX_CP];  // binomial rows n and n-1 (bez_binomials; filled by cgrt_commit_scene)
};
struct SceneDev {
    int nobj, nbvh, ntex, nbez;
    // object indices by class, each list ascending (filled by cgrt_commit_scene): the closest-hit loop is the lexicographic minimum
    // of (len, index), so the classes can be walked separately — planes three at a time for instruction-level parallelism
    int nplane, nsphere, ndeferred;
    unsigned char plane_ix[CGRT_MAX_OBJECTS], sphere_ix[CGRT_MAX_OBJECTS], deferred_ix[CGRT_MAX_OBJECTS];
    ObjDev obj[CGRT_MAX_OBJECTS];
    BvhDev bvh[CGRT_MAX_BVH];
    TexDev tex[CGRT_MAX_TEX];
    BezDev bez[CGRT_MAX_BEZIER];
};

struct Hit {
    double t;
    d3 n;        // raw normal as Object::intersect returns it
    int obj;
    int prim;    // original triangle index or -1
};

struct TravCounters {
    unsigned long long node_visits, tri_tests;
};

// ---------------------------------------------------------------------------------------------------------------
// Triangle::intersect, objects.h:96-111. The reference evaluates four quotients det_k/det1 and compares them with
// 0 and 1; the same decisions are taken here from signs and one comparison (exactly equivalent for finite inputs
// whose quotients do not underflow), and the only division performed is the one that produces t.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool tri_intersect(const TriRec *T, d3 o, d3 d, double &t) {
    const double2 *tq = reinterpret_cast<const double2 *>(T);  // pa, e1, e2 = 9 doubles: four 16-byte loads + one 8-byte
    double2 a0 = __ldg(tq), a1 = __ldg(tq + 1), a2 = __ldg(tq + 2), a3 = __ldg(tq + 3);
    double a4 = __ldg(reinterpret_cast<const double *>(tq + 4));
    d3 pa = mk(a0.x, a0.y, a1.x);
    d3 e1 = mk(a1.y, a2.x, a2.y);
    d3 e2 = mk(a3.x, a3.y, a4);
    d3 s = pa - o;
    double det1 = det3(d, e1, e2);
    if (det1 == 0.0 || det1 != det1) return false;  // x/0 -> inf/nan never satisfies all four tests
    double det3v = det3(d, s, e2);
    double det4v = det3(d, e1, s);
    bool pos = det1 > 0.0;
    // det3/det1 >= 0  <=>  det3 == 0 or sign(det3) == sign(det1)
    if (!(det3v == 0.0 || ((det3v > 0.0) == pos))) return false;
    if (!(det4v == 0.0 || ((det4v > 0.0) == pos))) return false;
    // (det3+det4)/det1 <= 1  <=>  det3+det4 <= det1 (det1 > 0)  |  >= det1 (det1 < 0): RN division is monotone and
    // q(x,x) = 1 exactly, q(x',x) > 1 + 2^-53 for the next double x' > x.
    double sum = det3v + det4v;
    if (pos ? !(sum <= det1) : !(sum >= det1)) return false;
    double det2 = det3(s, e1, e2);
    double q = det2 / det1;
    if (!(q > 0.0)) return false;
    t = q;
    return true;
}

// ---------------------------------------------------------------------------------------------------------------
// BVH traversal: closest triangle with t < tmax (strict), t > 0. Stack in local memory (depth <= 64).
//
// The box test never decides a hit, it only has to be conservative. Node boxes are float and padded by CGRT_BOX_PAD at
// build time; a ray whose origin lies within CGRT_F32_BOUND of the world origin is tested in fp32 (origin and 1/dir
// rounded to float): with |coordinates| <= 64 the rounding of the origin (<= 3.8e-6), of the subtraction (<= 7.6e-6)
// and the relative error of 1/dir and of the product (<= 3e-7 * 128) move a slab plane by less than 5e-5 < CGRT_BOX_PAD
// in position space, so the float interval of the padded box always contains the exact interval of the true box.
// Rays that start farther out (photons that left through the open front of the room and came back) take the fp64 slab.
// The triangle test itself is always the reference's fp64 arithmetic (tri_intersect).
// ---------------------------------------------------------------------------------------------------------------
#define CGRT_F32_BOUND 64.0
#define CGRT_BOX_PAD 8e-5

struct SlabRay {
    float ox, oy, oz, ix, iy, iz;  // fp32 path
    d3 o, id;                      // fp64 path
    bool exact;
};
__device__ __forceinline__ SlabRay make_slab_ray(d3 o, d3 d, bool f32_ok) {
    SlabRay r;
    r.exact = !(f32_ok && fabs(o.x) <= CGRT_F32_BOUND && fabs(o.y) <= CGRT_F32_BOUND && fabs(o.z) <= CGRT_F32_BOUND);
    r.o = o;
    r.id = mk(0, 0, 0);
    if (r.exact) r.id = mk(1.0 / d.x, 1.0 / d.y, 1.0 / d.z);  // three fp64 divisions: only for the rare far-origin ray
    r.ox = (float)o.x; r.oy = (float)o.y; r.oz = (float)o.z;
    r.ix = 1.0f / (float)d.x; r.iy = 1.0f / (float)d.y; r.iz = 1.0f / (float)d.z;
    return r;
}
// NaNs (0 * inf) are dropped by fmin/fmax.
__device__ __forceinline__ bool slab64(float lx, float ly, float lz, float hx, float hy, float hz, const SlabRay &r, double tmax, float &tnear) {
    double tx0 = ((double)lx - r.o.x) * r.id.x, tx1 = ((double)hx - r.o.x) * r.id.x;
    double ty0 = ((double)ly - r.o.y) * r.id.y, ty1 = ((double)hy - r.o.y) * r.id.y;
    double tz0 = ((double)lz - r.o.z) * r.id.z, tz1 = ((double)hz - r.o.z) * r.id.z;
    double tn = fmax(fmax(fmin(tx0, tx1), fmin(ty0, ty1)), fmax(fmin(tz0, tz1), 0.0));
    double tf = fmin(fmin(fmax(tx0, tx1), fmax(ty0, ty1)), fmin(fmax(tz0, tz1), tmax));
    tnear = (float)tn;
    return tn <= tf;
}
__device__ __forceinline__ bool slab32(float lx, float ly, float lz, float hx, float hy, float hz, const SlabRay &r, float tmax_up, float &tnear) {
    float tx0 = (lx - r.ox) * r.ix, tx1 = (hx - r.ox) * r.ix;
    float ty0 = (ly - r.oy) * r.iy, ty1 = (hy - r.oy) * r.iy;
    float tz0 = (lz - r.oz) * r.iz, tz1 = (hz - r.oz) * r.iz;
    float tn = fmaxf(fmaxf(fminf(tx0, tx1), fminf(ty0, ty1)), fmaxf(fminf(tz0, tz1), 0.0f));
    float tf = fminf(fminf(fmaxf(tx0, tx1), fmaxf(ty0, ty1)), fminf(fmaxf(tz0, tz1), tmax_up));
    tnear = tn;
    return tn <= tf;
}
__device__ __forceinline__ bool slab_any(float lx, float ly, float lz, float hx, float hy, float hz, const SlabRay &r, double tmax, float tmax_up,
                                         float &tnear) {
    return r.exact ? slab64(lx, ly, lz, hx, hy, hz, r, tmax, tnear) : slab32(lx, ly, lz, hx, hy, hz, r, tmax_up, tnear);
}
// Does the ray reach the (padded) root box of a tree before tmax? Asked for every segment of every photon, most of which never come near
// the mesh — and, in the reference's open room, by photons that bounce on between the infinite planes far outside it. The float slab
// test is made conservative for ANY origin by widening the box with the rounding of THIS ray instead of switching to fp64 for far
// origins: the origin rounds by <= 2^-24 |o|, the subtraction by <= 2^-24 (|o| + |l|), 1/d and the product move a plane by
// <= 1.8e-7 (|o| + |l|) in position space — together <= 3e-7 (|o| + 64) with |l| <= CGRT_F32_BOUND; 1e-6 (|o| + 64) is used.
// (Before: lanes with |o| > 64 took an fp64 slab test with three divisions, 2 lanes at a time: 6 % of the emission kernel's instructions.)
__device__ __forceinline__ bool root_box_hit(const BvhDev &B, d3 o, d3 d, double tmax) {
    if (!B.f32_ok) {  // a tree that itself reaches beyond CGRT_F32_BOUND: exact test (uniform branch)
        SlabRay r = make_slab_ray(o, d, false);
        float tn;
        return slab_any(B.root_lo[0], B.root_lo[1], B.root_lo[2], B.root_hi[0], B.root_hi[1], B.root_hi[2], r, tmax, __double2float_ru(tmax), tn);
    }
    const float ox = (float)o.x, oy = (float)o.y, oz = (float)o.z;
    const float ix = 1.0f / (float)d.x, iy = 1.0f / (float)d.y, iz = 1.0f / (float)d.z;
    const float pad = 1e-6f * (fmaxf(fmaxf(fabsf(ox), fabsf(oy)), fabsf(oz)) + (float)CGRT_F32_BOUND);
    const float tx0 = (B.root_lo[0] - pad - ox) * ix, tx1 = (B.root_hi[0] + pad - ox) * ix;
    const float ty0 = (B.root_lo[1] - pad - oy) * iy, ty1 = (B.root_hi[1] + pad - oy) * iy;
    const float tz0 = (B.root_lo[2] - pad - oz) * iz, tz1 = (B.root_hi[2] + pad - oz) * iz;
    const float tn = fmaxf(fmaxf(fminf(tx0, tx1), fminf(ty0, ty1)), fmaxf(fminf(tz0, tz1), 0.0f));
    const float tf = fminf(fminf(fmaxf(tx0, tx1), fmaxf(ty0, ty1)), fminf(fmaxf(tz0, tz1), __double2float_ru(tmax)));
    return tn <= tf;
}

// ---------------------------------------------------------------------------------------------------------------
// Closest-hit search over the 4-wide nodes. One node visit = one 128-byte line = four box tests;
// the children that are hit are entered nearest first (sorting network over four 32-bit keys: entry distance with the slot number in the
// two lowest mantissa bits) and the others pushed farthest first (predicated stores: three unconditional stack stores per visit were
// measured 11 % slower, the traversal is sensitive to every extra L1 transaction). F32ONLY: the instantiation for trees that lie within
// CGRT_F32_BOUND (every mesh of the BASELINE scenes), without any fp64 box arithmetic: a ray that starts farther out than the bound is
// re-based for the box tests only — its entry distance t0 into the padded root box is taken in fp64 once, the float slabs then run
// from o + d t0 (on the root box, inside the bound) against best - t0; the triangle test keeps the original origin and the reference's
// fp64 arithmetic. Otherwise SlabRay picks per ray.
// (Measured and rejected on the 2-wide tree that preceded this one: a "while-while" ordering that parks lanes on their leaf until the
// warp reconverges, 8.8 vs 7.0 ms; postponing the fp64 triangle tests to after the loop behind a conservative float classification of
// every leaf, 5.21 vs 5.14 ms; L1 prefetch of the pushed children, 5.03 vs 4.89 ms. The 2-wide tree itself: 5.09 vs 4.61 ms.)
// ---------------------------------------------------------------------------------------------------------------
#ifndef CGRT_BVH_STACK
#define CGRT_BVH_STACK 160   /* three pushes per wide level; cgrt_commit_scene refuses a deeper tree */
#endif
__device__ __forceinline__ float f4c(const float4 &v, int j) { return j == 0 ? v.x : (j == 1 ? v.y : (j == 2 ? v.z : v.w)); }
__device__ __forceinline__ void cswap(unsigned int &a, unsigned int &b) {
    const unsigned int lo = min(a, b), hi = max(a, b);
    a = lo; b = hi;
}

template <bool COUNT, bool F32ONLY>
__device__ __forceinline__ bool bvh4_closest(const BvhDev &B, d3 o, d3 d, double tmax, double &t_out, int &leaf_out, TravCounters *tc) {
    double t0 = 0.0;
    SlabRay R;
    float ox, oy, oz, ix, iy, iz;
    if (F32ONLY) {
        d3 ob = o;
        if (!(fabs(o.x) <= CGRT_F32_BOUND && fabs(o.y) <= CGRT_F32_BOUND && fabs(o.z) <= CGRT_F32_BOUND)) {
            const double jx = 1.0 / d.x, jy = 1.0 / d.y, jz = 1.0 / d.z;
            const double tx0 = ((double)B.root_lo[0] - o.x) * jx, tx1 = ((double)B.root_hi[0] - o.x) * jx;
            const double ty0 = ((double)B.root_lo[1] - o.y) * jy, ty1 = ((double)B.root_hi[1] - o.y) * jy;
            const double tz0 = ((double)B.root_lo[2] - o.z) * jz, tz1 = ((double)B.root_hi[2] - o.z) * jz;
            const double tn = fmax(fmax(fmin(tx0, tx1), fmin(ty0, ty1)), fmax(fmin(tz0, tz1), 0.0));
            const double tf = fmin(fmin(fmax(tx0, tx1), fmax(ty0, ty1)), fmin(fmax(tz0, tz1), tmax));
            if (!(tn <= tf)) { t_out = tmax; leaf_out = -1; return false; }  // misses the root box
            t0 = tn * (1.0 - 1e-12);  // never beyond the true entry
            ob = o + d * t0;
        }
        ox = (float)ob.x; oy = (float)ob.y; oz = (float)ob.z;
        ix = 1.0f / (float)d.x; iy = 1.0f / (float)d.y; iz = 1.0f / (float)d.z;
        R.exact = false;
    } else {
        R = make_slab_ray(o, d, B.f32_ok != 0);
        ox = R.ox; oy = R.oy; oz = R.oz; ix = R.ix; iy = R.iy; iz = R.iz;
    }
    // Float slabs in the form t = fma(plane, 1/d, -o/d) with the near and far plane of each axis picked by the sign of 1/d — per ray that
    // is a choice of ADDRESS inside the node (lox.. or hix..), so a box costs six fused multiply-adds and four min/max instead of twelve
    // operations and ten min/max. Rounding: the constant c = fl(-o * (1/d)) is off by u |o / d|, i.e. u |o| <= 3.8e-6 in position space, on
    // top of the origin's own rounding (3.8e-6), the relative error 2u of 1/d over a distance <= 128 (1.5e-5) and the final rounding
    // (7.6e-6): 3.1e-5 < CGRT_BOX_PAD, like the subtract-then-multiply form. A component of d so small that plane * (1/d) overflows
    // gives inf - inf = NaN, which min/max drop: that axis then does not constrain the box (conservative).
    const float cx = -(ox * ix), cy = -(oy * iy), cz = -(oz * iz);
    const int sxo = ix < 0.f ? 3 : 0, syo = iy < 0.f ? 3 : 0, szo = iz < 0.f ? 3 : 0;  // float4 index of the near plane: lo (0) or hi (3)
    double best = tmax;
    float best_up = __double2float_ru(tmax - t0);
    int best_leaf = -1;
    int stack[CGRT_BVH_STACK];
    int sp = 0;
    int node = B.root_is_leaf ? ~0 : 0;
    for (;;) {
        if (node >= 0) {
            const float4 *q = reinterpret_cast<const float4 *>(B.nodes4 + node);
            const int4 ch = __ldg(reinterpret_cast<const int4 *>(q + 6));
            if (COUNT) tc->node_visits += 4;
            unsigned int key[4];
            if (!F32ONLY && R.exact) {
                const float4 lx = __ldg(q), ly = __ldg(q + 1), lz = __ldg(q + 2), hx = __ldg(q + 3), hy = __ldg(q + 4), hz = __ldg(q + 5);
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    float tn;
                    const bool h = slab64(f4c(lx, j), f4c(ly, j), f4c(lz, j), f4c(hx, j), f4c(hy, j), f4c(hz, j), R, best, tn);
                    key[j] = h ? ((__float_as_uint(tn) & ~3u) | (unsigned int)j) : 0xffffffffu;
                }
            } else {
                const float4 nx = __ldg(q + sxo), fx = __ldg(q + 3 - sxo), ny = __ldg(q + 1 + syo), fy = __ldg(q + 4 - syo);
                const float4 nz = __ldg(q + 2 + szo), fz = __ldg(q + 5 - szo);
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const float tn = fmaxf(fmaxf(fmaf(f4c(nx, j), ix, cx), fmaf(f4c(ny, j), iy, cy)), fmaxf(fmaf(f4c(nz, j), iz, cz), 0.0f));
                    const float tf = fminf(fminf(fmaf(f4c(fx, j), ix, cx), fmaf(f4c(fy, j), iy, cy)), fminf(fmaf(f4c(fz, j), iz, cz), best_up));
                    key[j] = (tn <= tf) ? ((__float_as_uint(tn) & ~3u) | (unsigned int)j) : 0xffffffffu;  // tn >= 0: its bits order like the value
                }
            }
            // empty slots hold an inverted box far outside the scene in the binary node's place: mask them by their link
            if (ch.z == CGRT_NO_CHILD) key[2] = 0xffffffffu;
            if (ch.w == CGRT_NO_CHILD) key[3] = 0xffffffffu;
            cswap(key[0], key[1]); cswap(key[2], key[3]); cswap(key[0], key[2]); cswap(key[1], key[3]); cswap(key[1], key[2]);
            if (key[0] == 0xffffffffu) {
                if (sp == 0) break;
                node = stack[--sp];
            } else {
                // links of the sorted slots, without branches; the stack takes the far ones, farthest first
                int c[4];
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    // ch[slot] by funnel shifts (a clamped shift by 32 picks the high word): no branches, no local-memory indexing
                    const unsigned int s1 = (key[k] & 1u) << 5, s2 = (key[k] & 2u) << 4;
                    const unsigned int lo = __funnelshift_rc((unsigned int)ch.x, (unsigned int)ch.y, s1);
                    const unsigned int hi = __funnelshift_rc((unsigned int)ch.z, (unsigned int)ch.w, s1);
                    c[k] = (int)__funnelshift_rc(lo, hi, s2);
                }
                if (key[3] != 0xffffffffu) stack[sp++] = c[3];
                if (key[2] != 0xffffffffu) stack[sp++] = c[2];
                if (key[1] != 0xffffffffu) stack[sp++] = c[1];
                node = c[0];
            }
        } else {
            const int leaf = ~node;
            if (COUNT) tc->tri_tests++;
            double t;
            if (tri_intersect(B.tris + leaf, o, d, t) && t < best) {
                best = t;
                best_up = __double2float_ru(t - t0);
                best_leaf = leaf;
            }
            if (sp == 0) break;
            node = stack[--sp];
        }
    }
    t_out = best;
    leaf_out = best_leaf;
    return best_leaf >= 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Bezier surface of revolution (bezier.h). The reference solves F(t,u,theta)=0 by Newton from 10 random starts;
// here the same Newton iteration (same F, same Jacobian, same acceptance test) is started from a deterministic
// seed grid, and the nearest accepted root is kept (SURVEY Q14: parity for this primitive is statistical).
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ bool box_any_face_hit(const double *b, d3 o, d3 d) {  // bezier.h:72-126, objects.h:166-200
    const double e = 1e-4;
    double xmax = b[0], xmin = b[1], ymax = b[2], ymin = b[3], zmax = b[4], zmin = b[5];
    double t; d3 p;
    t = (xmax - o.x) / d.x; p = o + d * t;
    if (t > 0 && p.y >= ymin - e && p.y <= ymax + e && p.z >= zmin - e && p.z <= zmax + e) return true;
    t = (xmin - o.x) / d.x; p = o + d * t;
    if (t > 0 && p.y >= ymin - e && p.y <= ymax + e && p.z >= zmin - e && p.z <= zmax + e) return true;
    t = (ymax - o.y) / d.y; p = o + d * t;
    if (t > 0 && p.x >= xmin - e && p.x <= xmax + e && p.z >= zmin - e && p.z <= zmax + e) return true;
    t = (ymin - o.y) / d.y; p = o + d * t;
    if (t > 0 && p.x >= xmin - e && p.x <= xmax + e && p.z >= zmin - e && p.z <= zmax + e) return true;
    t = (zmax - o.z) / d.z; p = o + d * t;
    if (t > 0 && p.x >= xmin - e && p.x <= xmax + e && p.y >= ymin - e && p.y <= ymax + e) return true;
    t = (zmin - o.z) / d.z; p = o + d * t;
    if (t > 0 && p.x >= xmin - e && p.x <= xmax + e && p.y >= ymin - e && p.y <= ymax + e) return true;
    return false;
}

// Bernstein value of the profile curve (bezier.h:30-35,127-134) and the reference's "gradient" (bezier.h:37-40,135-142):
//   dB(n,i,t) = i * B(n-1,i-1,t) - (n-i) * B(n-1,i,t)
// which is NOT the derivative n * (B(n-1,i-1) - B(n-1,i)) of the Bernstein basis (the correct form is commented out at
// bezier.h:39). The reference's Newton Jacobian and its surface normals are built from this quantity, so the picture
// depends on it and it is reproduced as is (SURVEY Appendix E: gradP(0) = (0,32,-8), not 3*(P1-P0) = (0,36,0)).
// The two binomial rows, by the recurrence every evaluation used to repeat (2n fp64 divisions per Newton iteration); computed once per
// surface on the host with the same IEEE operations.
__host__ __device__ inline void bez_binomials(int ncp, double *C, double *Cm) {
    int n = ncp - 1;
    for (int i = 0; i < CGRT_MAX_CP; i++) { C[i] = 0.0; Cm[i] = 0.0; }
    C[0] = 1.0; Cm[0] = 1.0;
    for (int i = 1; i <= n; i++) C[i] = C[i - 1] * (double)(n - i + 1) / (double)i;
    for (int i = 1; i <= n - 1; i++) Cm[i] = Cm[i - 1] * (double)(n - i) / (double)i;
}
__device__ __forceinline__ void bez_eval(const BezDev &Z, double u, d3 &P, d3 &dP) {
    int n = Z.ncp - 1;
    const double *C = Z.C, *Cm = Z.Cm;
    double pu[CGRT_MAX_CP], pv[CGRT_MAX_CP];
    pu[0] = 1.0; pv[0] = 1.0;
    for (int i = 1; i <= n; i++) { pu[i] = pu[i - 1] * u; pv[i] = pv[i - 1] * (1.0 - u); }
    P = mk(0, 0, 0); dP = mk(0, 0, 0);
    for (int i = 0; i <= n; i++) {
        double b = C[i] * pv[n - i] * pu[i];
        double db = 0.0;
        if (i > 0) db += Cm[i - 1] * pv[n - i] * pu[i - 1] * (double)i;          // B(n-1, i-1, u) * i
        if (i < n) db -= Cm[i] * pv[n - 1 - i] * pu[i] * (double)(n - i);        // B(n-1, i, u) * (n-i)
        d3 c = mk(Z.cp[i][0], Z.cp[i][1], Z.cp[i][2]);
        P = P + c * b;
        dP = dP + c * db;
    }
}

__device__ __forceinline__ d3 bez_F(const BezDev &Z, d3 par, d3 o, d3 d, d3 &P, d3 &dP, double &s, double &c) {  // bezier.h:144-149
    bez_eval(Z, par.y, P, dP);
    sincos(par.z, &s, &c);  // handed back: the Jacobian of the next Newton step needs the same pair
    d3 surf = mk(P.z * s, P.y, P.z * c);
    return o + d * par.x - mk(Z.pos[0], Z.pos[1], Z.pos[2]) - surf;
}

// One Newton solve (bezier.h:163-214) from seed number `seed` of the deterministic 4 x 4 grid (u0 = 1/8, 3/8, 5/8, 7/8 times four
// t0 across the ray's passage by the axis; theta0 from the seed point, bezier.h:243-247). Returns whether the iterate is accepted
// (bezier.h:257) and then its t and the un-oriented normal of bezier.h:215-224.
#define CGRT_BEZ_SEEDS 16
#ifndef CGRT_BEZ_MAXIT
/* bezier.h:170 caps a solve at 100 steps. A start that has not converged after 40 almost never does: with 16 deterministic starts per ray a
 * cap of 40 changes 0.011 % of the pixels of the c1 image by more than 1 % (mean relative difference 2e-5, same hitpoints) and takes the
 * half-warp solver from 10.1 to 5.8 ms per round — every ray that misses the vase pays the cap in full. */
#define CGRT_BEZ_MAXIT 40
#endif
__device__ __forceinline__ bool bezier_newton_seed(const BezDev &Z, d3 o, d3 d, int seed, double &t_out, d3 &nrm_out) {
    const d3 pos = mk(Z.pos[0], Z.pos[1], Z.pos[2]);
    const double rmax = Z.box[0] - Z.pos[0];
    const double tc = dot(pos - o, d);  // closest approach to the axis point
    const double tlo = fmax(tc - 2.0 * rmax - (Z.box[2] - Z.box[3]), 0.0), thi = tc + 2.0 * rmax + (Z.box[2] - Z.box[3]);
    const int iu = seed >> 2, it = seed & 3;
    double u0 = (iu + 0.5) * 0.25;
    double t0 = tlo + (thi - tlo) * (it + 0.5) * 0.25;
    d3 pt = o + d * t0 - pos;
    double theta = (pt.z < 0) ? 3.14159265 + atan(pt.x / pt.z) : atan(pt.x / pt.z);
    d3 par = mk(t0, u0, theta);
    d3 P, dP;
    double s, c;
    d3 F = bez_F(Z, par, o, d, P, dP, s, c);
    int iter = 0;
    while (sqrt(dot(F, F)) > 1e-6 && iter < CGRT_BEZ_MAXIT) {  // bezier.h:170
        iter++;
        // Jacobian columns (bezier.h:150-162)
        d3 a = d;
        d3 b = mk(-s * dP.z, -dP.y, -c * dP.z);
        d3 cc = mk(-c * P.z, 0.0, s * P.z);
        double D = det3(a, b, cc);
        if (D < 1e-4 && D > -1e-4) {  // vec3.h:105: singular -> the reference jitters; we nudge deterministically
            par = mk(par.x + 0.037, par.y + 0.029 * ((iter & 1) ? 1 : -1), par.z + 0.041);
            F = bez_F(Z, par, o, d, P, dP, s, c);
            continue;
        }
        // inverse (vec3.h:109-117) applied to F (vec3.h:99-101)
        // one reciprocal and nine products instead of the reference's nine quotients (vec3.h:109-117): the step differs from the
        // reference's in the last bits only, Newton corrects itself, and the roots of this primitive are compared statistically anyway
        // (the reference draws its starting points at random, SURVEY Q14). 10.1 -> 7.9 ms per round on c1.
        const double iD = 1.0 / D;
        d3 ra = mk((b.y * cc.z - b.z * cc.y) * iD, (cc.y * a.z - cc.z * a.y) * iD, (a.y * b.z - a.z * b.y) * iD);
        d3 rb = mk((cc.x * b.z - cc.z * b.x) * iD, (a.x * cc.z - a.z * cc.x) * iD, (b.x * a.z - b.z * a.x) * iD);
        d3 rc = mk((b.x * cc.y - cc.x * b.y) * iD, (cc.x * a.y - cc.y * a.x) * iD, (a.x * b.y - a.y * b.x) * iD);
        d3 step = ra * F.x + rb * F.y + rc * F.z;
        par = par - step;
        F = bez_F(Z, par, o, d, P, dP, s, c);
    }
    if (!(sqrt(dot(F, F)) < 1e-4 && par.x > 0 && par.y <= 1 && par.y >= 0)) return false;  // bezier.h:257
    t_out = par.x;
    d3 g = normalize(dP);  // bezier.h:215-224
    nrm_out = mk(g.y * s, -g.z, g.y * c);
    return true;
}
// bezier.h:272-281: orient the normal against the ray, then the top-cap disc (which overrides len even when farther, but is only
// reported when Newton also hit, bezier.h:289).
__device__ __forceinline__ void bezier_finish(const BezDev &Z, d3 o, d3 d, double &len, d3 &nrm) {
    const d3 pos = mk(Z.pos[0], Z.pos[1], Z.pos[2]);
    nrm = nrm * ((dot(nrm, d) < 0) ? 1.0 : -1.0);
    double newt = Z.box[2] - o.y;
    if (newt > 0.1) {
        newt = newt / d.y;
        d3 np = o + d * newt;
        if ((np.x - pos.x) * (np.x - pos.x) + (np.z - pos.z) * (np.z - pos.z) <= Z.umin_r2) {
            len = newt;
            nrm = mk(0, 1, 0);
        }
    }
}
// Bezier::intersect (bezier.h:225-290), one thread: the seeds in order, the nearest accepted root wins (the first one on ties).
__device__ bool bezier_intersect(const BezDev &Z, d3 o, d3 d, double &len, d3 &nrm) {
    if (!box_any_face_hit(Z.box, o, d)) return false;
    bool flag = false;
    len = CGRT_INF;
    for (int seed = 0; seed < CGRT_BEZ_SEEDS; seed++) {
        double t; d3 nv;
        if (bezier_newton_seed(Z, o, d, seed, t, nv) && t < len) { len = t; nrm = nv; flag = true; }
    }
    bezier_finish(Z, o, d, len, nrm);
    return flag;
}
// The same for one ray per HALF-WARP: lane j of the half runs seed j, the minimum of (t, seed) is found by shuffles. All 16 lanes of
// the half must call it with the same ray; every lane returns the result.
__device__ __forceinline__ bool bezier_intersect_halfwarp(const BezDev &Z, d3 o, d3 d, double &len, d3 &nrm) {
    const unsigned int lane = threadIdx.x & 31u, half_mask = (lane < 16u) ? 0x0000ffffu : 0xffff0000u;
    if (!box_any_face_hit(Z.box, o, d)) return false;  // uniform within the half
    double t = CGRT_INF; d3 nv = mk(0, 0, 0);
    bool ok = bezier_newton_seed(Z, o, d, (int)(lane & 15u), t, nv);
    if (!ok) t = CGRT_INF;
    int who = ok ? (int)(lane & 15u) : 16;
#pragma unroll
    for (int off = 8; off >= 1; off >>= 1) {  // lexicographic minimum of (t, seed) over the 16 lanes
        double t2 = __shfl_xor_sync(half_mask, t, off);
        int w2 = __shfl_xor_sync(half_mask, who, off);
        if (t2 < t || (t2 == t && w2 < who)) { t = t2; who = w2; }
    }
    if (who >= 16) return false;
    const int src = (int)(lane & 16u) + who;
    nv.x = __shfl_sync(half_mask, nv.x, src); nv.y = __shfl_sync(half_mask, nv.y, src); nv.z = __shfl_sync(half_mask, nv.z, src);
    len = t; nrm = nv;
    bezier_finish(Z, o, d, len, nrm);
    return true;
}

// ---------------------------------------------------------------------------------------------------------------
// The closest-hit loop of trace(), main.cpp:50-63: objects in insertion order, strict <, nearest starts at INF —
// i.e. the lexicographic minimum of (len, object index) over the objects that report a hit. That formulation is
// order-independent, which is what lets a thread block split the loop in two:
//   phase 1  every thread evaluates the analytic primitives of its own ray (planes, spheres, Bezier) in fp64;
//   phase 2  per BVH-backed object (mesh, displaced floor) the rays whose padded root box is reachable are compacted
//            into a shared-memory work list with a warp ballot + one shared atomic per warp, and the FIRST `count`
//            threads of the block traverse one listed ray each. Incoherent photon rays mostly miss the meshes, so
//            without the compaction a warp would sit through a traversal with 2-3 live lanes (measured: 2.4).
// A BVH candidate replaces the current nearest iff t < nearest, or t == nearest and its object precedes the holder:
// the traversal limit is `nearest` or the next double above it accordingly, and its own test stays strict.
// ---------------------------------------------------------------------------------------------------------------
template <int BLOCK>
struct TraceShared {
    double ox[BLOCK], oy[BLOCK], oz[BLOCK], dx[BLOCK], dy[BLOCK], dz[BLOCK];
    double lim[BLOCK];            // in: traversal limit of the listed ray; out: closest t
    int leaf[BLOCK];              // out: 1 if the deferred object won
    double near_in[BLOCK];        // in: nearest so far
    int id_in[BLOCK];             // in: its object id; out: primitive id of the new hit
    unsigned short list[BLOCK];   // compacted thread slots
    unsigned int count;
    unsigned int scratch[8];      // per-kernel block aggregates
};

__device__ __forceinline__ double next_up(double x) { return __longlong_as_double(__double_as_longlong(x) + 1); }  // x > 0 finite

// Plane part of Plane::intersect (objects.h:505-508): len = (p - o).n / d.n, a hit iff len > 0.
// A photon that has just bounced off a plane starts ON it: the numerator is then exactly 0 (or a few ulp). 0 / x is +-0 or NaN, never
// > 0, so the reference reports no hit; the quotient is not formed here in that case because a zero operand sends the fp64 division
// down its slow path — measured at 15 % of all instructions of the photon kernel, executed by ~5 lanes of 32.
__device__ __forceinline__ double plane_len(const ObjDev &O, d3 o, d3 d) {
    d3 n = mk(O.b[0], O.b[1], O.b[2]);
    d3 dd = mk(O.a[0], O.a[1], O.a[2]) - o;
    double num = dot(dd, n);
    if (num == 0.0) return 0.0;
    return num / dot(d, n);
}

struct HitAcc {
    double nearest;
    int id, prim;
    d3 nrm;
};

// phase 1: the cheap analytic primitives of one ray (planes, spheres), in object order. Meshes, displaced floors and Bezier
// surfaces are "deferred objects": phase 2 resolves them with the lanes that actually need them packed densely.
__device__ __forceinline__ void plane_take(const SceneDev &S, int i, double len, HitAcc &A) {
    if (len > 0 && len < A.nearest) {
        const ObjDev &O = S.obj[i];
        A.id = i; A.nearest = len; A.nrm = mk(O.b[0], O.b[1], O.b[2]); A.prim = -1;
    }
}
__device__ __forceinline__ void analytic_phase(const SceneDev &S, d3 o, d3 d, HitAcc &A) {
    A.nearest = CGRT_INF; A.id = -1; A.prim = -1; A.nrm = mk(0, 0, 0);
    // planes (objects.h:505-524; the displaced mesh of a bump plane is a phase-2 candidate), ascending index, strict <: the first of
    // several planes at the same distance keeps the hit, as in the reference's loop. Three independent quotients are in flight at a time.
    int k = 0;
    for (; k + 3 <= S.nplane; k += 3) {
        const int i0 = S.plane_ix[k], i1 = S.plane_ix[k + 1], i2 = S.plane_ix[k + 2];
        const double l0 = plane_len(S.obj[i0], o, d), l1 = plane_len(S.obj[i1], o, d), l2 = plane_len(S.obj[i2], o, d);
        plane_take(S, i0, l0, A); plane_take(S, i1, l1, A); plane_take(S, i2, l2, A);
    }
    for (; k < S.nplane; k++) {
        const int i = S.plane_ix[k];
        plane_take(S, i, plane_len(S.obj[i], o, d), A);
    }
    // spheres (objects.h:45-68) after the planes: a sphere at exactly the distance of the holder wins iff it precedes it in the object list
    for (k = 0; k < S.nsphere; k++) {
        const int i = S.sphere_ix[k];
        const ObjDev &O = S.obj[i];
        d3 l = mk(O.a[0], O.a[1], O.a[2]) - o;
        double tca = dot(l, d);
        double l2 = dot(l, l);
        if (!(tca < 0 && l2 > O.r2)) {
            double d2 = dot(l, l) - tca * tca;
            if (!(d2 > O.r2)) {
                double thc = sqrt(O.r2 - d2);
                double t0 = tca - thc, t1 = tca + thc;
                double len = (t0 < 0) ? t1 : t0;
                if (len < A.nearest || (len == A.nearest && i < A.id)) {
                    d3 p = o + d * len;
                    A.id = i; A.nearest = len; A.prim = -1;
                    A.nrm = normalize(p - mk(O.a[0], O.a[1], O.a[2]));
                }
            }
        }
    }
}
__device__ __forceinline__ bool is_deferred(const ObjDev &O) { return O.bvh >= 0 || O.kind == OBJ_BEZIER; }
// phase 2, per deferred object i: does this ray have to visit it, and (meshes) up to which t (exclusive)?
__device__ __forceinline__ bool deferred_wanted(const SceneDev &S, int i, d3 o, d3 d, const HitAcc &A, double &lim) {
    const ObjDev &O = S.obj[i];
    lim = (A.id > i) ? next_up(A.nearest) : A.nearest;
    if (O.kind == OBJ_BEZIER) return box_any_face_hit(S.bez[O.aux].box, o, d);  // the first test of Bezier::intersect (bezier.h:226-231)
    if (O.kind == OBJ_PLANE) {  // objects.h:513-517: only when the plane itself is hit, and only lenp < len
        double len = plane_len(O, o, d);
        if (!(len > 0)) return false;
        lim = len < lim ? len : lim;
    }
    return root_box_hit(S.bvh[O.bvh], o, d, lim);
}
__device__ __forceinline__ void bvh_merge(const SceneDev &S, int i, int leaf, double t, HitAcc &A) {
    const ObjDev &O = S.obj[i];
    const BvhDev &B = S.bvh[O.bvh];
    const TriRec &T = B.tris[leaf];
    d3 nv = mk(T.n[0], T.n[1], T.n[2]) * B.orient_sign;
    if (O.kind == OBJ_MESH && O.objtype == 2) nv = nv * ((nv.y > 0) ? 1.0 : -1.0);  // objects.h:434-436
    A.id = i; A.nearest = t; A.nrm = nv; A.prim = B.tri_id[leaf];
}

// Resolve deferred object i for one ray and merge it into A with the (len, index) order of main.cpp:55-63.
template <bool COUNT, bool BEZ, bool F32 = false>
__device__ __forceinline__ bool deferred_resolve(const SceneDev &S, int i, d3 o, d3 d, double lim, HitAcc &A, TravCounters *tc) {
    const ObjDev &O = S.obj[i];
    if (O.kind == OBJ_BEZIER) {
        if (BEZ) {
            double len; d3 nv;
            if (bezier_intersect(S.bez[O.aux], o, d, len, nv) && (len < A.nearest || (len == A.nearest && i < A.id))) {
                A.id = i; A.nearest = len; A.nrm = nv; A.prim = -1;
                return true;
            }
        }
        return false;
    }
    double t; int leaf;
    if (!bvh4_closest<COUNT, F32>(S.bvh[O.bvh], o, d, lim, t, leaf, tc)) return false;
    bvh_merge(S, i, leaf, t, A);
    return true;
}

// Block-cooperative form (eye pass, parity hooks): every thread of the block must call it.
template <int BLOCK, bool COUNT, bool F32 = false>
__device__ __forceinline__ bool closest_hit_block(const SceneDev &S, bool active, d3 o, d3 d, Hit &h, TraceShared<BLOCK> &sm, TravCounters *tc) {
    HitAcc A;
    A.nearest = CGRT_INF; A.id = -1; A.prim = -1; A.nrm = mk(0, 0, 0);
    if (active) analytic_phase(S, o, d, A);
    const int tid = threadIdx.x, lane = tid & 31;
    for (int i = 0; i < S.nobj; i++) {  // uniform control flow: S is uniform
        const ObjDev &O = S.obj[i];
        if (!is_deferred(O)) continue;
        double lim = 0;
        bool want = active && deferred_wanted(S, i, o, d, A, lim);
        if (tid == 0) sm.count = 0;
        __syncthreads();
        unsigned int mask = __ballot_sync(0xffffffffu, want);
        unsigned int base = 0;
        if (mask) {
            if (lane == __ffs(mask) - 1) base = atomicAdd(&sm.count, (unsigned int)__popc(mask));
            base = __shfl_sync(0xffffffffu, base, __ffs(mask) - 1);
        }
        if (want) {
            sm.list[base + __popc(mask & ((1u << lane) - 1u))] = (unsigned short)tid;
            sm.ox[tid] = o.x; sm.oy[tid] = o.y; sm.oz[tid] = o.z;
            sm.dx[tid] = d.x; sm.dy[tid] = d.y; sm.dz[tid] = d.z;
            sm.lim[tid] = lim;
            sm.near_in[tid] = A.nearest; sm.id_in[tid] = A.id;
        }
        __syncthreads();
        if (O.kind == OBJ_BEZIER) {
            // one listed ray per half-warp, one Newton seed per lane; every half runs the same number of rounds
            const int half = tid >> 4, nhalf = BLOCK / 16, cnt = (int)sm.count;
            for (int r = 0; r * nhalf < cnt; r++) {
                const int e = r * nhalf + half;
                const bool live = e < cnt;
                const int s = live ? sm.list[e] : 0;
                double len; d3 nv;
                bool hit = live && bezier_intersect_halfwarp(S.bez[O.aux], mk(sm.ox[s], sm.oy[s], sm.oz[s]), mk(sm.dx[s], sm.dy[s], sm.dz[s]), len, nv);
                if (live) __syncwarp((tid & 16) ? 0xffff0000u : 0x0000ffffu);  // all 16 lanes have read the ray before lane 0 overwrites it
                hit = hit && (len < sm.near_in[s] || (len == sm.near_in[s] && i < sm.id_in[s]));
                if (live && (tid & 15) == 0) {
                    sm.leaf[s] = hit ? 1 : 0;
                    if (hit) { sm.lim[s] = len; sm.ox[s] = nv.x; sm.oy[s] = nv.y; sm.oz[s] = nv.z; sm.id_in[s] = -1; }
                }
            }
        } else if (tid < (int)sm.count) {
            int s = sm.list[tid];
            HitAcc R;
            R.nearest = sm.near_in[s]; R.id = sm.id_in[s]; R.prim = -1; R.nrm = mk(0, 0, 0);
            bool hit = deferred_resolve<COUNT, false, F32>(S, i, mk(sm.ox[s], sm.oy[s], sm.oz[s]), mk(sm.dx[s], sm.dy[s], sm.dz[s]), sm.lim[s], R, tc);
            sm.leaf[s] = hit ? 1 : 0;
            if (hit) {
                sm.lim[s] = R.nearest; sm.ox[s] = R.nrm.x; sm.oy[s] = R.nrm.y; sm.oz[s] = R.nrm.z; sm.id_in[s] = R.prim;
            }
        }
        __syncthreads();
        if (want && sm.leaf[tid]) { A.id = i; A.nearest = sm.lim[tid]; A.nrm = mk(sm.ox[tid], sm.oy[tid], sm.oz[tid]); A.prim = sm.id_in[tid]; }
        __syncthreads();  // results are consumed before the next deferred object re-uses the arrays
    }
    h.obj = A.id; h.t = A.nearest; h.n = A.nrm; h.prim = A.prim;
    return A.id >= 0;
}

// Texture::color, texture.h:39-72; Plane::getSurfaceColor objects.h:533-539
__device__ __forceinline__ d3 surface_color(const SceneDev &S, int obj, d3 point) {
    const ObjDev &O = S.obj[obj];
    d3 flat = mk(O.col[0], O.col[1], O.col[2]);
    if (O.kind != OBJ_PLANE || O.tex < 0) return flat;
    const TexDev &T = S.tex[O.tex];
    const double texteps = 1e-2;
    d3 n = mk(T.n[0], T.n[1], T.n[2]);
    d3 dd = point - mk(T.p[0], T.p[1], T.p[2]);
    dd = dd - n * dot(dd, n);
    int r, c;
    if (dd.x < texteps && dd.x > -texteps) {
        if (0 < dd.y && dd.y < T.lenx && 0 < dd.z && dd.z < T.leny) {
            r = (int)floor(dd.y / T.lenx * T.H);
            c = (int)floor(dd.z / T.leny * T.W);
        } else return flat;
    } else if (dd.y < texteps && dd.y > -texteps) {
        if (0 < dd.x && dd.x < T.lenx && 0 < dd.z && dd.z < T.leny) {
            c = (int)floor(dd.x / T.lenx * T.W);
            r = (int)floor(dd.z / T.leny * T.H);
        } else return flat;
    } else if (dd.z < texteps && dd.z > -texteps) {
        if (0 < dd.x && dd.x < T.lenx && 0 < dd.y && dd.y < T.leny) {
            c = (int)floor(dd.x / T.lenx * T.W);
            r = T.H - 1 - (int)floor(dd.y / T.leny * T.H);
        } else return flat;
    } else {
        return flat;
    }
    r = r < 0 ? 0 : (r >= T.H ? T.H - 1 : r);
    c = c < 0 ? 0 : (c >= T.W ? T.W - 1 : c);
    uchar4 tx = __ldg(T.texels + (size_t)r * T.W + c);
    return mk((double)tx.x / 256.0, (double)tx.y / 256.0, (double)tx.z / 256.0);
}

// hash.h:35-42: ix = (int)floor((x - XMIN) / celllength). The quotient is first formed with a reciprocal multiply (|error| <= 2 ulp);
// floor() of it equals floor() of the IEEE quotient unless the product lies within a few ulp of an integer, and only then is the
// division actually performed. Same integers as the reference, three fp64 divisions fewer on almost every call.
__host__ __device__ __forceinline__ int cell_floor_div(double num, double den, double inv_den) {
    double q = num * inv_den;
    double f = floor(q);
    double tol = fabs(q) * 1e-15 + 1e-300;
    if (q - f < tol || (f + 1.0) - q < tol) f = floor(num / den);
    return (int)f;
}
__host__ __device__ __forceinline__ void cell_coord(d3 p, double celllength, double inv, int &ix, int &iy, int &iz) {
    ix = cell_floor_div(p.x - (-35.0), celllength, inv);
    iy = cell_floor_div(p.y - (-35.0), celllength, inv);
    iz = cell_floor_div(p.z - (-15.0), celllength, inv);
}
__host__ __device__ __forceinline__ uint32_t cell_hash(int ix, int iy, int iz, uint32_t hashsize) {
    return (((uint32_t)ix * 73856093u) ^ ((uint32_t)iy * 19349663u) ^ ((uint32_t)iz * 83492791u)) % hashsize;
}

}  // namespace cgrt
