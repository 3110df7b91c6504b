// cgrt_host.hpp — host-side C++ mirror of CGRayTracing's scene / render surface on top of the C ABI (include/cgrt.h).
//
// The reference keeps every scene object as a C++ class with four virtuals (headers/objects.h:17-24) and calls
// render(objs) once (main.cpp:401). This header keeps those names, constructor argument orders and meanings, so a
// main() written against the reference compiles against it with `using namespace cgrt_host;` — but nothing here
// computes on the CPU: the classes are descriptors; describe() hands them to a cgrt_ctx, and render() / intersect() /
// getSurfaceColor() run the sm_100a kernels behind libcgrt.so. Without a GPU every entry point throws (no CPU fallback).
//
//   reference                                            here
//   Vec3 (vec3.h:11-92)                                  Vec3 (plain value type; host arithmetic only builds descriptors)
//   Object::intersect / getSurfaceColor / getReflection  same signatures; GPU-backed single-ray queries (cgrt_intersect_batch)
//   Sphere(c,r,sc,refl,transp,ec)      objects.h:28-38   Sphere(c,r,sc,refl,transp,ec)
//   Plane(p,n,sc,refl,transp,tx,ec)    objects.h:480     Plane(p,n,sc,refl,transp,tx,ec)
//   TriangleMesh(file,a,b,sc,refl,transp,type,ec) :338   TriangleMesh(file,a,b,sc,refl,transp,type,ec)  (same 3 text formats)
//   Bezier(points,pos,sc,refl,transp,type,ec) bezier.h:44  Bezier(points,pos,sc,refl,transp,type,ec)
//   Texture(data,n,p,lx,ly,flag)       texture.h:19      Texture(data,n,p,lx,ly,flag)  (data = vector<vector<Vec3>> of byte/256)
//   Hashtable(hashsize,celllength)     hash.h:22         Hashtable(hashsize,celllength): grid parameters + hash/compute_coord on the GPU
//   render(objs) + global image[][]    main.cpp:169,33   render(objs, RenderOptions) -> Image
#ifndef CGRT_HOST_HPP_
#define CGRT_HOST_HPP_

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <memory>
#include <sstream>
#include <stdexcept>
#include <string>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <vector>

#include "cgrt.h"

namespace cgrt_host {

struct Error : std::runtime_error {
    int status;
    Error(int st, const std::string &what) : std::runtime_error(what), status(st) {}
};

// ---------------------------------------------------------------------------------------------------------------------
struct Vec3 {
    double x, y, z;
    Vec3() : x(0), y(0), z(0) {}
    Vec3(double v) : x(v), y(v), z(v) {}  // the reference passes `0` for "no emission colour"
    Vec3(double x_, double y_, double z_) : x(x_), y(y_), z(z_) {}
    Vec3 operator+(const Vec3 &o) const { return Vec3(x + o.x, y + o.y, z + o.z); }
    Vec3 operator-(const Vec3 &o) const { return Vec3(x - o.x, y - o.y, z - o.z); }
    Vec3 operator-() const { return Vec3(-x, -y, -z); }
    Vec3 operator*(double f) const { return Vec3(x * f, y * f, z * f); }
    Vec3 operator*(const Vec3 &o) const { return Vec3(x * o.x, y * o.y, z * o.z); }
    Vec3 mul(const Vec3 &o) const { return *this * o; }
    double dot(const Vec3 &o) const { return x * o.x + y * o.y + z * o.z; }
    Vec3 cross(const Vec3 &o) const { return Vec3(y * o.z - z * o.y, z * o.x - x * o.z, x * o.y - y * o.x); }
    Vec3 copy() const { return *this; }
    Vec3 &normalize() {
        double len = std::sqrt(x * x + y * y + z * z);
        if (len > 0) { x *= 1 / len; y *= 1 / len; z *= 1 / len; }
        return *this;
    }
    const double *data() const { return &x; }
};

// ---------------------------------------------------------------------------------------------------------------------
// One GPU context with RAII and status -> exception translation.
class Context {
public:
    explicit Context(int device = 0) {
        int st = cgrt_create(device, &ctx_);
        if (st != CGRT_OK) throw Error(st, "cgrt_create failed (status " + std::to_string(st) + "): no usable CUDA device, and there is no CPU fallback");
    }
    ~Context() { cgrt_destroy(ctx_); }
    Context(const Context &) = delete;
    Context &operator=(const Context &) = delete;
    cgrt_ctx *get() const { return ctx_; }
    void check(int st) const {
        if (st != CGRT_OK) throw Error(st, std::string("libcgrt: ") + cgrt_last_error(ctx_));
    }

private:
    cgrt_ctx *ctx_ = nullptr;
};

// ---------------------------------------------------------------------------------------------------------------------
// Texture(data, n, p, lx, ly, flag) — texture.h:19. `data[i][j]` are texels as the reference stores them: byte/256.
class Texture {
public:
    Texture() : height(0), width(0), lenx(0), leny(0), isbump(false) {}
    Texture(const std::vector<std::vector<Vec3>> &data, const Vec3 &n, const Vec3 &p, double lx, double ly, bool flag = false)
        : height((int)data.size()), width(data.empty() ? 0 : (int)data[0].size()), normal(n), pos(p), lenx(lx), leny(ly), isbump(flag) {
        rgb.resize((size_t)height * width * 3);
        for (int i = 0; i < height; i++)
            for (int j = 0; j < width; j++) {
                const Vec3 &t = data[i][j];
                const double c[3] = {t.x, t.y, t.z};
                for (int k = 0; k < 3; k++) rgb[((size_t)i * width + j) * 3 + k] = (uint8_t)std::lround(c[k] * 256.0);  // exact: texel = byte/256
            }
    }
    // raw bytes as stbi_load(..., 3) returns them (main.cpp:300)
    Texture(const uint8_t *bytes, int w, int h, const Vec3 &n, const Vec3 &p, double lx, double ly, bool flag = false)
        : height(h), width(w), normal(n), pos(p), lenx(lx), leny(ly), isbump(flag), rgb(bytes, bytes + (size_t)w * h * 3) {}
    bool empty() const { return rgb.empty(); }
    int describe(const Context &c) const {
        int id = -1;
        c.check(cgrt_add_texture(c.get(), rgb.data(), width, height, normal.data(), pos.data(), lenx, leny, isbump ? 1 : 0, &id));
        return id;
    }
    int height, width;
    Vec3 normal, pos;
    double lenx, leny;
    bool isbump;
    std::vector<uint8_t> rgb;
};

// ---------------------------------------------------------------------------------------------------------------------
// The plugin surface, objects.h:17-24. describe() is the one addition: it serialises the object into a context.
class Object {
public:
    virtual ~Object() {}
    virtual int describe(const Context &c) const = 0;
    virtual double getTransparency() const = 0;
    virtual double getReflection() const = 0;

    // Closest hit of THIS object, as the reference's virtual returns it: len and the object's raw normal. Runs on the GPU
    // through a private single-object context (built on first use) — meant for spot checks, not for bulk work.
    bool intersect(const Vec3 &rayorig, const Vec3 &raydir, double &len, Vec3 &normalvector) const {
        const Context &c = solo();
        double t = 0, nr[3] = {0, 0, 0};
        int32_t obj = -1;
        c.check(cgrt_intersect_batch(c.get(), 1, rayorig.data(), raydir.data(), &t, nullptr, nr, &obj, nullptr, nullptr));
        if (obj < 0) return false;
        len = t;
        normalvector = Vec3(nr[0], nr[1], nr[2]);
        return true;
    }
    Vec3 getSurfaceColor(const Vec3 &point) const {
        const Context &c = solo();
        double col[3];
        c.check(cgrt_surface_color(c.get(), 0, 1, point.data(), col));
        return Vec3(col[0], col[1], col[2]);
    }

private:
    const Context &solo() const {
        if (!solo_) {
            solo_.reset(new Context());
            describe(*solo_);
            solo_->check(cgrt_commit_scene(solo_->get()));
        }
        return *solo_;
    }
    mutable std::unique_ptr<Context> solo_;
};

class Sphere : public Object {
public:
    Sphere(const Vec3 &c, double r, const Vec3 &sc, double refl = 0, double transp = 0, const Vec3 &ec = 0)
        : center(c), radius(r), surfaceColor(sc), emissionColor(ec), transparency(transp), reflection(refl) {}
    int describe(const Context &c) const override {
        int id = -1;
        c.check(cgrt_add_sphere(c.get(), center.data(), radius, surfaceColor.data(), reflection, transparency, &id));
        return id;
    }
    double getTransparency() const override { return transparency; }
    double getReflection() const override { return reflection; }
    Vec3 center;
    double radius;
    Vec3 surfaceColor, emissionColor;
    double transparency, reflection;
};

class Plane : public Object {
public:
    Plane(const Vec3 &p, const Vec3 &n, const Vec3 &sc, double refl = 0, double transp = 0, const Texture &tx = Texture(), const Vec3 &ec = 0)
        : position(p), normal(n), surfaceColor(sc), transparency(transp), reflection(refl), texture(tx) { (void)ec; }
    int describe(const Context &c) const override {
        int tex = texture.empty() ? -1 : texture.describe(c);  // the reference copies the Texture into the Plane (objects.h:481)
        int id = -1;
        c.check(cgrt_add_plane(c.get(), position.data(), normal.data(), surfaceColor.data(), reflection, transparency, tex, &id));
        return id;
    }
    double getTransparency() const override { return transparency; }
    double getReflection() const override { return reflection; }
    Vec3 position, normal, surfaceColor;
    double transparency, reflection;
    Texture texture;
};

// TriangleMesh(file, a, b, sc, refl, transp, typeofdata, ec) — objects.h:338-403. The three text formats of the reference:
//   0  blocks "begin / vertex x y z (x3) / end"                                  (model/lowpolybunny.txt, model/test.txt)
//   1  "<nv>", nv lines "v  x y z", "<nf>", nf lines "f a b c" (1-based)           (model/dragon.txt, model/tri.txt)
//   2  like 1 with "v x y z" and faces "f a/b/c d/e/f g/h/i" (first index of each triple) (model/Mesh000.obj)
// Every vertex becomes Vec3(x, y, -z) * a + b (objects.h:348,365,384).
class TriangleMesh : public Object {
public:
    TriangleMesh(const char *filename, double a, const Vec3 &b, const Vec3 &sc, double refl = 0, double transp = 0, int typeofdata = 0,
                 const Vec3 &ec = 0)
        : surfaceColor(sc), transparency(transp), reflection(refl), objtype(typeofdata) {
        (void)ec;
        std::ifstream in(filename);
        if (!in) throw Error(CGRT_ERR_INVALID, std::string("cannot open mesh file ") + filename);
        std::vector<Vec3> verts;
        std::string line, tag;
        auto xf = [&](double x, double y, double z) { return Vec3(x, y, -z) * a + b; };
        while (std::getline(in, line)) {
            std::istringstream ss(line);
            if (!(ss >> tag)) continue;
            if (typeofdata == 0) {
                double x, y, z;
                if (tag == "vertex" && (ss >> x >> y >> z)) push(xf(x, y, z));
            } else if (tag == "v") {
                double x, y, z;
                if (ss >> x >> y >> z) verts.push_back(xf(x, y, z));
            } else if (tag == "f") {
                std::string t;
                int id[3], k = 0;
                while (k < 3 && (ss >> t)) id[k++] = std::atoi(t.c_str());  // "a" or "a/b/c": atoi stops at '/'
                if (k == 3)
                    for (int q = 0; q < 3; q++) {
                        if (id[q] < 1 || id[q] > (int)verts.size()) throw Error(CGRT_ERR_INVALID, "mesh face index out of range");
                        push(verts[(size_t)id[q] - 1]);
                    }
            }
        }
        if (tri9.empty() || tri9.size() % 9) throw Error(CGRT_ERR_INVALID, std::string("no triangles parsed from ") + filename);
    }
    // already-transformed triangles (pa, pb, pc) x n
    TriangleMesh(const std::vector<double> &triangles9, const Vec3 &sc, double refl = 0, double transp = 0, int typeofdata = 0)
        : tri9(triangles9), surfaceColor(sc), transparency(transp), reflection(refl), objtype(typeofdata) {}
    int describe(const Context &c) const override {
        int id = -1;
        c.check(cgrt_add_mesh(c.get(), tri9.data(), (int)(tri9.size() / 9), surfaceColor.data(), reflection, transparency, objtype, &id));
        return id;
    }
    double getTransparency() const override { return transparency; }
    double getReflection() const override { return reflection; }
    size_t size() const { return tri9.size() / 9; }
    std::vector<double> tri9;
    Vec3 surfaceColor;
    double transparency, reflection;
    int objtype;

private:
    void push(const Vec3 &v) { tri9.push_back(v.x); tri9.push_back(v.y); tri9.push_back(v.z); }
};

class Bezier : public Object {
public:
    Bezier(const std::vector<Vec3> &pts, const Vec3 &pos, const Vec3 &sc, double refl = 0, double transp = 0, int typeofdata = 0, const Vec3 &ec = 0)
        : points(pts), position(pos), surfaceColor(sc), transparency(transp), reflection(refl) { (void)typeofdata; (void)ec; }
    int describe(const Context &c) const override {
        std::vector<double> cp;
        for (const Vec3 &p : points) { cp.push_back(p.x); cp.push_back(p.y); cp.push_back(p.z); }
        int id = -1;
        c.check(cgrt_add_bezier(c.get(), cp.data(), (int)points.size(), position.data(), surfaceColor.data(), reflection, transparency, &id));
        return id;
    }
    double getTransparency() const override { return transparency; }
    double getReflection() const override { return reflection; }
    std::vector<Vec3> points;
    Vec3 position, surfaceColor;
    double transparency, reflection;
};

// ---------------------------------------------------------------------------------------------------------------------
// Hashtable(hashsize, celllength) — hash.h:22-42. Only the grid parameters live on the host; keys come from the GPU.
class Hashtable {
public:
    Hashtable(int hashsize_, double celllength_) : hashsize(hashsize_), celllength_in(celllength_) {
        num_of_cell_per_dim = (int)std::ceil(70.0 / celllength_);  // SIZE_OF_SCENE = 70, hash.h:11,25-26
        celllength = 70.0 / num_of_cell_per_dim;
    }
    // compute_coord + hash for n positions (xyz interleaved): key[n], ixyz[3n] (either may be null)
    void keys(const Context &c, int64_t n, const double *pos, uint32_t *key, int32_t *ixyz) const {
        c.check(cgrt_hash_keys(c.get(), n, pos, hashsize, celllength_in, key, ixyz));
    }
    int hashsize, num_of_cell_per_dim;
    double celllength_in, celllength;
};

// ---------------------------------------------------------------------------------------------------------------------
// trace(org, dir, objs, flux, adj, flag, depth, htable, x, y) — main.cpp:42 — for a batch of rays. The scene (`objs`) and the table
// (`htable`) are the context's: describe() the objects into it and commit first. flag = true: eye rays, weight = adj, (x, y) = pixel,
// hitpoints are inserted (before cgrt_build_grid); flag = false: photons, weight = flux, deposits (after cgrt_build_grid), ray k draws the
// random numbers of photon index first_index + k.
inline void trace(const Context &c, const std::vector<Vec3> &org, const std::vector<Vec3> &dir, const std::vector<Vec3> &weight, bool flag, int depth,
                  const std::vector<int32_t> &x = std::vector<int32_t>(), const std::vector<int32_t> &y = std::vector<int32_t>(), uint64_t first_index = 0) {
    static_assert(sizeof(Vec3) == 3 * sizeof(double), "Vec3 is three packed doubles");
    if (dir.size() != org.size() || weight.size() != org.size() || (flag && (x.size() != org.size() || y.size() != org.size())))
        throw Error(CGRT_ERR_INVALID, "trace: array lengths differ");
    c.check(cgrt_trace(c.get(), (int64_t)org.size(), org.empty() ? nullptr : org[0].data(), dir.empty() ? nullptr : dir[0].data(),
                       weight.empty() ? nullptr : weight[0].data(), flag ? 1 : 0, depth, x.empty() ? nullptr : x.data(), y.empty() ? nullptr : y.data(), first_index));
}

// ---------------------------------------------------------------------------------------------------------------------
// render(): main.cpp:169-266. Every literal of the reference is a field with the reference's value as default.
struct RenderOptions {
    int width = 1024, height = 768;      // main.cpp:28-29
    int num_of_samples = 1;              // :177
    bool depth_of_field = false;         // trace the thin-lens ray of :203-207 instead of the pinhole ray
    int num_photon = 2560000;            // :223 — photons per "thread"
    int num_threads = 8;                 // :224 — the reference traces num_photon * num_threads photons in total (:222,256)
    int rounds = 1;                      // per-round radius/flux updates the total is split into (reference: per photon, SURVEY Q1)
    int hashsize = 1000001;              // :184
    int accum_mode = 0;                  // 0: fp64 atomics, 1: float32 x4 accumulators
    bool per_photon_update = false;      // true: the reference's own rule, main.cpp:119-122 — every accepted photon shrinks the radius at once
                                         // (one GPU; `rounds` then only says how often filter radii are refreshed). false: one update per round
    uint64_t seed = 20261018ull;
    int device = 0;
    bool peer_exchange = false;          // num_gpus > 1: false: ncclAllReduce inside cgrt_round_update (measured fastest at 8 GPUs); true: exchange
                                         // the accumulators of a round over peer memory, fused with the update (cgrt_peer_*; fastest at 2 GPUs)
    int num_gpus = 1;                    // > 1: devices device .. device+num_gpus-1 of this box, one context and one host thread per GPU:
                                         // image rows and photon index ranges are split between them, NCCL (through the C ABI) carries the
                                         // hitpoint records and the per-round accumulators (SURVEY section 8e)
    int sppm = CGRT_SPPM_OFF;            // CGRT_SPPM_JITTER / CGRT_SPPM_CORNER: stochastic PPM, a new eye pass every round and per-pixel statistics
                                         // (cgrt_set_sppm); per-round update only. With num_gpus > 1 every round's eye pass is row-tiled and
                                         // its records all-gathered over NCCL; peer_exchange is not supported with it
};

struct Image {
    int width = 0, height = 0;
    std::vector<double> rgb;    // image[h][w] of main.cpp:33 (row 0 at the bottom), linear radiance
    std::vector<uint8_t> rgb8;  // what main.cpp:403-411 hands to stbi_write_png: tone-mapped, gamma 2.2, flipped
    Vec3 at(int h, int w) const { const double *p = &rgb[((size_t)h * width + w) * 3]; return Vec3(p[0], p[1], p[2]); }
};

// Where the ranks of one process (one host thread per GPU) hand each other their peer handles.
struct PeerHub {
    explicit PeerHub(int world) : blobs((size_t)world * CGRT_PEER_HANDLE_BYTES), world_(world) {}
    // deposits this rank's handle, returns when every rank has (or one has failed)
    bool exchange(int rank, const char *blob) {
        std::unique_lock<std::mutex> lk(m);
        if (blob) std::memcpy(&blobs[(size_t)rank * CGRT_PEER_HANDLE_BYTES], blob, CGRT_PEER_HANDLE_BYTES); else failed = true;
        arrived++;
        cv.notify_all();
        cv.wait(lk, [&] { return arrived >= world_; });
        return !failed;
    }
    std::vector<char> blobs;
    std::mutex m;
    std::condition_variable cv;
    int arrived = 0, world_;
    bool failed = false;
};

// One rank of render(): the whole of main.cpp:169-266 on one GPU for its share of the rows and of the photon indices. comm == nullptr:
// the single-GPU render.
inline Image render_rank(const std::vector<Object *> &objs, const RenderOptions &opt, int rank, int world, void *comm, cgrt_counters *counters,
                         PeerHub *hub = nullptr) {
    Context c(opt.device + rank);
    cgrt_config cfg;
    cgrt_default_config(&cfg);
    cfg.width = opt.width; cfg.height = opt.height; cfg.num_of_samples = opt.num_of_samples; cfg.use_dof = opt.depth_of_field ? 1 : 0;
    cfg.hashsize = opt.hashsize; cfg.accum_mode = opt.accum_mode; cfg.seed = opt.seed;
    cfg.update_mode = opt.per_photon_update ? 0 : 1;
    c.check(cgrt_set_config(c.get(), &cfg));
    for (const Object *o : objs) o->describe(c);  // object id = position in objs, like the reference's loop index (main.cpp:55)
    c.check(cgrt_commit_scene(c.get()));
    // main.cpp:185-219: contiguous row tiles, the remainder to the low ranks
    const int base = opt.height / world, rem = opt.height % world;
    const int y0 = rank * base + (rank < rem ? rank : rem), y1 = y0 + base + (rank < rem ? 1 : 0);
    if (opt.sppm) {  // every round traces its own eye pass (below); the communicator is attached first, as cgrt_set_sppm requires
        if (comm) c.check(cgrt_set_comm(c.get(), comm, world));
        c.check(cgrt_set_sppm(c.get(), opt.sppm));
    } else if (y1 > y0) {
        c.check(cgrt_eye_pass(c.get(), y0, y1));
    }
    if (comm && !opt.sppm) {
        c.check(cgrt_allgather_hitpoints(c.get(), comm, world));
        if (!hub) c.check(cgrt_set_comm(c.get(), comm, world));  // cgrt_round_update all-reduces the accumulators from now on
    }
    if (!opt.sppm) c.check(cgrt_build_grid(c.get()));  // hash.h:43-54 as a sorted grid
    if (hub) {  // the accumulators of a round are exchanged over peer memory, fused with the update
        char blob[CGRT_PEER_HANDLE_BYTES];
        int st = cgrt_peer_export(c.get(), blob);
        bool ok = hub->exchange(rank, st == CGRT_OK ? blob : nullptr);
        c.check(st);
        if (!ok) throw Error(CGRT_ERR_CUDA, "a peer rank failed to export its accumulator block");
        c.check(cgrt_peer_attach(c.get(), rank, world, hub->blobs.data()));
    }
    const uint64_t total = (uint64_t)opt.num_photon * (uint64_t)opt.num_threads;
    const int rounds = opt.rounds < 1 ? 1 : opt.rounds;
    uint64_t done = 0;
    for (int r = 0; r < rounds; r++) {                // main.cpp:221-249
        const uint64_t n = total / rounds + ((uint64_t)r < total % rounds ? 1 : 0);
        const uint64_t pb = n / world, pr = n % world;  // this rank's index range of the round
        const uint64_t first = done + (uint64_t)rank * pb + ((uint64_t)rank < pr ? (uint64_t)rank : pr);
        const uint64_t mine = pb + ((uint64_t)rank < pr ? 1 : 0);
        if (opt.sppm && comm) {  // this rank's row tile, the union of all tiles, the same grid on every rank
            c.check(cgrt_sppm_eye_pass(c.get(), (uint32_t)r, y0, y1));
            c.check(cgrt_allgather_hitpoints(c.get(), comm, world));
            c.check(cgrt_build_grid(c.get()));
        } else if (opt.sppm) {
            c.check(cgrt_sppm_begin_round(c.get(), (uint32_t)r));
        }
        if (mine) c.check(cgrt_photon_pass(c.get(), first, mine));
        c.check(cgrt_round_update(c.get()));
        done += n;
    }
    Image img;
    img.width = opt.width; img.height = opt.height;
    img.rgb.resize((size_t)opt.width * opt.height * 3);
    img.rgb8.resize(img.rgb.size());
    c.check(cgrt_gather_image(c.get(), (double)total, img.rgb.data(), img.rgb8.data()));  // main.cpp:252-258 (the library applies num_of_samples), 403-411
    if (counters) c.check(cgrt_get_counters(c.get(), counters));
    if (comm) c.check(cgrt_set_comm(c.get(), nullptr, 1));
    return img;
}

inline Image render(const std::vector<Object *> &objs, const RenderOptions &opt = RenderOptions(), cgrt_counters *counters = nullptr) {
    const int world = opt.num_gpus < 1 ? 1 : opt.num_gpus;
    if (opt.sppm && world > 1 && opt.peer_exchange)
        throw Error(CGRT_ERR_INVALID, "SPPM on several GPUs exchanges over NCCL: the peer exchange (peer_exchange = true) is not supported with it");
    if (opt.sppm && opt.per_photon_update) throw Error(CGRT_ERR_INVALID, "SPPM needs the per-round update (per_photon_update = false)");
    if (world == 1) return render_rank(objs, opt, 0, 1, nullptr, counters);
    std::vector<int> devs((size_t)world);
    for (int k = 0; k < world; k++) devs[(size_t)k] = opt.device + k;
    std::vector<void *> comms((size_t)world, nullptr);
    int rc = cgrt_comm_init_all(world, devs.data(), comms.data());
    if (rc != 0) throw Error(rc, "cgrt_comm_init_all failed (NCCL missing, or fewer GPUs than num_gpus?)");
    std::vector<Image> imgs((size_t)world);
    std::vector<cgrt_counters> ctrs((size_t)world);
    std::vector<std::string> errs((size_t)world);
    std::vector<int> stat((size_t)world, 0);
    PeerHub hub(world);
    std::vector<std::thread> th;
    for (int k = 0; k < world; k++)
        th.emplace_back([&, k] {
            try { imgs[(size_t)k] = render_rank(objs, opt, k, world, comms[(size_t)k], &ctrs[(size_t)k], opt.peer_exchange ? &hub : nullptr); }
            catch (const Error &e) { stat[(size_t)k] = e.status ? e.status : CGRT_ERR_CUDA; errs[(size_t)k] = e.what(); }
        });
    for (auto &t : th) t.join();
    for (void *cm : comms) cgrt_comm_destroy(cm);
    for (int k = 0; k < world; k++)
        if (stat[(size_t)k]) throw Error(stat[(size_t)k], "rank " + std::to_string(k) + ": " + errs[(size_t)k]);
    if (counters) {  // the job's totals: per-rank work counters add up, the hitpoint set is replicated
        *counters = ctrs[0];
        for (int k = 1; k < world; k++) {
            counters->eye_segments += ctrs[(size_t)k].eye_segments; counters->photon_segments += ctrs[(size_t)k].photon_segments;
            counters->diffuse_hits += ctrs[(size_t)k].diffuse_hits; counters->candidates += ctrs[(size_t)k].candidates;
            counters->deposits += ctrs[(size_t)k].deposits; counters->gathered_hits += ctrs[(size_t)k].gathered_hits;
            counters->exact_tests += ctrs[(size_t)k].exact_tests; counters->gpu_launches += ctrs[(size_t)k].gpu_launches;
        }
    }
    return imgs[0];  // every rank holds the same picture
}

// ---------------------------------------------------------------------------------------------------------------------
// Asset containers shipped with the package (cgraytracing_b200/assets, written by tools/make_assets.py)
inline std::vector<uint8_t> read_texture_asset(const std::string &path, int &w, int &h) {
    std::ifstream in(path, std::ios::binary);
    char magic[8];
    int32_t wh[2];
    if (!in.read(magic, 8) || std::string(magic, 8) != "CGRTTEX1" || !in.read((char *)wh, 8)) throw Error(CGRT_ERR_INVALID, "not a .cgrttex file: " + path);
    w = wh[0]; h = wh[1];
    std::vector<uint8_t> rgb((size_t)w * h * 3);
    if (!in.read((char *)rgb.data(), (std::streamsize)rgb.size())) throw Error(CGRT_ERR_INVALID, "truncated texture: " + path);
    return rgb;
}
// -> triangles after the loader arithmetic of objects.h:348,365,384: Vec3(x, y, -z) * a + b
inline std::vector<double> read_mesh_asset(const std::string &path, double a, const Vec3 &b) {
    std::ifstream in(path, std::ios::binary);
    char magic[8];
    int32_t nn[2];
    if (!in.read(magic, 8) || std::string(magic, 8) != "CGRTMSH1" || !in.read((char *)nn, 8)) throw Error(CGRT_ERR_INVALID, "not a .cgrtmesh file: " + path);
    if (nn[0] < 0 || nn[1] < 0) throw Error(CGRT_ERR_INVALID, "corrupt mesh header: " + path);
    std::vector<double> v((size_t)nn[0] * 3);
    std::vector<int32_t> f((size_t)nn[1] * 3);
    if (!in.read((char *)v.data(), (std::streamsize)(v.size() * 8)) || !in.read((char *)f.data(), (std::streamsize)(f.size() * 4)))
        throw Error(CGRT_ERR_INVALID, "truncated mesh: " + path);
    std::vector<double> tri9;
    tri9.reserve(f.size() * 3);
    for (int32_t id : f) {
        if (id < 0 || id >= nn[0]) throw Error(CGRT_ERR_INVALID, "mesh face index out of range: " + path);
        Vec3 p = Vec3(v[(size_t)id * 3], v[(size_t)id * 3 + 1], -v[(size_t)id * 3 + 2]) * a + b;
        tri9.push_back(p.x); tri9.push_back(p.y); tri9.push_back(p.z);
    }
    return tri9;
}

}  // namespace cgrt_host
#endif  // CGRT_HOST_HPP_
