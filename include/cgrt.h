/* cgrt.h — C ABI of the B200-native progressive-photon-mapping hot path (libcgrt.so).
 *
 * This is the drop-in boundary for CGRayTracing's trace()/render() path: the reference's host classes
 * (Object/Sphere/Plane/TriangleMesh/Bezier/Texture/Hashtable, headers/objects.h, bezier.h, texture.h, hash.h) stay on
 * the host as thin descriptors (cgraytracing_b200/host/cgrt_host.hpp); everything they compute on the hot path is
 * done behind these entry points by hand-written sm_100a kernels. Plain pointers and sizes only; no C++/torch types.
 *
 * Conventions: every function returns 0 on success or a negative cgrt_status; never throws; no global state; one
 * opaque cgrt_ctx per GPU; calls on one ctx are not thread-safe; the caller owns every host buffer; the ctx owns all
 * device memory. All `double*`/`int*` arguments are HOST pointers unless the name ends in `_dev`.
 * Citations are file:line in the reference (haoyuzhao123/CGRayTracing).
 */
#ifndef CGRT_H_
#define CGRT_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cgrt_ctx cgrt_ctx;

typedef enum cgrt_status {
    CGRT_OK = 0,
    CGRT_ERR_INVALID = -1,   /* bad argument / call order */
    CGRT_ERR_CUDA = -2,      /* a CUDA call failed; see cgrt_last_error */
    CGRT_ERR_NO_DEVICE = -3, /* no usable GPU: there is NO CPU fallback */
    CGRT_ERR_CAPACITY = -4,  /* a fixed-size table (objects, textures, BVHs, queue) is full, or a fixed-point sum left its range (accum_mode 2) */
    CGRT_ERR_NCCL = -5
} cgrt_status;

/* Every compile-time constant of render()/trace() (main.cpp:28-36, 177-184, 222-224) as a field. */
typedef struct cgrt_config {
    int32_t width, height;      /* main.cpp:28-29 */
    int32_t max_depth;          /* MAX_DEPTH, main.cpp:35 */
    int32_t num_of_samples;     /* main.cpp:177 */
    int32_t use_dof;            /* 1: trace the thin-lens ray of main.cpp:203-207 instead of the pinhole ray of :209 */
    int32_t hashsize;           /* Hashtable(hashsize, r), main.cpp:184 */
    int32_t accum_mode;         /* 0: fp64 atomics (parity), 1: one red.global.add.v4.f32 per deposit (fast), 2: fixed point — every accepted
                                 * pair adds round-half-even(cf * 2^22) to int64 sums, cf = ((float)f * (float)flux) * (float)(1/pi), so flux,
                                 * radii, counts and image are the same bits on every run and any GPU count. A value cf > 2^16 or a round's
                                 * M > 2^24 (per hitpoint; SPPM: per pixel) makes the next synchronising call return CGRT_ERR_CAPACITY.
                                 * Any other value is CGRT_ERR_INVALID. update_mode 0 always uses 0. */
    int32_t update_mode;        /* 1 (default): one radius/flux update per round against the round-start radius (SURVEY Q1 "U2", the rule that
                                 * shards over GPUs); 0: the reference's own rule, main.cpp:119-122 — every accepted photon shrinks the radius at
                                 * once and later photons are tested against the shrunk radius ("U1"; one GPU, fp64 accumulators) */
    double alpha;               /* main.cpp:36 */
    double focus_plane;         /* main.cpp:178 */
    double lens_radius;         /* main.cpp:179 */
    double lightorg[3];         /* main.cpp:180 */
    double camorg[3];           /* main.cpp:181 */
    uint64_t seed;              /* Philox key (replaces srand(time), main.cpp:229,269) */
} cgrt_config;

typedef struct cgrt_counters {
    uint64_t eye_segments, photon_segments; /* trace() calls that reached the closest-hit loop, main.cpp:50 */
    uint64_t diffuse_hits;                  /* photon hits on diffuse surfaces, main.cpp:101 */
    uint64_t candidates, deposits;          /* hitpoints scanned / accepted in the 27-cell gather, main.cpp:114-116 */
    uint64_t node_visits, tri_tests;        /* only filled by cgrt_count_traversal (a counting build of the same traversal) */
    uint64_t hitpoints;                     /* "hitpoints: %d", main.cpp:265 */
    uint64_t gpu_launches;                  /* kernels launched by this ctx so far */
    uint64_t gathered_hits;                 /* diffuse hits that went through the 27-cell gather (= diffuse_hits unless culling is on) */
    uint64_t exact_tests;                   /* (hit, hitpoint) pairs that passed the fp32 prefilter and took the fp64 test of main.cpp:116 */
    uint64_t cell_groups;                   /* deposit kernel: groups of hits in one cell that shared one reading of the 27 bucket lists */
    uint64_t staged_candidates;             /* bucket entries read for those groups (each once per group, not once per hit) */
} cgrt_counters;

/* ---- lifecycle ------------------------------------------------------------------------------------------------ */
int cgrt_create(int device, cgrt_ctx **out);
int cgrt_destroy(cgrt_ctx *ctx);
const char *cgrt_last_error(const cgrt_ctx *ctx); /* never NULL */
int cgrt_version(void);
void cgrt_default_config(cgrt_config *cfg);       /* the reference's literals */
int cgrt_set_config(cgrt_ctx *ctx, const cgrt_config *cfg);
/* The CUDA stream (cudaStream_t as void*) all kernels of this ctx are launched on; time with events on THIS stream. */
int cgrt_get_stream(cgrt_ctx *ctx, void **stream);
int cgrt_synchronize(cgrt_ctx *ctx);

/* ---- scene: same argument meaning as the reference constructors; object ids are insertion order (main.cpp:355-378) */
/* Texture(data,n,p,lx,ly,flag) texture.h:19 with data[i][j] = rgb8/256 (main.cpp:303-316). rgb is h*w*3 bytes. */
int cgrt_add_texture(cgrt_ctx *ctx, const uint8_t *rgb, int w, int h, const double n[3], const double p[3], double lenx,
                     double leny, int isbump, int *tex_id);
/* Sphere(c,r,sc,refl,transp) objects.h:28-38 */
int cgrt_add_sphere(cgrt_ctx *ctx, const double c[3], double r, const double col[3], double refl, double transp, int *obj_id);
/* Plane(p,n,sc,refl,transp,tx) objects.h:480; tex_id < 0: untextured. A bump texture on an n=(0,1,0) plane builds the
 * displaced height-field mesh of objects.h:482-503 on the device. */
int cgrt_add_plane(cgrt_ctx *ctx, const double p[3], const double n[3], const double col[3], double refl, double transp,
                   int tex_id, int *obj_id);
/* TriangleMesh(...) objects.h:338-403 after loading: tri9 = ntri x (pa,pb,pc) world-space fp64; objtype = typeofdata. */
int cgrt_add_mesh(cgrt_ctx *ctx, const double *tri9, int ntri, const double col[3], double refl, double transp, int objtype,
                  int *obj_id);
/* Bezier(points,pos,sc,refl,transp) bezier.h:44-45; ncp <= 7. */
int cgrt_add_bezier(cgrt_ctx *ctx, const double *cp3, int ncp, const double pos[3], const double col[3], double refl,
                    double transp, int *obj_id);
/* Uploads, builds every LBVH (Morton codes -> radix sort -> Karras hierarchy -> refit) and freezes the scene. */
int cgrt_commit_scene(cgrt_ctx *ctx);

/* ---- parity hooks ---------------------------------------------------------------------------------------------- */
/* Closest hit of main.cpp:50-76 for n rays: t, face-forwarded normal, object id (-1 miss), into flag, primitive id
 * (original triangle index for meshes / height-fields, else -1). Any output may be NULL. */
int cgrt_intersect_batch(cgrt_ctx *ctx, int64_t n, const double *org, const double *dir, double *t, double *nrm,
                         double *nrm_raw, int32_t *obj, int32_t *into, int32_t *prim);
/* Hashtable ctor + compute_coord + hash (hash.h:22-42) for n positions: key[n], ixyz[3n] (either may be NULL). */
int cgrt_hash_keys(cgrt_ctx *ctx, int64_t n, const double *pos, int hashsize, double celllength_in, uint32_t *key,
                   int32_t *ixyz);
/* getSurfaceColor (objects.h:533-539 / texture.h:39-72) of object obj at n points. */
int cgrt_surface_color(cgrt_ctx *ctx, int obj, int64_t n, const double *pos, double *col);
/* Triangles of object obj's BVH in original order (mesh: as given; bump plane: objects.h:485-499). tri9 NULL: count only. */
int cgrt_object_triangles(cgrt_ctx *ctx, int obj, double *tri9, int64_t cap, int64_t *ntri);
/* The Philox sampling definitions: what = 0 sphere, 1 hemisphere about aux, 2 lens disc radius aux[0], 3 three U(0,1). */
int cgrt_sample(cgrt_ctx *ctx, uint64_t seed, uint32_t pass, uint64_t path, uint32_t dim, int what, const double aux[3],
                double out[3]);
/* Hand-written LSD radix sort (the one used for Morton codes and hitpoint keys): sorts key[n] (bits [0,nbits)) stably and
 * returns the permutation. */
int cgrt_radix_sort(cgrt_ctx *ctx, int64_t n, const uint64_t *key_in, int nbits, uint64_t *key_out, uint32_t *perm);
/* Counting build of the traversal kernel over n rays: fills counters.node_visits / tri_tests (roofline accounting). */
int cgrt_count_traversal(cgrt_ctx *ctx, int64_t n, const double *org, const double *dir, uint64_t *node_visits,
                         uint64_t *tri_tests);

/* ---- passes ---------------------------------------------------------------------------------------------------- */
/* Eye pass (main.cpp:183-219) over image rows [y0,y1) as an iterative wavefront; appends hitpoints. */
int cgrt_eye_pass(cgrt_ctx *ctx, int y0, int y1);
/* Tile-sharded eye pass: export this rank's unsorted hitpoint records / import the union (all-gather in between).
 * Records are CGRT_HP_RECORD_DOUBLES doubles each. The import refuses the whole set (CGRT_ERR_INVALID, the current set kept) when a
 * record's bucket key is >= hashsize or is not the cell key of its position, or when its pixel lies outside the image. */
#define CGRT_HP_RECORD_DOUBLES 12
int cgrt_export_hitpoints_dev(cgrt_ctx *ctx, void **records_dev, int64_t *count);
int cgrt_import_hitpoints_dev(cgrt_ctx *ctx, const void *records_dev, int64_t count);
/* hash.h:43-54 + main.cpp:98 as a sort-based grid: keys -> radix sort on (key, creation order) -> cell-start table. */
int cgrt_build_grid(cgrt_ctx *ctx);
/* Photons with global indices [first, first+count) (main.cpp:231-247): emit, bounce, deposit into the per-round
 * accumulators. Index k always draws the same Philox stream, whichever GPU traces it. */
int cgrt_photon_pass(cgrt_ctx *ctx, uint64_t first, uint64_t count);
/* trace() itself (main.cpp:42) for n caller-made rays: org, dir, weight are n x 3 host doubles; depth is the recursion depth the rays start at.
 * flag != 0, an eye ray (main.cpp:209): weight = adj, (x[i], y[i]) = the pixel (column, row) its hitpoints belong to; hitpoints are appended
 *   exactly as cgrt_eye_pass appends them (call before cgrt_build_grid; rays of one call that share a pixel take sample numbers k mod samples).
 * flag == 0, a photon (main.cpp:246): weight = flux; its diffuse hits deposit into the per-round accumulators like cgrt_photon_pass's (call
 *   after cgrt_build_grid; x, y unused). Ray k draws the random numbers of photon index first_index + k (bounce = depth onwards). */
int cgrt_trace(cgrt_ctx *ctx, int64_t n, const double *org, const double *dir, const double *weight, int flag, int depth,
               const int32_t *x, const int32_t *y, uint64_t first_index);
/* Device view of the per-round accumulators {dflux[3], m} (4 lanes per hitpoint, canonical order) for the all-reduce: fp64 (accum_mode
 * 0), float (1) or int64 fixed point {sum q[3], M} (2). */
int cgrt_accum_dev(cgrt_ctx *ctx, void **ptr_dev, int64_t *n_doubles);
/* ---- multi-GPU (SURVEY section 8e): NCCL is bound at run time (the copy already loaded in the process, else libnccl.so.2); none of
 * these is needed on one GPU. A communicator is an ncclComm_t passed as void*. ------------------------------------------------ */
/* Communicators without nccl.h on the host side: a 128-byte ncclUniqueId made on rank 0 and carried to the others by whatever the
 * launcher offers (one process per GPU), or all devices of one process at once (one thread per ctx). */
int cgrt_comm_unique_id(void *id128);
int cgrt_comm_init_rank(int device, int rank, int world, const void *id128, void **comm);
int cgrt_comm_init_all(int n, const int *devices /* NULL: 0..n-1 */, void **comms /* n */);
int cgrt_comm_destroy(void *comm);
/* Tile-sharded eye pass: all-gather the hitpoint records of every rank's rows (after cgrt_eye_pass(y0,y1), before cgrt_build_grid;
 * under SPPM after cgrt_sppm_eye_pass); every rank then builds the same grid from the union. */
int cgrt_allgather_hitpoints(cgrt_ctx *ctx, void *nccl_comm, int world);
/* Attach a communicator: from now on cgrt_round_update all-reduces the accumulators {dflux.xyz, m} over it, in stream order, before
 * applying the update (under SPPM: before the per-pixel fold; attach it before cgrt_set_sppm). In stream order: on a side stream under
 * the next round's trace launches it measured slower on 8 GPUs (NCCL's blocks do not fit next to the persistent trace kernels). NULL detaches. */
int cgrt_set_comm(cgrt_ctx *ctx, void *nccl_comm, int world);
/* The same exchange without a collective call, over peer memory (GPUs of one box, NVLink / NVSwitch): every rank's accumulators live in a
 * block all ranks have mapped; cgrt_round_update publishes "round deposited" flags and ONE kernel on a side stream reads every rank's
 * accumulators out of their memory, applies the update and clears the next round's buffer (double-buffered by round parity). Only the
 * next round's deposit kernel waits for it: the next round's trace runs underneath, and the skew between ranks is absorbed instead of
 * being paid every round. After cgrt_build_grid on every rank: export one 128-byte handle per rank, carry all of them to every rank
 * (the launcher's job: torch.distributed, MPI, or shared memory between the threads of one process), attach. Ranks may be processes
 * (CUDA IPC) or contexts of one process (peer access). A rank that does not arrive within 20 s raises an error on the others at the
 * next cgrt_synchronize instead of hanging them; cgrt_destroy waits for the peers' last reads before it frees the block. */
#define CGRT_PEER_HANDLE_BYTES 128
int cgrt_peer_export(cgrt_ctx *ctx, void *handle128);
int cgrt_peer_attach(cgrt_ctx *ctx, int rank, int world, const void *handles /* world x CGRT_PEER_HANDLE_BYTES, rank order */);
/* All-reduce the accumulators now, on the ctx stream, asynchronously (NULL: single GPU, no-op). For hosts that drive the collective
 * themselves; with cgrt_set_comm it is implied by cgrt_round_update. */
int cgrt_allreduce_accum(cgrt_ctx *ctx, void *nccl_comm);
/* Per-round radius/flux update (main.cpp:119-122 in its batched form, SURVEY Q1 "U2"), then clears the accumulators. */
int cgrt_round_update(cgrt_ctx *ctx);
/* main.cpp:252-258 (+ :403-411 when rgb8 != NULL: tone map, gamma, vertical flip). rgb: H*W*3 fp64, row h = image[h].
 * n_emitted = photons traced so far, the reference's num_photon*num_threads; the third factor of main.cpp:256, num_of_samples, is taken
 * from cgrt_config, so that every caller normalises a multi-sample image the same way. */
int cgrt_gather_image(cgrt_ctx *ctx, double n_emitted, double *rgb, uint8_t *rgb8);

/* ---- stochastic progressive photon mapping (SPPM, Hachisuka & Jensen 2009) ------------------------------------------
 * Every round traces a new eye pass; the statistics (accepted photons n, radius R2, flux tau) live per pixel, shared by all the
 * visible points one pixel's eye paths create in a round. Round r of eye path (pixel * samples + s) draws its camera from the Philox
 * stream (seed, pass 3, path, dim = r): jitter ux, uy in [0,1)^2 (JITTER only), then the lens sample when use_dof is set; the ray goes
 * through the image-plane point of main.cpp:188-198 with (w + ux, h + uy) in place of (w, h). Per-round update (update_mode 1) only.
 *
 * One GPU, per round: cgrt_sppm_begin_round(r) -> cgrt_photon_pass -> cgrt_round_update (folds the round's accumulators into the pixels).
 * Several GPUs (one ctx per GPU; a row tile of the eye pass and a photon index range per rank):
 *   cgrt_set_comm (optional) -> cgrt_set_sppm ->
 *   per round: cgrt_sppm_eye_pass(r, y0, y1) -> cgrt_allgather_hitpoints -> cgrt_build_grid
 *              -> cgrt_photon_pass(this rank's range) -> cgrt_round_update
 * Every rank builds the same grid from the same sorted union, so the visible-point accumulators line up across ranks: with a
 * communicator attached cgrt_round_update all-reduces them before the fold, and every rank holds the same pixel statistics. A host that
 * drives its own collectives imports the union with cgrt_import_hitpoints_dev (instead of cgrt_allgather_hitpoints) and reduces
 * cgrt_accum_dev itself (or with cgrt_allreduce_accum) before cgrt_round_update. The record exchange is accepted only between
 * cgrt_sppm_eye_pass and cgrt_build_grid; the peer-memory exchange (cgrt_peer_*) is refused under SPPM: its block is sized for a
 * fixed hitpoint count, and the visible-point count changes every round.
 * cgrt_gather_image then reads the pixels: tau / (pi R2 n_emitted num_of_samples). cgrt_download_hitpoints / cgrt_download_accum
 * return the current round's visible points (their r2 is the pixel radius the round used). */
#define CGRT_SPPM_OFF 0    /* default: PPM, one eye pass for the whole render */
#define CGRT_SPPM_JITTER 1 /* camera ray through a uniformly jittered point of the pixel, new every round */
#define CGRT_SPPM_CORNER 2 /* through the pixel corner as main.cpp:188-198; only the lens sample (use_dof) changes per round */
/* After cgrt_commit_scene (and cgrt_set_comm, if any), before any eye pass or grid. Allocates the W*H pixel statistics: n = 0, tau = 0,
 * R2 = (200/height)^2. */
int cgrt_set_sppm(cgrt_ctx *ctx, int mode);
/* Waits for the previous round's work, drops its visible points and grid, and traces the eye pass of `round` over rows [y0, y1)
 * (y1 < 0: all rows; y0 == y1: none) into a new visible-point set. The grid is not built: cgrt_build_grid builds it, with every visible
 * point at its pixel's current radius, after the records have been exchanged. */
int cgrt_sppm_eye_pass(cgrt_ctx *ctx, uint32_t round, int y0, int y1);
/* cgrt_sppm_eye_pass(round, 0, -1) followed by cgrt_build_grid: the one-call round of one GPU. */
int cgrt_sppm_begin_round(cgrt_ctx *ctx, uint32_t round);
/* Pixel statistics, row h = image[h]: tau H*W*3, r2 H*W, n H*W (any may be NULL). */
int cgrt_sppm_download_pixels(cgrt_ctx *ctx, double *tau, double *r2, int32_t *n);

/* ---- multi-run averaging (average.cpp:19-65), the reference's way of combining separately rendered images ------------ */
/* Bit-exact 8-bit mode: out[i] = sum over the n images of (img_k[i] / n) in integer arithmetic, exactly what average.cpp does with
 * n = 9 (truncating division before the sum; never overflows a byte). imgs: n host pointers to nbytes bytes each. */
int cgrt_average_u8(cgrt_ctx *ctx, int n, const uint8_t *const *imgs, int64_t nbytes, uint8_t *out);
/* Linear mode: mean of n fp64 radiance images (what cgrt_gather_image returns), optionally tone-mapped like main.cpp:403-411
 * into rgb8 (no vertical flip: the inputs are image[h][w] arrays, the output keeps their row order). rgb8 may be NULL. */
int cgrt_average_f64(cgrt_ctx *ctx, int n, const double *const *imgs, int64_t nvalues, double *mean, uint8_t *rgb8);

/* ---- downloads (canonical order: bucket ascending, creation order inside a bucket; main.cpp:252-254) ------------- */
int cgrt_num_hitpoints(cgrt_ctx *ctx, int64_t *n);
int cgrt_download_hitpoints(cgrt_ctx *ctx, double *pos, double *normal, double *f, double *flux, double *r2, int32_t *n,
                            int32_t *hw, uint32_t *key, uint32_t *seq);
/* The round's accumulators as the update reads them; accum_mode 2: sum q * 2^-22 and M. */
int cgrt_download_accum(cgrt_ctx *ctx, double *dflux, double *m);
int cgrt_download_grid(cgrt_ctx *ctx, uint32_t *cell_start /* hashsize+1 */);
int cgrt_get_counters(cgrt_ctx *ctx, cgrt_counters *out);
/* on != 0: the photon trace kernels run their counting build (same traversal + node-visit / triangle-test counters,
 * reported by cgrt_get_counters). Used outside timed regions to derive the algorithmic bytes of the roofline. */
int cgrt_set_counting(cgrt_ctx *ctx, int on);
/* on != 0: cgrt_photon_pass traces on a second internal stream into double-buffered deposit tables, so the trace of one chunk (or
 * of the next round) overlaps the sort + deposit of the previous one. Everything a caller can observe stays ordered on the stream
 * cgrt_get_stream returns. Off by default. With the r02 kernels on one B200 at 1000 W it is 1.2-3.3 % faster per round on c1-c4
 * (c3: 17.07 vs 17.33 ms, DESIGN.md section 4); the earlier 25.3 vs 24.2 ms against it predates those kernels. */
int cgrt_set_overlap(cgrt_ctx *ctx, int on);
/* on != 0 (default): photon hits whose cell is farther than 2 cells from every hitpoint are dropped before the gather — they
 * cannot pass the distance test of main.cpp:116 — and are not counted in counters.candidates. Deposits, accepted-photon
 * counts and images are identical either way; 0 makes counters.candidates equal the reference's scan count. */
int cgrt_set_culling(cgrt_ctx *ctx, int on);
/* on != 0: every photon kernel launch is bracketed by CUDA events on the ctx stream and cgrt_photon_pass ends with a
 * synchronise (per-kernel durations for the roofline). Off (default): cgrt_photon_pass is asynchronous. */
int cgrt_set_profiling(cgrt_ctx *ctx, int on);
/* Accumulated device time per phase on the ctx stream (CUDA events), milliseconds: [0] eye, [1] grid, [2] all photon trace launches,
 * [3] photon_deposit_kernel, [4] round update, [5] image gather, [6] deposit counting sort, and the split of [2]:
 * [9] photon_trace_kernel<emission>, [7] photon_traverse_kernel launches, [8] photon_trace_kernel<continuation> launches,
 * [10] cgrt_allgather_hitpoints (count exchange, record all-gather, unpacking). [4] includes the all-reduce of an attached communicator.
 * [2]-[4],[6]-[9] are only filled while profiling is on. */
int cgrt_get_timings(cgrt_ctx *ctx, double ms[12]);
/* Debug aid (the reference has none; it stands in for a memory checker): when the process runs with CGRT_GUARD=1 in its
 * environment every device buffer of a context sits between two 4 KiB fences of a known byte pattern. Synchronises and returns in
 * *damaged the number of fence bytes kernels have overwritten so far (released buffers included); 0 when the mode is off. */
int cgrt_check_guards(cgrt_ctx *ctx, uint64_t *damaged);
/* Photons one trace launch of cgrt_photon_pass takes (sized from free device memory at the first pass; 0 before it). */
int cgrt_photon_chunk(cgrt_ctx *ctx, uint64_t *photons_per_launch);
/* Bytes of one slot of the deposit table (record written per recorded photon hit, read once by the gather) under the context's
 * configuration — 64 with float or fixed-point accumulators, 96 with fp64 ones (NULL: 96): the unit of the measurement's compulsory-traffic accounting. */
int cgrt_deposit_record_bytes(const cgrt_ctx *ctx);
/* The library keeps the large device buffers of destroyed contexts (deposit tables, photon queues, ray queues) parked per device and
 * hands them to the next context: a render() creates and destroys one. Parked blocks are released automatically when an allocation
 * would otherwise fail; this call releases them now (device < 0: all devices). bytes_released may be NULL. */
int cgrt_release_cached_memory(int device, uint64_t *bytes_released);

#ifdef __cplusplus
}
#endif
#endif /* CGRT_H_ */
