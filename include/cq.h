/*
 * cq.h — C ABI of the B200 batched collision-query engine (libcq.so).
 *
 * This is the drop-in boundary for ONE path of kelian343/swift-game-engine:
 * the capsule CCD sweep / move-and-slide / raycast queries of
 * Game/CollisionQuery.swift against static triangle meshes (*.static.json).
 * The reference has no FFI of its own — the boundary there is the in-process
 * Swift class `CollisionQuery` (Game/CollisionQuery.swift:54-160).  Every entry
 * point below names the reference interface it replaces.
 *
 * Conventions
 *  - plain pointers + sizes, no C++/torch types; the library copies what it
 *    needs, callers keep ownership of every array they pass in;
 *  - return value: 0 = CQ_OK, negative = error (cq_last_error() has the text);
 *    nothing throws across the ABI.  The reference's "nil" (no hit) is
 *    triangle_index == -1 in the hit record;
 *  - a cq_world lives on the CUDA device that was current when it was created;
 *    one host thread at a time per world (the reference is MainActor-only and
 *    not re-entrant, CollisionQuery.swift:787-828);
 *  - triangle_index numbering = position in the degenerate-filtered soup, static
 *    set first, dynamic set offset by the static count
 *    (CollisionQuery.swift:776,782,1004);
 *  - there is NO CPU fallback: every call fails with CQ_ERR_CUDA when no device
 *    is usable.
 */
#ifndef CQ_H
#define CQ_H

#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CQ_OK 0
#define CQ_ERR_INVALID (-1)   /* bad argument */
#define CQ_ERR_CUDA (-2)      /* CUDA runtime error / no device */
#define CQ_ERR_IO (-3)        /* file missing / unreadable */
#define CQ_ERR_PARSE (-4)     /* malformed *.static.json */
#define CQ_ERR_NOT_FOUND (-5) /* unknown entity id */
#define CQ_ERR_NCCL (-6)      /* NCCL missing or failed (multi-GPU groups only) */

#define CQ_LAYER_ALL 0xFFFFFFFFu /* CollisionLayer.all, Components.swift:47-50 */
/* capsuleOverlapAll's default maxHits (CollisionQuery.swift:151) and the maxHits of move-and-slide's depenetration
 * (Systems.swift:751-767).  It is not a limit of cq_capsule_overlap_all_*: max_hits up to 8 runs a kernel that keeps
 * the hits in shared memory, larger values run the wide path (see cq_capsule_overlap_all_batch). */
#define CQ_MAX_OVERLAP_HITS 8
/* Device scratch bound of cq_capsule_overlap_all_batch: it runs in query chunks whose records fit 256 MiB. */
#define CQ_OVERLAP_ALL_CHUNK_BYTES ((size_t)256 << 20)
#define CQ_MANIFOLD_MAX 4        /* ContactManifoldCache.maxCount, Systems.swift:1160 */

typedef struct cq_world cq_world;
typedef struct cq_static_mesh_asset cq_static_mesh_asset;

/* ---- world construction ------------------------------------------------- */

/* One collidable entity = TransformComponent + StaticMeshComponent
 * (+ optional PhysicsBodyComponent.bodyType), as TriangleMeshSet.rebuild reads
 * them (CollisionQuery.swift:331-417).  `model` is TransformComponent.modelMatrix
 * (Components.swift:26-44), column-major like simd's matrix_float4x4. */
typedef struct cq_mesh_part {
    const float *positions_xyz; /* n_verts * 3, local space */
    const uint32_t *indices;    /* n_indices (3 per triangle), u16 widened by the caller */
    int32_t n_verts;
    int32_t n_indices;
    float model[16];
    uint32_t layer;        /* StaticMeshComponent.collisionLayer */
    float mu_s, mu_k;      /* SurfaceMaterial, Components.swift:704-716 */
    uint8_t flatten_ground;
    uint8_t is_dynamic;    /* body present && bodyType != .static  (CollisionQuery.swift:886-900) */
    uint16_t _pad;
    uint32_t entity_id;
} cq_mesh_part;

typedef struct cq_world_info {
    int32_t n_static_triangles;  /* after the |e1 x e2|^2 <= 1e-10 filter */
    int32_t n_dynamic_triangles;
    int32_t n_static_vertices;
    int32_t n_dynamic_vertices;
    int32_t n_static_nodes;      /* LBVH internal nodes */
    int32_t n_dynamic_nodes;
    int32_t n_parts;
    int32_t device;
    float build_ms;              /* device time of upload+filter+Morton+sort+tree+fit */
    float refit_ms;              /* device time of the last cq_world_update_transforms (the async call leaves it unchanged) */
    int32_t order;               /* CQ_ORDER_* the world was created with */
    float ref_order_ms;          /* wall time of the reference-order build (0 in canonical order) */
    int32_t n_ref_nodes;         /* nodes of the reference's own tree, both sets (0 in canonical order) */
    int32_t _reserved;
} cq_world_info;

/* Which of several EXACTLY equal candidates a query names.
 *
 * The reference walks its median-split BVH depth-first, right child first, and keeps the first triangle it visits on
 * exactly equal keys: strict `<` on toi (CollisionQuery.swift:1084) and ray t (:944), strict `>` on depth (:1172);
 * capsuleOverlapAll returns the first maxHits overlaps it visits (:1272-1274).  About a third of random sweeps against a
 * closed mesh end on an edge or vertex shared by two triangles and tie bit-exactly, and the move-and-slide contact
 * cache is keyed by triangle index (Systems.swift:1169-1204), so the choice is visible.
 *
 *  CQ_ORDER_REFERENCE (default): the library derives every triangle's visiting rank from the reference's own tree
 *      (cut on the device at world creation: attach_ref_order in csrc/cq_build.cu) and resolves ties / keeps the
 *      first maxHits overlaps by that rank; raycasts walk that tree with the reference's own slab test, so even the
 *      grazing hits its non-conservative test culls (:933, :1603-1631) come out the same.  Results equal the reference's
 *      for the same entity order.  Costs a device build at creation (DESIGN.md §2.1), none per query.
 *  CQ_ORDER_CANONICAL: tree-independent rule — ties go to the smallest triangle index, capsuleOverlapAll keeps the
 *      maxHits deepest (deepest first), a raycast returns the nearest triangle over ALL triangles.  No reference tree. */
#define CQ_ORDER_REFERENCE 0
#define CQ_ORDER_CANONICAL 1

/* StaticMeshComponent.triangleMaterials (Components.swift:323-351): surface materials per triangle of one part.  As in
 * TriangleMeshSet.rebuild (CollisionQuery.swift:363-369) the array is used only when `n` equals the part's triangle count
 * (n_indices / 3, before the degenerate filter) and silently ignored otherwise; triangles the filter drops take their
 * entry with them.  The arrays are copied by cq_world_create_ex. */
typedef struct cq_surface_material { /* SurfaceMaterial, Components.swift:704-716 */
    float mu_s, mu_k;
    uint8_t flatten_ground;
    uint8_t _pad[3];
} cq_surface_material; /* 12 bytes */
typedef struct cq_triangle_materials {
    uint32_t entity_id; /* the part (cq_mesh_part.entity_id) */
    int32_t n;
    const cq_surface_material *materials;
} cq_triangle_materials;

typedef struct cq_world_options {
    int32_t order;                                   /* CQ_ORDER_* */
    int32_t n_triangle_materials;                    /* entries of triangle_materials (0: every part uses its own material) */
    const cq_triangle_materials *triangle_materials; /* per-triangle materials of some parts, or NULL */
    int32_t _reserved[4];                            /* zero */
} cq_world_options; /* 32 bytes, as before the two fields were carved out of the reserved words */
void cq_world_options_default(cq_world_options *o);

/* Replaces CollisionQuery.init(world:activeEntityIDs:) (CollisionQuery.swift:57-59
 * -> StaticTriMesh.init :717-726).  Parts are taken in the given order (the
 * oracle fixes entity order = ascending id; the reference iterates a Dictionary).
 * A triangle set holds at most 2^26 (67,108,864) triangles after the degenerate filter.
 * cq_world_create = cq_world_create_ex with default options. */
int cq_world_create(const cq_mesh_part *parts, int32_t n_parts, cq_world **out);
int cq_world_create_ex(const cq_mesh_part *parts, int32_t n_parts, const cq_world_options *options, cq_world **out);
void cq_world_destroy(cq_world *w);
int cq_world_get_info(const cq_world *w, cq_world_info *info);

/* Replaces updateStaticTransforms / updateDynamicTransforms
 * (CollisionQuery.swift:69-83 -> TriangleMeshSet.updateTransforms :419-462 ->
 * BVH.refit :528-575): re-transform the entities' vertices, recompute triangle
 * bounds (no degenerate re-filter), refit the BVH.  models = n * 16 floats. */
int cq_world_update_transforms(cq_world *w, const uint32_t *entity_ids,
                               const float *models, int32_t n);

/* Stream-ordered twin of cq_world_update_transforms.  entity_ids / models are HOST arrays (n, n*16 floats, column-major
 * like cq_mesh_part.model); they are copied before the call returns, so the caller may reuse them at once.  stream: a
 * cudaStream_t cast to void*, NULL = the world's own stream.  Nothing is synchronised.
 *
 * Same semantics as the synchronous call: every id is checked before anything is queued (an unknown id returns
 * CQ_ERR_NOT_FOUND and queues nothing); n == 0 is a no-op; n < 0, or a NULL array with n > 0, returns CQ_ERR_INVALID;
 * every part with a matching entity_id takes the model, parts that contributed no triangle are skipped
 * (CollisionQuery.swift:427), and an id named twice takes its last model.  A set is refitted in full when at least a
 * quarter of its triangles moved (or CQ_REFIT_FULL is set in the environment), else only the moved leaves' ancestors;
 * either way a fixed number of kernel launches per set (at most 8) plus one host-to-device copy, however many parts moved.
 * refit_ms is left unchanged.
 *
 * Ordering contract (all three update calls: this one, cq_world_update_transforms and
 * cq_world_update_transforms_device; uncaptured):
 *  - the refit starts only after every launch already queued on this world, on any stream, has finished reading the
 *    trees: queries, crowd steps, agent separation and earlier refits alike;
 *  - every call made on the world after this one returns sees the new trees, whatever its stream: the *_device twins,
 *    the host-pointer batches, cq_crowd_step, agent separation, cq_world_read_soup and cq_world_read_counters.
 *
 * Back-pressure: the id -> part table is staged in one of 4 pinned slots of the world; a slot is reused once its copy has
 * completed.  When all 4 are still in flight the call waits on the host for the oldest copy, so at most 4 table
 * copies are queued at once.  A call that stages more parts than any call before it allocates larger staging buffers (pinned host and
 * device memory); cq_world_destroy frees them. */
int cq_world_update_transforms_async(cq_world *w, const uint32_t *entity_ids, const float *models, int32_t n, void *stream);

/* Device-resident twin: d_entity_ids (n ids) and d_models (n*16 floats, column-major like cq_mesh_part.model) are DEVICE
 * pointers, read by the kernels the call queues on `stream` (NULL = the world's stream), so the caller keeps them
 * unchanged until the stream has passed the call.  The call does not synchronise, allocate or touch host memory: the ids
 * are resolved and the table of moved parts is built on the device, from an index the world uploads at creation.
 *
 * Same semantics as the other two calls (every part with a matching entity_id takes the model, parts without triangles
 * are skipped, an id named twice takes the model of its last position, a set is refitted in full when at least a quarter
 * of its triangles moved or CQ_REFIT_FULL is set, refit_ms is left unchanged) and the same ordering contract.  Errors are
 * all-or-nothing and decided on the device: when any id is unknown the update changes nothing (no model row, vertex or
 * box is written), and *d_status (a device int32, may be NULL) receives the number of unknown ids, 0 on success, in
 * stream order.  NULL world, n < 0, or a NULL array with n > 0 return CQ_ERR_INVALID before any CUDA call; n == 0 returns
 * CQ_OK and queues nothing.
 *
 * Launches: a fixed number per call whatever n is and whatever moved: 2 (resolve the ids, build the table) plus, for
 * each set that has triangles, 13 (the part update, the 5 kernels of the full refit and the 7 of the dirty one, of which
 * the path not chosen exits at once): at most 28.  Fewer in canonical order (no reference tree: 4 fewer per set) and for
 * a set of one triangle (1 fewer).  The kernels of both paths stride over their work with grids of at most one resident
 * wave, so the unchosen path and an untouched set cost a few empty CTAs per SM, whatever the set's size.
 *
 * Stream capture: the call, and every *_device query twin below, may be recorded into a CUDA graph (see the capture
 * contract below the *_device twins). */
int cq_world_update_transforms_device(cq_world *w, const uint32_t *d_entity_ids, const float *d_models, int32_t n,
                                      int32_t *d_status, void *stream);

/* Read back the world-space soup (testing / material lookup on the host).
 * which: 0 = static set, 1 = dynamic set.  Any out pointer may be NULL. */
int cq_world_read_soup(const cq_world *w, int32_t which,
                       float *positions_xyz /* n_vertices*3 */,
                       uint32_t *indices /* n_triangles*3 */,
                       float *tri_aabbs /* n_triangles*6: min xyz, max xyz */,
                       uint32_t *tri_layers /* n_triangles */,
                       int32_t *tri_parts /* n_triangles: index into the parts array */);

/* Rebuild the world in place from a new parts array: afterwards every query, move-and-slide, separation, read and device
 * update answers exactly as a fresh cq_world_create_ex(parts, n_parts, options) would (the entity index of the device
 * updates included).  The new geometry is built aside and swapped in only on success: on any error (bad arguments, an
 * index out of range, a reference tree too deep, a CUDA error) the world keeps answering exactly as before, and
 * cq_last_error says why.  Before the swap it waits for every launch already queued on the world, on any stream, that may
 * read the old geometry (those launches see the old geometry), then releases it.  The device, streams, events, pinned
 * staging and launch scratch are kept.  Crowds created on the world stay valid with their records unchanged; triangle
 * indices already in them (contact caches) keep the old numbering, as the reference's controllers keep theirs across a
 * rebuild.  CUDA graphs recorded before a rebuild hold the old geometry's addresses and must not be replayed after it.
 * Synchronous: refused (CQ_ERR_INVALID, nothing enqueued) while the world's stream or a stream that launched work on the
 * world is being captured. */
int cq_world_rebuild(cq_world *w, const cq_mesh_part *parts, int32_t n_parts, const cq_world_options *options);

/* The reference's own tree of one set (which: 0 = static, 1 = dynamic), as the world built it on the device at creation:
 * order[p] = the set-local triangle at position p of the reference's triOrder, rank[t] = the position of set-local
 * triangle t in the reference's depth-first visiting order (0 = visited first).  Exact ties and capsuleOverlapAll's
 * maxHits cut follow this rank.  Either pointer may be NULL; each takes n_triangles of the set.  CQ_ERR_INVALID in
 * canonical order.  Not capturable. */
int cq_world_read_ref_order(const cq_world *w, int32_t which, int32_t *order, int32_t *rank);

/* The model matrix of every part (n_parts * 16 floats, column-major, in the order of the parts array given to
 * cq_world_create), as the last completed update left it.  Waits for queued updates like cq_world_read_soup. */
int cq_world_read_models(const cq_world *w, float *models_out);

typedef struct cq_material {
    float mu_s, mu_k;
    int32_t flatten_ground;
} cq_material;
/* TriangleMeshSet.materialForTriangle (CollisionQuery.swift:464-469); index is
 * the global triangle_index of a hit; out-of-range gives SurfaceMaterial.default. */
int cq_world_triangle_material(const cq_world *w, int32_t triangle_index, cq_material *out);

/* ---- static-mesh JSON loader ---------------------------------------------
 * Replaces StaticMeshLoader.loadStaticMeshAsset(named:) (StaticMeshLoader.swift:30-125).
 * Schema: StaticMeshLoader.swift:168-197.  Returns CQ_ERR_IO / CQ_ERR_PARSE where
 * the reference returns nil; invalid parts are skipped like the reference does. */
int cq_static_mesh_load(const char *path, cq_static_mesh_asset **out);
void cq_static_mesh_free(cq_static_mesh_asset *a);
int32_t cq_static_mesh_part_count(const cq_static_mesh_asset *a);
const char *cq_static_mesh_part_name(const cq_static_mesh_asset *a, int32_t part);
/* part transform, already converted row-major -> column-major (StaticMeshLoader.swift:127-134) */
int cq_static_mesh_part_transform(const cq_static_mesh_asset *a, int32_t part, float out_colmajor[16]);
/* hull = -1: the render mesh; hull >= 0: collisionHulls[hull].  Pointers stay valid until free. */
int32_t cq_static_mesh_hull_count(const cq_static_mesh_asset *a, int32_t part);
int cq_static_mesh_geometry(const cq_static_mesh_asset *a, int32_t part, int32_t hull,
                            const float **positions_xyz, int32_t *n_verts,
                            const uint32_t **indices, int32_t *n_indices);

/* ---- queries ------------------------------------------------------------- */

typedef struct cq_ray { /* raycast(origin:direction:maxDistance:mask:), CollisionQuery.swift:85 */
    float origin[3];
    float direction[3]; /* NOT normalised by the callee; maxDistance is in units of |direction| */
    float max_distance;
    uint32_t mask;
} cq_ray;

typedef struct cq_ray_hit { /* RaycastHit, CollisionQuery.swift:28-34 */
    float distance;
    float position[3];
    float normal[3];
    int32_t triangle_index; /* -1 = nil */
} cq_ray_hit;

#define CQ_CAST_ALL 0      /* capsuleCast          CollisionQuery.swift:96  */
#define CQ_CAST_BLOCKING 1 /* capsuleCastBlocking  CollisionQuery.swift:109 */
#define CQ_CAST_GROUND 2   /* capsuleCastGround    CollisionQuery.swift:122 */

typedef struct cq_capsule_cast { /* capsule axis is world +Y, `from` is the centre (:1025-1027) */
    float from[3];
    float delta[3];
    float radius;
    float half_height;
    uint32_t mask;
    float min_normal_y; /* CQ_CAST_GROUND only */
} cq_capsule_cast;

typedef struct cq_cast_hit { /* CapsuleCastHit, CollisionQuery.swift:36-43 */
    float toi;
    float position[3]; /* closest point ON THE TRIANGLE at toi (:1342) */
    float normal[3];
    float triangle_normal[3];
    int32_t triangle_index; /* -1 = nil */
} cq_cast_hit;

typedef struct cq_capsule { /* capsuleOverlap / capsuleOverlapAll, CollisionQuery.swift:137,148 */
    float from[3];
    float radius;
    float half_height;
    uint32_t mask;
} cq_capsule;

typedef struct cq_overlap_hit { /* CapsuleOverlapHit, CollisionQuery.swift:45-52 */
    float depth;
    float position[3];
    float normal[3];
    float triangle_normal[3];
    int32_t triangle_index; /* -1 = nil */
} cq_overlap_hit;

/* Per-query flags of the *_ex calls (one byte per query, may be NULL).
 * CQ_HIT_TIE: another accepted candidate had exactly the winning toi / t / depth, i.e. the triangle named depends on the
 * world's order rule (the "degenerate edge / vertex ties" of a closed mesh).  CQ_HIT_OVERFLOW: more than max_hits
 * triangles overlapped (capsuleOverlapAll; the same information as its `overflow` array). */
#define CQ_HIT_TIE 1
#define CQ_HIT_OVERFLOW 2

/* Host-pointer, synchronous batch calls (H2D, kernel, D2H inside the call). */
int cq_raycast_batch(cq_world *w, const cq_ray *rays, int32_t n, cq_ray_hit *out);
int cq_raycast_batch_ex(cq_world *w, const cq_ray *rays, int32_t n, cq_ray_hit *out, uint8_t *flags);
int cq_capsule_cast_batch_ex(cq_world *w, const cq_capsule_cast *q, int32_t n, int32_t mode, cq_cast_hit *out,
                             uint8_t *flags);
int cq_capsule_overlap_batch_ex(cq_world *w, const cq_capsule *q, int32_t n, cq_overlap_hit *out, uint8_t *flags);
int cq_capsule_cast_batch(cq_world *w, const cq_capsule_cast *q, int32_t n, int32_t mode,
                          cq_cast_hit *out);
int cq_capsule_overlap_batch(cq_world *w, const cq_capsule *q, int32_t n, cq_overlap_hit *out);
/* out = n * max_hits records; counts[i] = hits written for query i; overflow[i] (may be NULL) = 1 when more than
 * max_hits triangles overlapped.  CQ_ORDER_REFERENCE: the first max_hits triangles the reference visits, in its
 * visiting order (:1272-1274; its callers sort by depth themselves, Systems.swift:759).  CQ_ORDER_CANONICAL: the
 * max_hits deepest, deepest first (ties: smaller triangle index).  Slots past counts[i] hold nil records.
 * Any max_hits is accepted; values below 1 become 1 (max(1, maxHits), CollisionQuery.swift:157).  The call fails with
 * CQ_ERR_INVALID, before any CUDA call, only when n * max_hits * sizeof(cq_overlap_hit) overflows size_t.
 * max_hits <= CQ_MAX_OVERLAP_HITS: one kernel launch.  Larger max_hits: the wide path, always three launches (the pair
 * pool keeps each query's winners as a heap in the query's own output slots, one thread per query sorts them, one thread
 * per slot writes the records); it needs no scratch beyond the smaller path's, so its device call is captured like it.
 * This host-pointer call runs in query chunks so that its record scratch stays within CQ_OVERLAP_ALL_CHUNK_BYTES (one
 * query whose records exceed that is a chunk of its own): one set of launches per chunk, identical results. */
int cq_capsule_overlap_all_batch(cq_world *w, const cq_capsule *q, int32_t n, int32_t max_hits,
                                 cq_overlap_hit *out, int32_t *counts, uint8_t *overflow);

/* Device-pointer twins: inputs/outputs already resident in HBM, enqueued on
 * `stream` (a cudaStream_t cast to void*; NULL = the world's own stream), no
 * synchronisation.  Same record layouts as above.  Calls on one world may be
 * enqueued on any number of streams (from one host thread at a time): the
 * world's scratch blocks are handed from stream to stream behind events, so up
 * to four launches overlap and further ones queue behind them.
 * cq_world_update_transforms and cq_world_destroy wait for everything in flight; cq_world_update_transforms_async is
 * ordered against them by events instead (see its ordering contract).
 *
 * CUDA-graph capture: while `stream` is being captured (cudaStreamBeginCapture, torch.cuda.graph, ...), the *_device
 * query twins, cq_move_and_slide_device(_ex) and cq_move_and_slide_device_platforms, cq_agent_snapshot_device and
 * cq_move_and_slide_device_agents, cq_world_update_transforms_device, cq_world_platforms_device and
 * cq_agent_separation_device_async enqueue kernels, memsets, copies and (agent
 * separation) conditional WHILE nodes only: they neither wait on nor record nor create world events.  So:
 *  - a graph is ordered only by the stream it is launched on; the caller orders its replays against other work on the
 *    world, as for a synchronous call (e.g. synchronise before an uncaptured call on another stream);
 *  - kernel_launches counts the launches once, at capture; replays are not counted;
 *  - scalar arguments (n, mode, params, flags, n_platforms, the environment's CQ_REFIT_FULL) are recorded with the graph,
 *    and so are the cq_platform records of the host-array calls (cq_move_and_slide_device_ex): a replay carries
 *    characters with the records of the capture.  Device buffers are read at replay, so new models written into the
 *    same buffer move the parts of each replay, and cq_world_platforms_device + cq_move_and_slide_device_platforms
 *    give every replay the records of its own frame;
 *  - a call that would grow scratch, allocate, synchronise or create an event while capturing returns CQ_ERR_INVALID
 *    ("make one uncaptured call of this size first") before it enqueues anything, and leaves the capture valid; so does
 *    CQ_MAS_AGENTS when its grid needs more scratch than an uncaptured call gave it;
 *  - scratch blocks a graph recorded stay allocated when a later uncaptured call outgrows them (the call takes new
 *    blocks), so graphs stay valid until cq_world_destroy, which frees them: replay no graph after destroying its world;
 *  - cq_world_rebuild replaces the geometry whose addresses a graph recorded: replay no graph recorded before a rebuild
 *    after it (record it again);
 *  - cq_agent_separation_device and cq_agent_separation_batch (they synchronise to report the outcome), cq_crowd_step
 *    and the host-pointer calls (checked on the world's stream, or on `stream` where they take one) refuse a capture the
 *    same way.
 * Uncaptured calls behave as described everywhere else in this header. */
int cq_raycast_device(cq_world *w, const cq_ray *d_rays, int32_t n, cq_ray_hit *d_out, void *stream);
int cq_capsule_cast_device(cq_world *w, const cq_capsule_cast *d_q, int32_t n, int32_t mode,
                           cq_cast_hit *d_out, void *stream);
int cq_capsule_overlap_device(cq_world *w, const cq_capsule *d_q, int32_t n, cq_overlap_hit *d_out,
                              void *stream);
int cq_capsule_overlap_all_device(cq_world *w, const cq_capsule *d_q, int32_t n, int32_t max_hits,
                                  cq_overlap_hit *d_out, int32_t *d_counts, uint8_t *d_overflow,
                                  void *stream);
/* with per-query flags (device pointer, n bytes, may be NULL) */
int cq_raycast_device_ex(cq_world *w, const cq_ray *d_rays, int32_t n, cq_ray_hit *d_out, uint8_t *d_flags, void *stream);
int cq_capsule_cast_device_ex(cq_world *w, const cq_capsule_cast *d_q, int32_t n, int32_t mode, cq_cast_hit *d_out,
                              uint8_t *d_flags, void *stream);
int cq_capsule_overlap_device_ex(cq_world *w, const cq_capsule *d_q, int32_t n, cq_overlap_hit *d_out, uint8_t *d_flags,
                                 void *stream);

/* ---- move-and-slide ------------------------------------------------------
 * One call = one fixed step of KinematicMoveStopSystem.fixedUpdate's per-entity
 * body (Systems.swift:1842-1901) for n characters.  Kinematic platforms: the *_ex
 * variants below; agent hits between the characters: CQ_MAS_AGENTS. */

typedef struct cq_controller_params { /* CharacterControllerComponent tunables, Components.swift:353-404 */
    float radius;               /* 1.5  */
    float half_height;          /* 1.0  */
    float skin_width;           /* 0.3  */
    float ground_snap_skin;     /* 0.05 */
    float snap_distance;        /* 0.8  */
    float fall_probe_distance;  /* 200  */
    float ground_snap_max_speed;/* 5    */
    float ground_snap_max_toi;  /* 0.1  */
    float ground_snap_max_step; /* 0.1  */
    float ground_sweep_max_step;/* 0.1  */
    int32_t max_slide_iterations; /* 4  */
    float min_ground_dot;       /* 0.5  */
    uint32_t collision_mask;    /* all  */
} cq_controller_params;

typedef struct cq_character_state { /* PhysicsBodyComponent + CharacterControllerComponent state */
    double position[3];          /* PhysicsBodyComponent.position (Double), Components.swift:551 */
    double velocity[3];          /* linearVelocity (Double) */
    float ground_normal[3];
    float ground_distance;
    float side_contact_normal[3];
    int32_t ground_triangle_index;
    int32_t ground_transition_frames;
    int32_t side_contact_frames;
    int32_t manifold_frames;     /* contactManifoldFrames */
    int32_t manifold_count;      /* contactManifoldTriangles.count */
    int32_t manifold_triangles[CQ_MANIFOLD_MAX];
    float manifold_normals[CQ_MANIFOLD_MAX][3];
    uint8_t grounded;
    uint8_t grounded_near;
    uint8_t ground_sliding;
    uint8_t _pad[5];
} cq_character_state; /* 168 bytes */

#define CQ_MAS_APPLY_GRAVITY 1u /* run GravitySystem's rule first (Systems.swift:603-619) */
/* Every character of the batch is a solid agent (AgentCollisionComponent defaults, Components.swift): each slide
 * iteration also sweeps the capsule against every other character's capsule, taken from a snapshot of positions and
 * (post-gravity) velocities made before any character of the step moves (AgentSweepSolver / collectAgentStates,
 * Systems.swift:1023-1091, 1592-1611), and HitSelector (1378-1399) picks between the static and the agent hit.
 * The batch is the crowd: characters of different calls do not see each other, and a host-pointer call runs as one
 * chunk.  Calls with this flag on one world must be stream-ordered (they share the snapshot scratch). */
#define CQ_MAS_AGENTS 2u

/* A kinematic platform as PlatformCarry.computeDelta sees it (Systems.swift:644-732): the world AABB of its
 * collision mesh under the CURRENT transform (meshWorldAABB, :627-642) and its motion over this fixed step
 * (positionF - prevPositionF).  Its triangles are ordinary dynamic-set parts of the world. */
typedef struct cq_platform {
    float aabb_min[3];
    float aabb_max[3];
    float delta[3];
} cq_platform;

void cq_controller_params_default(cq_controller_params *p);
void cq_character_state_init(cq_character_state *s, const float position[3], const float velocity[3]);

int cq_move_and_slide_batch(cq_world *w, cq_character_state *inout, int32_t n,
                            const cq_controller_params *params, float dt,
                            const float gravity[3], uint32_t flags);
int cq_move_and_slide_device(cq_world *w, cq_character_state *d_inout, int32_t n,
                             const cq_controller_params *params, float dt,
                             const float gravity[3], uint32_t flags, void *stream);

/* Same step with kinematic platforms: before the velocity gate every character is carried by the platform it
 * stands on / pushed by a platform moving into its side (applyPlatformDelta, Systems.swift:1618-1633).
 * Platforms are taken in the given order (the reference iterates a Dictionary). */
int cq_move_and_slide_batch_ex(cq_world *w, cq_character_state *inout, int32_t n,
                               const cq_controller_params *params, float dt, const float gravity[3],
                               uint32_t flags, const cq_platform *platforms, int32_t n_platforms);
int cq_move_and_slide_device_ex(cq_world *w, cq_character_state *d_inout, int32_t n,
                                const cq_controller_params *params, float dt, const float gravity[3],
                                uint32_t flags, const cq_platform *platforms /* HOST pointer */,
                                int32_t n_platforms, void *stream);

/* Kinematic platform records from the world, on the device: d_out[i] (a cq_platform, DEVICE pointer, n records) gets
 * the world AABB of entity d_entity_ids[i] (device, n ids) and the motion d_deltas[3i..3i+2] (device, n*3 floats,
 * positionF - prevPositionF, which the caller owns as in the reference).  Written in stream order on `stream` (NULL = the
 * world's stream), without synchronising, allocating or touching host memory, so a graph can rebuild the records every
 * replay and hand them to cq_move_and_slide_device_platforms.
 *
 * aabb_min / aabb_max are the min / max over the world-space vertices of every part with a matching entity_id, in both
 * sets, as left by every update queued on the world before this call: meshWorldAABB (Systems.swift:627-642) of the
 * current model, computed with the same float32 operations as the transform update.  One difference from
 * meshWorldAABB: parts without triangles do not contribute (updates skip them, CollisionQuery.swift:427, so their world
 * vertices are not current); an id whose parts all lack triangles gets the empty box (min = +inf, max = -inf), which
 * overlaps no capsule, so its record is inert.  An unknown id gets the empty box and a zero delta, inert too.  Records
 * are independent: *d_status (a device int32, may be NULL) receives the number of unknown ids, 0 on success, in stream
 * order, and every known id still gets its record.  NULL world, n < 0, or a NULL array with n > 0 return CQ_ERR_INVALID
 * before any CUDA call; n == 0 returns CQ_OK and queues nothing.
 *
 * Ordering is that of every launcher: the call sees every update queued before it on any stream, and the next
 * asynchronous update waits until it has read the vertices.  Launches: 1 whatever n is, one CTA per id (at most one
 * resident wave, striding over the ids); the cost grows with the vertex count of the named entities.  May be recorded
 * into a CUDA graph (see the capture contract below the *_device twins). */
int cq_world_platforms_device(cq_world *w, const uint32_t *d_entity_ids, const float *d_deltas, int32_t n,
                              cq_platform *d_out, int32_t *d_status, void *stream);

/* Device-platform twin of cq_move_and_slide_device_ex: the same step, with results equal to it byte for byte for the
 * same records (CQ_MAS_AGENTS included), except that d_platforms is a DEVICE pointer to n_platforms records that the
 * kernels read when they execute.  A graph that recorded this call therefore uses whatever the buffer holds at replay
 * (e.g. what cq_world_platforms_device wrote earlier in the same graph); n_platforms is a scalar recorded with the
 * graph, like n.  Any n_platforms >= 0 is accepted (the host-array calls take at most 64, because their records travel
 * in the kernel arguments); the cost is linear in n_platforms per character, as in the reference.  n_platforms < 0, or
 * a NULL d_platforms with n_platforms > 0, return CQ_ERR_INVALID before any CUDA call, as do the checks of the _ex
 * call.  Launches: the same as cq_move_and_slide_device_ex. */
int cq_move_and_slide_device_platforms(cq_world *w, cq_character_state *d_inout, int32_t n,
                                       const cq_controller_params *params, float dt, const float gravity[3],
                                       uint32_t flags, const cq_platform *d_platforms, int32_t n_platforms,
                                       void *stream);

/* ---- a crowd moved in slices ------------------------------------------------
 * CQ_MAS_AGENTS in two stages, so that the slices of one crowd can move on different GPUs (or in different calls) and
 * still see each other: every slice first writes the snapshot records of its own characters into its range of one
 * crowd-wide snapshot array, the array is made whole (cq_group_gather_records / cq_group_gather_records_local, 32-byte
 * records), then every slice moves its characters against the whole snapshot.  An agent's identity is its position in
 * the snapshot array. */
typedef struct cq_agent_snapshot {   /* collectAgentStates (Systems.swift:1592-1611), one per character */
    float position[3]; float _reserved0;   /* positionF */
    float velocity[3]; float _reserved1;   /* post-gravity linearVelocity as Float */
} cq_agent_snapshot;                      /* 32 bytes */

/* d_out[i] (DEVICE, n records) = the snapshot of d_states[i] (DEVICE, n records) that a CQ_MAS_AGENTS step with the same
 * dt, gravity and flags takes: the gravity rule of CQ_MAS_APPLY_GRAVITY, then position and velocity converted to float;
 * the reserved words are written as zero.  One launch on `stream` (NULL = the world's stream), no scratch, no
 * synchronisation, no allocation.  NULL world, n < 0, or a NULL array with n > 0 return CQ_ERR_INVALID before any CUDA
 * call; n == 0 returns CQ_OK and queues nothing. */
int cq_agent_snapshot_device(cq_world *w, const cq_character_state *d_states, int32_t n, float dt, const float gravity[3],
                             uint32_t flags, cq_agent_snapshot *d_out, void *stream);

/* One CQ_MAS_AGENTS step of the characters d_inout[0..n) (DEVICE), which are agents first_agent .. first_agent + n - 1
 * of the crowd whose snapshot is d_agents[0..n_agents) (DEVICE).  Each slice builds the crowd's whole agent grid from
 * the snapshot and moves only its own characters.  When every slice of a crowd is snapshotted first
 * (cq_agent_snapshot_device) and then moved with the same dt, gravity, flags and platforms, the records equal one
 * cq_move_and_slide_device_platforms(..., CQ_MAS_AGENTS) call on the whole crowd, byte for byte.  Platforms are a
 * DEVICE array read when the kernels run, as in cq_move_and_slide_device_platforms.
 * CQ_ERR_INVALID before any CUDA call: flags without CQ_MAS_AGENTS; n, n_agents or first_agent below 0;
 * first_agent + n > n_agents; a NULL array with a count above 0; any check of cq_move_and_slide_device_platforms.
 * n == 0 returns CQ_OK and queues nothing.  Stream-ordered with the other CQ_MAS_AGENTS calls on the world (they share
 * the grid scratch); may be recorded into a CUDA graph (see the capture contract above).
 * Launches: 14, plus 7 for the processing order when n >= 65,536 on a world of >= 262,144 static triangles (the
 * launches of cq_move_and_slide_device_platforms with CQ_MAS_AGENTS on n characters), whatever n_agents is. */
int cq_move_and_slide_device_agents(cq_world *w, cq_character_state *d_inout, int32_t n, const cq_agent_snapshot *d_agents,
                                    int32_t n_agents, int32_t first_agent, const cq_controller_params *params, float dt,
                                    const float gravity[3], uint32_t flags, const cq_platform *d_platforms,
                                    int32_t n_platforms, void *stream);

/* ---- resident crowd ------------------------------------------------------
 * The full-record calls above move 2 x 168 bytes per character per step across PCIe, which bounds them near 230 M
 * characters/s per GPU whatever the kernel does.  A crowd keeps the records in HBM between steps — they are private to
 * KinematicMoveStopSystem in the reference as well (CharacterControllerComponent, the contact-manifold cache) — and a
 * step exchanges what the rest of the frame exchanges with that system: PhysicsBodyComponent.linearVelocity in (what
 * GravitySystem / PhysicsIntentSystem left there, Systems.swift:228-233, 603-619), the pose out: 24 + 56 bytes per
 * character instead of 336.  Results are those of cq_move_and_slide_batch_ex on the same records, bit for bit. */
typedef struct cq_crowd cq_crowd;

typedef struct cq_crowd_pose {
    double position[3];
    double velocity[3];
    int32_t ground_triangle_index;
    uint8_t grounded;
    uint8_t grounded_near;
    uint8_t ground_sliding;
    uint8_t _pad;
} cq_crowd_pose; /* 56 bytes */

/* initial: n full records (host); the crowd lives on the world's device and must be destroyed before the world. */
int cq_crowd_create(cq_world *w, const cq_character_state *initial, int32_t n, cq_crowd **out);
void cq_crowd_destroy(cq_crowd *c);
int32_t cq_crowd_size(const cq_crowd *c);
/* One fixed step for every character.  velocity_in_xyz: n*3 doubles (host) written into the records first, NULL = keep
 * the stored velocities; pose_out: n records (host), NULL = nothing is copied back.  Pinned host memory
 * (cq_host_alloc) gives full PCIe bandwidth; copies and kernels of successive chunks overlap. */
int cq_crowd_step(cq_crowd *c, const double *velocity_in_xyz, const cq_controller_params *params, float dt,
                  const float gravity[3], uint32_t flags, const cq_platform *platforms, int32_t n_platforms,
                  cq_crowd_pose *pose_out);
/* Full records out of / into the crowd (host pointers, n records). */
int cq_crowd_read(cq_crowd *c, cq_character_state *out);
int cq_crowd_write(cq_crowd *c, const cq_character_state *in);
/* The resident records (device pointer, n records) for the *_device entry points, e.g. cq_agent_separation_device. */
cq_character_state *cq_crowd_device_states(cq_crowd *c);

/* AgentSeparationSystem.fixedUpdate (Systems.swift:1906-2210) over the batch — every character a solid agent, entity
 * order = index order: `iterations` (reference default 2) sweeps of {rebuild the XZ grid with cell 2r + separation_margin,
 * resolve overlapping pairs SEQUENTIALLY in index order: positional correction split by inverse mass, closing velocity
 * removed, each agent's share of the push vetoed by a blocking capsule cast when use_query != 0}, then per agent a
 * <= 2-cast slide from its pre-separation position (SlideOptions.agentSeparation) and a ground snap; position and
 * velocity are written back through Float as the reference does.  The sequential semantics are reproduced exactly (the
 * turns are scheduled along their conflict DAG).  mass_weight: AgentCollisionComponent.massWeight per character
 * (<= 0 = immovable), NULL = 1.0.  separation_margin 0.2, height_margin 0.1 are the reference defaults.  n < 2 is a
 * no-op.  The _device variant is stream-ordered but synchronises the stream once at its end to report the outcome; on
 * an error neither call changes any record.  Errors: CQ_ERR_INVALID "the crowd spans more than 2^31 grid cells" and
 * "agents drifted more than 15 cells within one sweep", CQ_ERR_CUDA "the turn schedule stalled". */
int cq_agent_separation_batch(cq_world *w, cq_character_state *inout, int32_t n, const cq_controller_params *params,
                              const float *mass_weight, int32_t iterations, float separation_margin, float height_margin,
                              int32_t use_query);
int cq_agent_separation_device(cq_world *w, cq_character_state *d_inout, int32_t n, const cq_controller_params *params,
                               const float *d_mass_weight, int32_t iterations, float separation_margin, float height_margin,
                               int32_t use_query, void *stream);

/* Outcome of an agent separation, as cq_agent_separation_device_async writes it to *d_status. */
#define CQ_SEP_STATUS_OK 0
#define CQ_SEP_STATUS_GRID 1    /* the crowd spans more than 2^31 grid cells (synchronous calls: CQ_ERR_INVALID) */
#define CQ_SEP_STATUS_DRIFT 2   /* agents drifted more than 15 cells within one sweep (synchronous calls: CQ_ERR_INVALID) */
#define CQ_SEP_STATUS_STALLED 3 /* the turn schedule made no progress (synchronous calls: CQ_ERR_CUDA) */

/* Stream-ordered twin of cq_agent_separation_device: the same sweeps with the same results, byte for byte, queued on
 * `stream` (NULL = the world's stream).  The call never synchronises and never reads device memory back, so it may be
 * recorded into a CUDA graph (see the capture contract above).  Uncaptured, each attempt is a launch of an instantiated
 * graph the world caches.  Every outcome is decided on the device: each sweep queues
 * its attempts for the safety radii R = 1, 3, 7, 15 up front, and an attempt runs only when the sweep is not finished
 * and nothing failed; an agent that drifted more than R cells restores the sweep's inputs on the device for the next.
 *
 * Errors are all-or-nothing: on any non-zero status the records are left byte for byte unchanged.  *d_status (a device
 * int32, may be NULL) receives CQ_SEP_STATUS_* in stream order.  NULL world, NULL params, n < 0, or a NULL d_inout with
 * n > 0 return CQ_ERR_INVALID before any CUDA call; n < 2 returns CQ_OK and queues nothing (d_status is not written).
 * Ordering against transform updates is that of every other launcher (see the update calls' ordering contract).
 *
 * Launches: a fixed number for given n and iterations, whatever drifted or failed: 3 + 23 * max(1, iterations) (per
 * sweep: 11 to rebuild the grid, 3 per attempt).  The rounds each attempt's device-side loop runs (3 kernels per round,
 * as many rounds as the conflict DAG is deep) are not known when the call returns and are not counted;
 * cq_agent_separation_device and cq_agent_separation_batch add them after their synchronisation. */
int cq_agent_separation_device_async(cq_world *w, cq_character_state *d_inout, int32_t n, const cq_controller_params *params,
                                     const float *d_mass_weight, int32_t iterations, float separation_margin,
                                     float height_margin, int32_t use_query, int32_t *d_status, void *stream);

/* ---- the GPUs of one box -----------------------------------------------------
 * The path shards by independent units (characters, sweeps, rays): mesh and trees are replicated on every GPU (the build
 * is deterministic, so every replica is identical), each GPU processes one contiguous range of the units, and nothing
 * is exchanged inside the algorithm.  The one collective a caller may want — the result records of all ranks in one
 * place — goes through NCCL over NVLink / NVSwitch.  The reference has no counterpart: its query object is built once
 * per scene (SceneServices.swift:45-50) and used by one thread.
 *
 * NCCL is loaded at run time (libnccl.so.2); every call below returns CQ_ERR_NCCL when it cannot be. */
typedef struct cq_group cq_group;
typedef struct cq_multi_world cq_multi_world;
#define CQ_GROUP_ID_BYTES 128

/* Contiguous range [lo, hi) of rank `rank`: lo = rank*n/n_ranks, hi = (rank+1)*n/n_ranks.  Ranges tile [0, n) exactly
 * and differ by at most one unit. */
void cq_shard_range(int64_t n_units, int32_t n_ranks, int32_t rank, int64_t *lo, int64_t *hi);

/* One process per GPU: rank 0 makes the id, the host ships its 128 bytes to the other ranks (MPI, a socket, a file,
 * torch.distributed ...), every rank then joins on the device that is current in its process. */
int cq_group_unique_id(uint8_t id[CQ_GROUP_ID_BYTES]);
int cq_group_create_rank(int32_t n_ranks, int32_t rank, const uint8_t id[CQ_GROUP_ID_BYTES], cq_group **out);
/* One process driving n GPUs: devices = NULL means 0 .. n_gpus-1. */
int cq_group_create_local(int32_t n_gpus, const int32_t *devices, cq_group **out);
void cq_group_destroy(cq_group *g);
int32_t cq_group_size(const cq_group *g);
int32_t cq_group_rank(const cq_group *g);              /* -1 for a local group */
int32_t cq_group_device(const cq_group *g, int32_t i); /* device of the i-th member (rank groups: i = 0) */

/* All-gather of fixed-size result records.  The batch of n_units records is sharded by cq_shard_range; d_local holds
 * this rank's shard, d_all (n_units * record_bytes bytes, device memory) receives the whole batch in unit order on
 * every rank.  Enqueued on `stream` (cudaStream_t), no synchronisation.  Equal shards: one ncclAllGather; ragged
 * shards: one ncclBroadcast per rank inside an NCCL group, straight to each shard's offset. */
int cq_group_gather_records(cq_group *g, const void *d_local, int64_t n_units, size_t record_bytes, void *d_all,
                            void *stream);
/* The same for a local group: one (d_local, d_all, stream) triple per device, in member order; streams = NULL uses
 * the group's own streams (cq_group_synchronize waits for them). */
int cq_group_gather_records_local(cq_group *g, const void *const *d_local, int64_t n_units, size_t record_bytes,
                                  void *const *d_all, void *const *streams);
int cq_group_synchronize(cq_group *g);

/* A world replicated on every device of a LOCAL group, and host-pointer batch calls sharded over the replicas: one
 * worker thread per device runs the single-GPU copy / compute pipeline on its contiguous range of the batch, results
 * land in the caller's arrays in unit order.  Same results as the single-GPU calls, byte for byte. */
int cq_world_create_multi(cq_group *g, const cq_mesh_part *parts, int32_t n_parts, const cq_world_options *options,
                          cq_multi_world **out);
void cq_multi_world_destroy(cq_multi_world *mw);
int32_t cq_multi_world_size(const cq_multi_world *mw);
cq_world *cq_multi_world_replica(cq_multi_world *mw, int32_t i); /* for the *_device entry points (set the device first) */
int cq_multi_update_transforms(cq_multi_world *mw, const uint32_t *entity_ids, const float *models, int32_t n);
int cq_multi_raycast_batch(cq_multi_world *mw, const cq_ray *rays, int32_t n, cq_ray_hit *out);
int cq_multi_capsule_cast_batch(cq_multi_world *mw, const cq_capsule_cast *q, int32_t n, int32_t mode, cq_cast_hit *out);
/* CQ_MAS_AGENTS is refused here (use cq_multi_move_and_slide_batch_ex). */
int cq_multi_move_and_slide_batch(cq_multi_world *mw, cq_character_state *inout, int32_t n,
                                  const cq_controller_params *params, float dt, const float gravity[3], uint32_t flags);
/* The step of cq_move_and_slide_batch_ex (0..64 host platforms) sharded over the replicas, CQ_MAS_AGENTS included: the
 * batch is one crowd.  With agents, each replica snapshots its shard (cq_agent_snapshot_device) into its range of a
 * crowd-sized snapshot buffer, one NCCL all-gather of the 32-byte records makes the snapshot whole on every replica, and
 * each replica moves its shard against it (cq_move_and_slide_device_agents).  Records equal cq_move_and_slide_batch_ex
 * on one GPU, byte for byte.  The multi world keeps the per-replica buffers (grown on demand, freed by
 * cq_multi_world_destroy).  Without agents: cq_multi_move_and_slide_batch plus platforms. */
int cq_multi_move_and_slide_batch_ex(cq_multi_world *mw, cq_character_state *inout, int32_t n,
                                     const cq_controller_params *params, float dt, const float gravity[3], uint32_t flags,
                                     const cq_platform *platforms, int32_t n_platforms);

/* ---- instrumentation ------------------------------------------------------
 * Work counters of the last device/batch call, accumulated on the device when
 * counting is enabled (off by default; the reference's CollisionQueryStats,
 * CollisionQuery.swift:280-290, plus the node count the roofline formula needs). */
typedef struct cq_counters {
    uint64_t queries;          /* BVH traversals started */
    uint64_t nodes_visited;    /* child boxes tested (32 B each, algorithmic) */
    uint64_t candidates;       /* = capsuleCandidateCount: tri AABB overlaps swept AABB, layer ok */
    uint64_t distance_evals;   /* segmentTriangleDistance evaluations actually executed */
    uint64_t kernel_launches;  /* kernels launched by this library since the last reset */
} cq_counters;
/* mode: CQ_COUNT_OFF; CQ_COUNT_REFERENCE — `candidates` equals the reference's capsuleCandidateCount (a counting launch
 * then queues every candidate of the whole sweep's box, as the reference does; results are the same, the launch is slower);
 * CQ_COUNT_PATH — the counters of the path as shipped: sweeps that already hold a hit cull nodes and triangles against the
 * box of the capsule swept to that hit and drop candidates that cannot matter before evaluating them, so `nodes_visited`,
 * `candidates` and `distance_evals` are what the kernel really touched (bench.py's roofline figures use this mode). */
#define CQ_COUNT_OFF 0
#define CQ_COUNT_REFERENCE 1
#define CQ_COUNT_PATH 2
int cq_world_set_counting(cq_world *w, int32_t mode);
int cq_world_read_counters(cq_world *w, cq_counters *out, int32_t reset);

/* pinned host memory for the batch calls (optional; plain malloc'ed memory works too) */
void *cq_host_alloc(size_t bytes);
void cq_host_free(void *p);

const char *cq_last_error(void);
const char *cq_version(void);

#ifdef __cplusplus
}
#endif
#endif /* CQ_H */
