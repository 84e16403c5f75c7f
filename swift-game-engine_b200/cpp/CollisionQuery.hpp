// CollisionQuery.hpp — C++ host-side mirror of the reference's `final class CollisionQuery`
// (Game/CollisionQuery.swift:54-160) over the C ABI of include/cq.h.  Header-only; link with libcq.so.
//
// The reference's toolchain (Swift) is absent from this environment, so this is the compiled-language
// host layer; swift/CollisionQuery.swift is the same thing as Swift source.  Method names, argument
// meaning and error behaviour follow the reference: single-query methods return std::optional (nil =
// no hit / empty world), nothing throws for "no hit"; only construction failure (no CUDA device, bad
// mesh) throws.  Batched overloads take spans of records and are what a crowd system should call.
#pragma once
#include <cstdint>
#include <optional>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/cq.h"

namespace cqhost {

struct Float3 {
    float x, y, z;
};

struct SurfaceMaterial { // Components.swift:704-716
    float muS = 0.8f, muK = 0.6f;
    bool flattenGround = false;
};

struct RaycastHit { // CollisionQuery.swift:28-34
    float distance;
    Float3 position, normal;
    int triangleIndex;
    SurfaceMaterial material;
};
struct CapsuleCastHit { // CollisionQuery.swift:36-43
    float toi;
    Float3 position, normal, triangleNormal;
    int triangleIndex;
    SurfaceMaterial material;
};
struct CapsuleOverlapHit { // CollisionQuery.swift:45-52
    float depth;
    Float3 position, normal, triangleNormal;
    int triangleIndex;
    SurfaceMaterial material;
};

class CollisionQuery {
  public:
    // init(world:activeEntityIDs:) — the caller flattens its (Transform, StaticMesh, body type) entities into parts
    // referenceOrder (default): exact ties, capsuleOverlapAll overflow and grazing rays come out as in the reference's own
    // tree and visiting order (CQ_ORDER_REFERENCE, include/cq.h); false = the tree-independent rule, no host build.
    // triangleMaterials: StaticMeshComponent.triangleMaterials of the parts that have them (used when there is one entry per
    // triangle of the part, ignored otherwise — CollisionQuery.swift:363-369); the library copies them.
    explicit CollisionQuery(const std::vector<cq_mesh_part> &parts, bool referenceOrder = true,
                            const std::vector<cq_triangle_materials> &triangleMaterials = {}) {
        cq_world_options opt;
        cq_world_options_default(&opt);
        opt.order = referenceOrder ? CQ_ORDER_REFERENCE : CQ_ORDER_CANONICAL;
        opt.n_triangle_materials = (int32_t)triangleMaterials.size();
        opt.triangle_materials = triangleMaterials.empty() ? nullptr : triangleMaterials.data();
        if (cq_world_create_ex(parts.data(), (int32_t)parts.size(), &opt, &w_) != CQ_OK)
            throw std::runtime_error(std::string("cq_world_create: ") + cq_last_error());
    }
    ~CollisionQuery() { cq_world_destroy(w_); }
    CollisionQuery(const CollisionQuery &) = delete;
    CollisionQuery &operator=(const CollisionQuery &) = delete;

    // updateStaticTransforms / updateDynamicTransforms (CollisionQuery.swift:69-83): entity ids + new modelMatrix each
    bool updateTransforms(const std::vector<uint32_t> &entities, const std::vector<float> &models16) {
        return cq_world_update_transforms(w_, entities.data(), models16.data(), (int32_t)entities.size()) == CQ_OK;
    }
    // the same update queued on `stream` (a cudaStream_t; nullptr = the world's own stream) without waiting; the arrays are
    // copied before the call returns, and every later call on the world sees the new pose (include/cq.h)
    bool updateTransformsAsync(const std::vector<uint32_t> &entities, const std::vector<float> &models16, void *stream = nullptr) {
        return cq_world_update_transforms_async(w_, entities.data(), models16.data(), (int32_t)entities.size(), stream) == CQ_OK;
    }

    std::optional<RaycastHit> raycast(Float3 origin, Float3 direction, float maxDistance, uint32_t mask = CQ_LAYER_ALL) {
        cq_ray r = {{origin.x, origin.y, origin.z}, {direction.x, direction.y, direction.z}, maxDistance, mask};
        cq_ray_hit h;
        if (cq_raycast_batch(w_, &r, 1, &h) != CQ_OK || h.triangle_index < 0) return std::nullopt;
        return RaycastHit{h.distance, f3(h.position), f3(h.normal), h.triangle_index, material(h.triangle_index)};
    }
    std::optional<CapsuleCastHit> capsuleCast(Float3 from, Float3 delta, float radius, float halfHeight,
                                              uint32_t mask = CQ_LAYER_ALL) {
        return cast(from, delta, radius, halfHeight, mask, CQ_CAST_ALL, 0.0f);
    }
    std::optional<CapsuleCastHit> capsuleCastBlocking(Float3 from, Float3 delta, float radius, float halfHeight,
                                                      uint32_t mask = CQ_LAYER_ALL) {
        return cast(from, delta, radius, halfHeight, mask, CQ_CAST_BLOCKING, 0.0f);
    }
    std::optional<CapsuleCastHit> capsuleCastGround(Float3 from, Float3 delta, float radius, float halfHeight,
                                                    float minNormalY, uint32_t mask = CQ_LAYER_ALL) {
        return cast(from, delta, radius, halfHeight, mask, CQ_CAST_GROUND, minNormalY);
    }
    std::optional<CapsuleOverlapHit> capsuleOverlap(Float3 from, float radius, float halfHeight,
                                                    uint32_t mask = CQ_LAYER_ALL) {
        cq_capsule c = {{from.x, from.y, from.z}, radius, halfHeight, mask};
        cq_overlap_hit h;
        if (cq_capsule_overlap_batch(w_, &c, 1, &h) != CQ_OK || h.triangle_index < 0) return std::nullopt;
        return ov(h);
    }
    std::vector<CapsuleOverlapHit> capsuleOverlapAll(Float3 from, float radius, float halfHeight, int maxHits = 8,
                                                     uint32_t mask = CQ_LAYER_ALL) {
        if (maxHits < 1) maxHits = 1; // max(1, maxHits), CollisionQuery.swift:157
        if (maxHits > CQ_MAX_OVERLAP_HITS) maxHits = CQ_MAX_OVERLAP_HITS;
        cq_capsule c = {{from.x, from.y, from.z}, radius, halfHeight, mask};
        cq_overlap_hit h[CQ_MAX_OVERLAP_HITS];
        int32_t count = 0;
        std::vector<CapsuleOverlapHit> out;
        if (cq_capsule_overlap_all_batch(w_, &c, 1, maxHits, h, &count, nullptr) != CQ_OK) return out;
        for (int i = 0; i < count; i++) out.push_back(ov(h[i]));
        return out;
    }

    // batched forms (what replaces the per-entity loops of KinematicMoveStopSystem / AgentSeparationSystem)
    bool capsuleCastBatch(const cq_capsule_cast *q, int32_t n, int mode, cq_cast_hit *out) {
        return cq_capsule_cast_batch(w_, q, n, mode, out) == CQ_OK;
    }
    bool raycastBatch(const cq_ray *rays, int32_t n, cq_ray_hit *out) { return cq_raycast_batch(w_, rays, n, out) == CQ_OK; }
    // KinematicMoveStopSystem.fixedUpdate body for n characters (Systems.swift:1842-1901)
    bool moveAndSlide(cq_character_state *inout, int32_t n, const cq_controller_params &p, float dt,
                      const float gravity[3], bool applyGravity = true) {
        return cq_move_and_slide_batch(w_, inout, n, &p, dt, gravity, applyGravity ? CQ_MAS_APPLY_GRAVITY : 0u) == CQ_OK;
    }
    // the same with kinematic platforms (PlatformCarry, Systems.swift:644-732) and, with agents = true, capsule-capsule CCD
    // between the characters of the batch (AgentSweepSolver, Systems.swift:1053-1091)
    bool moveAndSlide(cq_character_state *inout, int32_t n, const cq_controller_params &p, float dt, const float gravity[3],
                      const cq_platform *platforms, int32_t nPlatforms, bool agents, bool applyGravity = true) {
        uint32_t flags = (applyGravity ? CQ_MAS_APPLY_GRAVITY : 0u) | (agents ? CQ_MAS_AGENTS : 0u);
        return cq_move_and_slide_batch_ex(w_, inout, n, &p, dt, gravity, flags, platforms, nPlatforms) == CQ_OK;
    }
    // AgentSeparationSystem.fixedUpdate (Systems.swift:2136-2210); massWeight may be null (1.0 each)
    bool agentSeparation(cq_character_state *inout, int32_t n, const cq_controller_params &p, const float *massWeight = nullptr,
                         int iterations = 2, float separationMargin = 0.2f, float heightMargin = 0.1f, bool useQuery = true) {
        return cq_agent_separation_batch(w_, inout, n, &p, massWeight, iterations, separationMargin, heightMargin,
                                         useQuery ? 1 : 0) == CQ_OK;
    }

    cq_world *handle() const { return w_; }

  private:
    static Float3 f3(const float *v) { return {v[0], v[1], v[2]}; }
    SurfaceMaterial material(int tri) const {
        cq_material m;
        cq_world_triangle_material(w_, tri, &m);
        return {m.mu_s, m.mu_k, m.flatten_ground != 0};
    }
    CapsuleOverlapHit ov(const cq_overlap_hit &h) const {
        return {h.depth, f3(h.position), f3(h.normal), f3(h.triangle_normal), h.triangle_index, material(h.triangle_index)};
    }
    std::optional<CapsuleCastHit> cast(Float3 from, Float3 delta, float radius, float halfHeight, uint32_t mask, int mode,
                                       float minNormalY) {
        cq_capsule_cast q = {{from.x, from.y, from.z}, {delta.x, delta.y, delta.z}, radius, halfHeight, mask, minNormalY};
        cq_cast_hit h;
        if (cq_capsule_cast_batch(w_, &q, 1, mode, &h) != CQ_OK || h.triangle_index < 0) return std::nullopt;
        return CapsuleCastHit{h.toi, f3(h.position), f3(h.normal), f3(h.triangle_normal), h.triangle_index,
                              material(h.triangle_index)};
    }
    cq_world *w_ = nullptr;
};

} // namespace cqhost
