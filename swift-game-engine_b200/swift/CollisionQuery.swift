// CollisionQuery.swift — Swift binding of libcq.so (SOURCE ONLY: no Swift toolchain exists in the build
// environment, so this file has never been compiled; see INTEGRATION.md).
//
// Drop-in for the reference's `final class CollisionQuery` (Game/CollisionQuery.swift:54-160): same method
// names and signatures, implemented over the C ABI of include/cq.h through a module map
// (`module CQ { header "cq.h" link "cq" }`).  The engine's `World` is flattened into `cq_mesh_part`s by
// `makeParts(world:activeEntityIDs:)` exactly as `TriangleMeshSet.rebuild` walks it (:331-417).
import CQ
import simd

public final class CollisionQuery {
    private var handle: OpaquePointer?
    /// Set membership as the library sees it (cq_mesh_part.is_dynamic): updateStaticTransforms / updateDynamicTransforms
    /// only move entities of their own set, like TriangleMeshSet.updateTransforms, which skips entities without a slice
    /// in the addressed set (CollisionQuery.swift:427).
    private var dynamicIDs: Set<UInt32> = []
    private var knownIDs: Set<UInt32> = []
    /// Text of the last library error (cq_last_error()); nil when the last call succeeded.  The reference reports failure
    /// through Optionals only, so every query keeps answering nil on error and this is where the reason can be read.
    public private(set) var lastError: String?

    /// `referenceOrder`: exact ties and capsuleOverlapAll overflow resolved in the reference's own visiting order
    /// (CQ_ORDER_REFERENCE, the library's default); false selects the tree-independent rule (include/cq.h).
    public init(world: World, activeEntityIDs: Set<UInt32>? = nil, referenceOrder: Bool = true) {
        let built = CollisionQuery.makeParts(world: world, activeEntityIDs: activeEntityIDs)
        var parts = built.parts
        // the library copies everything it needs during cq_world_create: point the parts at the arrays only for the call
        var options = cq_world_options()
        cq_world_options_default(&options)
        options.order = referenceOrder ? Int32(CQ_ORDER_REFERENCE) : Int32(CQ_ORDER_CANONICAL)
        var h: OpaquePointer?
        // StaticMeshComponent.triangleMaterials (CollisionQuery.swift:363-369): handed over per part; the library applies the
        // reference's rule (used when there is one entry per triangle, ignored otherwise)
        var perTri: [cq_triangle_materials] = []
        let rc: Int32 = CollisionQuery.withMaterialArrays(built.triangleMaterials, &perTri) {
            perTri.withUnsafeBufferPointer { tm in
                options.n_triangle_materials = Int32(tm.count)
                options.triangle_materials = tm.baseAddress
                return CollisionQuery.withArrays(built.positions, built.indices, &parts) {
                    cq_world_create_ex(&parts, Int32(parts.count), &options, &h)
                }
            }
        }
        handle = rc == CQ_OK ? h : nil // on failure every query answers nil (no CPU fallback exists)
        lastError = rc == CQ_OK ? nil : String(cString: cq_last_error())
        for p in built.parts {
            knownIDs.insert(p.entity_id)
            if p.is_dynamic != 0 { dynamicIDs.insert(p.entity_id) }
        }
    }

    deinit { cq_world_destroy(handle) }

    public func updateStaticTransforms(world: World, entities: [Entity], activeEntityIDs: Set<UInt32>? = nil) {
        update(world: world, entities: entities.filter { !dynamicIDs.contains($0.id) }, activeEntityIDs: activeEntityIDs)
    }

    public func updateDynamicTransforms(world: World, entities: [Entity], activeEntityIDs: Set<UInt32>? = nil) {
        update(world: world, entities: entities.filter { dynamicIDs.contains($0.id) }, activeEntityIDs: activeEntityIDs)
    }

    public func raycast(origin: SIMD3<Float>, direction: SIMD3<Float>, maxDistance: Float,
                        mask: UInt32 = CollisionLayer.all) -> RaycastHit? {
        var r = cq_ray(origin: (origin.x, origin.y, origin.z), direction: (direction.x, direction.y, direction.z),
                       max_distance: maxDistance, mask: mask)
        var h = cq_ray_hit()
        guard cq_raycast_batch(handle, &r, 1, &h) == CQ_OK, h.triangle_index >= 0 else { return nil }
        return RaycastHit(distance: h.distance, position: v3(h.position), normal: v3(h.normal),
                          triangleIndex: Int(h.triangle_index), material: material(h.triangle_index))
    }

    public func capsuleCast(from: SIMD3<Float>, delta: SIMD3<Float>, radius: Float, halfHeight: Float,
                            mask: UInt32 = CollisionLayer.all) -> CapsuleCastHit? {
        cast(from, delta, radius, halfHeight, mask, CQ_CAST_ALL, 0)
    }

    public func capsuleCastBlocking(from: SIMD3<Float>, delta: SIMD3<Float>, radius: Float, halfHeight: Float,
                                    mask: UInt32 = CollisionLayer.all) -> CapsuleCastHit? {
        cast(from, delta, radius, halfHeight, mask, CQ_CAST_BLOCKING, 0)
    }

    public func capsuleCastGround(from: SIMD3<Float>, delta: SIMD3<Float>, radius: Float, halfHeight: Float,
                                  minNormalY: Float, mask: UInt32 = CollisionLayer.all) -> CapsuleCastHit? {
        cast(from, delta, radius, halfHeight, mask, CQ_CAST_GROUND, minNormalY)
    }

    public func capsuleOverlap(from: SIMD3<Float>, radius: Float, halfHeight: Float,
                               mask: UInt32 = CollisionLayer.all) -> CapsuleOverlapHit? {
        var c = cq_capsule(from: (from.x, from.y, from.z), radius: radius, half_height: halfHeight, mask: mask)
        var h = cq_overlap_hit()
        guard cq_capsule_overlap_batch(handle, &c, 1, &h) == CQ_OK, h.triangle_index >= 0 else { return nil }
        return overlapHit(h)
    }

    public func capsuleOverlapAll(from: SIMD3<Float>, radius: Float, halfHeight: Float, maxHits: Int = 8,
                                  mask: UInt32 = CollisionLayer.all) -> [CapsuleOverlapHit] {
        let cap = min(max(1, maxHits), Int(CQ_MAX_OVERLAP_HITS))
        var c = cq_capsule(from: (from.x, from.y, from.z), radius: radius, half_height: halfHeight, mask: mask)
        var hits = [cq_overlap_hit](repeating: cq_overlap_hit(), count: cap)
        var count: Int32 = 0
        guard cq_capsule_overlap_all_batch(handle, &c, 1, Int32(cap), &hits, &count, nil) == CQ_OK else { return [] }
        return hits.prefix(Int(count)).map(overlapHit)
    }

    /// Batched replacement of KinematicMoveStopSystem.fixedUpdate's per-entity loop (Systems.swift:1842-1901).
    public func moveAndSlide(states: inout [cq_character_state], params: cq_controller_params, dt: Float,
                             gravity: SIMD3<Float> = SIMD3<Float>(0, -98, 0), applyGravity: Bool = true) -> Bool {
        var p = params
        var g = (gravity.x, gravity.y, gravity.z)
        return withUnsafePointer(to: &g) { gp in
            gp.withMemoryRebound(to: Float.self, capacity: 3) {
                cq_move_and_slide_batch(handle, &states, Int32(states.count), &p, dt, $0,
                                        applyGravity ? UInt32(CQ_MAS_APPLY_GRAVITY) : 0) == CQ_OK
            }
        }
    }

    /// The same step with kinematic platforms (PlatformCarry, Systems.swift:644-732) and, with `agents`, capsule-capsule
    /// CCD between the characters of the batch (AgentSweepSolver / HitSelector, Systems.swift:1053-1091, 1378-1399).
    public func moveAndSlide(states: inout [cq_character_state], params: cq_controller_params, dt: Float,
                             gravity: SIMD3<Float> = SIMD3<Float>(0, -98, 0), platforms: [cq_platform], agents: Bool,
                             applyGravity: Bool = true) -> Bool {
        var p = params
        var g = (gravity.x, gravity.y, gravity.z)
        let flags = (applyGravity ? UInt32(CQ_MAS_APPLY_GRAVITY) : 0) | (agents ? UInt32(CQ_MAS_AGENTS) : 0)
        return withUnsafePointer(to: &g) { gp in
            gp.withMemoryRebound(to: Float.self, capacity: 3) {
                cq_move_and_slide_batch_ex(handle, &states, Int32(states.count), &p, dt, $0, flags, platforms,
                                           Int32(platforms.count)) == CQ_OK
            }
        }
    }

    /// Batched AgentSeparationSystem.fixedUpdate (Systems.swift:2136-2210), sequential pair-resolution semantics kept.
    public func agentSeparation(states: inout [cq_character_state], params: cq_controller_params, massWeights: [Float]? = nil,
                                iterations: Int = 2, separationMargin: Float = 0.2, heightMargin: Float = 0.1,
                                useQuery: Bool = true) -> Bool {
        var p = params
        return cq_agent_separation_batch(handle, &states, Int32(states.count), &p, massWeights, Int32(max(1, iterations)),
                                         separationMargin, heightMargin, useQuery ? 1 : 0) == CQ_OK
    }

    // MARK: - private

    private func v3(_ t: (Float, Float, Float)) -> SIMD3<Float> { SIMD3<Float>(t.0, t.1, t.2) }

    private func material(_ tri: Int32) -> SurfaceMaterial {
        var m = cq_material()
        cq_world_triangle_material(handle, tri, &m)
        return SurfaceMaterial(muS: m.mu_s, muK: m.mu_k, flattenGround: m.flatten_ground != 0)
    }

    private func overlapHit(_ h: cq_overlap_hit) -> CapsuleOverlapHit {
        CapsuleOverlapHit(depth: h.depth, position: v3(h.position), normal: v3(h.normal),
                          triangleNormal: v3(h.triangle_normal), triangleIndex: Int(h.triangle_index),
                          material: material(h.triangle_index))
    }

    private func cast(_ from: SIMD3<Float>, _ delta: SIMD3<Float>, _ radius: Float, _ halfHeight: Float, _ mask: UInt32,
                      _ mode: Int32, _ minNormalY: Float) -> CapsuleCastHit? {
        var q = cq_capsule_cast(from: (from.x, from.y, from.z), delta: (delta.x, delta.y, delta.z), radius: radius,
                                half_height: halfHeight, mask: mask, min_normal_y: minNormalY)
        var h = cq_cast_hit()
        guard cq_capsule_cast_batch(handle, &q, 1, mode, &h) == CQ_OK, h.triangle_index >= 0 else { return nil }
        return CapsuleCastHit(toi: h.toi, position: v3(h.position), normal: v3(h.normal),
                              triangleNormal: v3(h.triangle_normal), triangleIndex: Int(h.triangle_index),
                              material: material(h.triangle_index))
    }

    private func update(world: World, entities: [Entity], activeEntityIDs: Set<UInt32>?) {
        let tStore = world.store(TransformComponent.self)
        let filtered = entities.filter { activeEntityIDs?.contains($0.id) ?? true }
        var ids: [UInt32] = []
        var models: [Float] = []
        for e in filtered {
            guard let t = tStore[e], knownIDs.contains(e.id) else { continue } // `guard let slice = slices[e] else { continue }`
            ids.append(e.id)
            let m = t.modelMatrix
            for c in [m.columns.0, m.columns.1, m.columns.2, m.columns.3] { models += [c.x, c.y, c.z, c.w] }
        }
        if ids.isEmpty { return }
        let rc = cq_world_update_transforms(handle, ids, models, Int32(ids.count))
        lastError = rc == CQ_OK ? nil : String(cString: cq_last_error())
    }

    /// Stream-ordered update (cq_world_update_transforms_async): entity ids + column-major model matrices (16 floats each),
    /// queued on `stream` (a cudaStream_t; nil = the world's own stream) without waiting.  The arrays are copied before
    /// the call returns; every later call on the world sees the new pose.
    public func updateTransformsAsync(ids: [UInt32], models: [Float], stream: UnsafeMutableRawPointer? = nil) -> Bool {
        let rc = cq_world_update_transforms_async(handle, ids, models, Int32(ids.count), stream)
        lastError = rc == CQ_OK ? nil : String(cString: cq_last_error())
        return rc == CQ_OK
    }

    /// Entities with Transform + StaticMesh (collides), ascending id (the reference iterates a Dictionary, i.e. in
    /// per-process random order — World.swift:99-118; the library fixes the order so triangle numbering is stable).
    /// Geometry is returned as plain Swift arrays; `withArrays` lends their storage to the C structs for one call.
    /// StaticMeshComponent.triangleMaterials (per-triangle materials, CollisionQuery.swift:363-369) travel beside the parts
    /// as (entity id, materials) pairs and reach the library through cq_world_options.triangle_materials.
    private static func makeParts(world: World, activeEntityIDs: Set<UInt32>?)
        -> (parts: [cq_mesh_part], positions: [[Float]], indices: [[UInt32]],
            triangleMaterials: [(UInt32, [cq_surface_material])]) {
        let tStore = world.store(TransformComponent.self)
        let mStore = world.store(StaticMeshComponent.self)
        let pStore = world.store(PhysicsBodyComponent.self)
        var parts: [cq_mesh_part] = []
        var positions: [[Float]] = []
        var indices: [[UInt32]] = []
        var triangleMaterials: [(UInt32, [cq_surface_material])] = []
        let entities = world.query(TransformComponent.self, StaticMeshComponent.self).sorted { $0.id < $1.id }
        for e in entities {
            if let active = activeEntityIDs, !active.contains(e.id) { continue }
            guard let t = tStore[e], let m = mStore[e], m.collides else { continue }
            if let perTri = m.triangleMaterials {
                triangleMaterials.append((e.id, perTri.map {
                    cq_surface_material(mu_s: $0.muS, mu_k: $0.muK, flatten_ground: $0.flattenGround ? 1 : 0, _pad: (0, 0, 0))
                }))
            }
            let mesh = m.collisionMesh ?? m.mesh
            var pos: [Float] = []
            pos.reserveCapacity(mesh.streams.positions.count * 3)
            for p in mesh.streams.positions { pos += [p.x, p.y, p.z] }
            let idx32: [UInt32] = mesh.indices16?.map { UInt32($0) } ?? mesh.indices32 ?? []
            var part = cq_mesh_part()
            part.n_verts = Int32(mesh.streams.positions.count)
            part.n_indices = Int32(idx32.count)
            let mm = t.modelMatrix
            withUnsafeMutableBytes(of: &part.model) { raw in
                let f = raw.bindMemory(to: Float.self)
                var k = 0
                for c in [mm.columns.0, mm.columns.1, mm.columns.2, mm.columns.3] { f[k] = c.x; f[k + 1] = c.y; f[k + 2] = c.z; f[k + 3] = c.w; k += 4 }
            }
            part.layer = m.collisionLayer
            part.mu_s = m.material.muS
            part.mu_k = m.material.muK
            part.flatten_ground = m.material.flattenGround ? 1 : 0
            part.is_dynamic = (pStore[e].map { $0.bodyType != .static } ?? false) ? 1 : 0
            part.entity_id = e.id
            parts.append(part)
            positions.append(pos)
            indices.append(idx32)
        }
        return (parts, positions, indices, triangleMaterials)
    }

    /// Runs `body` with `out` holding one cq_triangle_materials per entry, pointing at that entry's storage (valid only
    /// inside the call).
    private static func withMaterialArrays<R>(_ lists: [(UInt32, [cq_surface_material])], _ out: inout [cq_triangle_materials],
                                              _ body: () -> R) -> R {
        func go(_ k: Int) -> R {
            if k == lists.count { return body() }
            return lists[k].1.withUnsafeBufferPointer { mp in
                out.append(cq_triangle_materials(entity_id: lists[k].0, n: Int32(mp.count), materials: mp.baseAddress))
                return go(k + 1)
            }
        }
        out.removeAll()
        return go(0)
    }

    /// Runs `body` with every part pointing at its arrays' storage (valid only inside the call; nothing is leaked).
    private static func withArrays<R>(_ positions: [[Float]], _ indices: [[UInt32]], _ parts: inout [cq_mesh_part],
                                      _ body: () -> R) -> R {
        func go(_ k: Int) -> R {
            if k == parts.count { return body() }
            return positions[k].withUnsafeBufferPointer { pp in
                indices[k].withUnsafeBufferPointer { ip in
                    parts[k].positions_xyz = pp.baseAddress
                    parts[k].indices = ip.baseAddress
                    return go(k + 1)
                }
            }
        }
        return go(0)
    }
}
