/*
 * libbepucuda — C ABI of the B200-native constraint solver + integrator for bepuphysics2.
 *
 * This is the drop-in boundary. The reference has no FFI at this seam (SURVEY.md §8b): the
 * solver is a C# class constructed inside Simulation.Create. The entry points below are what
 * a C# `CudaTimestepper : ITimestepper` (BepuPhysics/ITimestepper.cs:L15-34) P/Invokes in
 * place of `simulation.Solve(dt, threadDispatcher)` (BepuPhysics/Simulation.cs:L278-290).
 * Every pointer is a raw host pointer taken straight from the reference's own pinned
 * `Buffer<T>.Memory` fields (BepuUtilities/Memory/Buffer.cs:L13-21); no layout conversion is
 * required on the C# side. INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - every function returns an int32 status: 0 = ok, negative = error; the message for the
 *     last error on a context is available through bepucuda_last_error.
 *   - no exceptions cross the boundary; a context is used from one thread at a time.
 *   - the context owns all device memory, streams, CUDA graphs and events.
 *   - there is NO CPU fallback: if no CUDA device is usable, bepucuda_create fails with
 *     BEPUCUDA_ERR_NO_DEVICE.
 */
#ifndef BEPUCUDA_H
#define BEPUCUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BEPUCUDA_OK 0
#define BEPUCUDA_ERR_INVALID_ARGUMENT (-1)
#define BEPUCUDA_ERR_NO_DEVICE (-2)
#define BEPUCUDA_ERR_CUDA (-3)
/* Unknown constraint type id: the host shim should fall back to Simulation.Solve for the frame. */
#define BEPUCUDA_ERR_UNSUPPORTED_TYPE (-4)
/* A synchronized batch references the same dynamic body twice (ConstraintBatch invariant,
 * BepuPhysics/Solver.cs:L348-960 debug validators). */
#define BEPUCUDA_ERR_BATCH_INVARIANT (-5)
#define BEPUCUDA_ERR_BAD_STATE (-6)
#define BEPUCUDA_ERR_OUT_OF_MEMORY (-7)

typedef struct bepucuda_ctx bepucuda_ctx;

/* How the (substep, stage, batch) sequence of Solver.Solve (Solver_Solve.cs:L1419-1479) is sequenced
 * on the device. */
enum bepucuda_execution_mode {
    BEPUCUDA_EXEC_GRAPH = 0,      /* one kernel per (batch, stage) chained by programmatic dependent launch, whole frame captured in a CUDA graph */
    BEPUCUDA_EXEC_STREAM = 2      /* the same launches issued directly on the stream, no graph (profiling with ncu; the exchange-callback sharding) */
    /* 1 and 3 were a persistent cooperative kernel (grid barrier per stage) and a dataflow kernel (per-body version dependencies); both measured
     * slower than the graph on every benchmark configuration (profiles/r02_summary.md) and were removed: bepucuda_create rejects them. */
};

typedef struct bepucuda_config {
    int32_t device_ordinal;   /* CUDA device to own; one context <-> one GPU */
    /* 1 = kernels compiled with -fmad=false: bit-identical to a non-contracting fp32 CPU evaluation
     * (RyuJIT does not contract Vector<float> expressions; SURVEY.md §7-5). 0 = FMA contraction on (fast). */
    int32_t strict_fp;
    int32_t execution_mode;   /* enum bepucuda_execution_mode */
    int32_t reserved[5];      /* reserved[0]: unused; reserved[1]: 1 disables programmatic dependent launch between stage kernels */
} bepucuda_config;

/* Declarative stand-in for the user's IPoseIntegratorCallbacks struct (BepuPhysics/PoseIntegrator.cs:L42-94).
 * Covers Demos/DemoCallbacks.cs:L12-105 (DemoPoseIntegratorCallbacks) exactly:
 *   PrepareForIntegration(dt): linearDampingDt = pow(clamp(1 - linear_damping, 0, 1), dt), same angular, gravityDt = gravity * dt
 *   IntegrateVelocity: v.linear = (v.linear + gravityDt) * linearDampingDt; v.angular *= angularDampingDt
 * This is the one API narrowing of the drop-in (SURVEY.md §7 hard part 4). */
typedef struct bepucuda_integrator_desc {
    float gravity[3];
    float linear_damping;
    float angular_damping;
    int32_t angular_integration_mode;           /* AngularIntegrationMode: 0 Nonconserving, 1 ConserveMomentum, 2 ConserveMomentumWithGyroscopicTorque */
    int32_t allow_substeps_for_unconstrained;   /* IPoseIntegratorCallbacks.AllowSubstepsForUnconstrainedBodies */
    int32_t integrate_velocity_for_kinematics;  /* IPoseIntegratorCallbacks.IntegrateVelocityForKinematics */
} bepucuda_integrator_desc;

/* Replaces SimulationProfiler's Solver / PoseIntegrator stage timers (BepuPhysics/SimulationProfiler.cs:L6-75). */
typedef struct bepucuda_timings {
    float solve_ms;                 /* device time of the last bepucuda_solve (CUDA events on the context stream) */
    float upload_ms;                /* device-side time of the uploads since the previous solve (H2D copies + transposes) */
    float download_ms;              /* device-side time of the last downloads */
    int64_t constraint_count;       /* active constraints (empty fallback lanes excluded) */
    int64_t constraint_iterations;  /* sum over substeps of constraint_count * velocity_iterations(substep) */
    int64_t stage_count;            /* (batch, stage) barriers executed per solve */
    int64_t kernel_launches;        /* kernels launched (or graph kernel nodes executed) by the last solve */
    int64_t algorithmic_bytes;      /* SURVEY.md §8d compulsory-traffic model for the last solve */
    int64_t h2d_bytes;              /* bytes copied host->device since the previous solve */
    int64_t d2h_bytes;              /* bytes copied device->host by the last downloads */
    int32_t device_batch_count;     /* synchronized batches + fallback dependency levels */
    int32_t fallback_level_count;   /* dependency levels the sequential fallback batch was split into */
} bepucuda_timings;

/* Lifetime. Replaces: construction of Solver<TIntegrationCallbacks> in Simulation.Create (Simulation.cs:L135-141). */
int32_t bepucuda_create(const bepucuda_config* cfg, bepucuda_ctx** out);
int32_t bepucuda_destroy(bepucuda_ctx* ctx);
const char* bepucuda_last_error(bepucuda_ctx* ctx);

/* Static type registry query (mirrors TypeProcessor.BodiesPerConstraint / ConstrainedDegreesOfFreedom,
 * Constraints/TypeProcessor.cs:L31-39, and sizeof(TPrestepData)/sizeof(Vector<float>)).
 * Returns BEPUCUDA_ERR_UNSUPPORTED_TYPE for ids the device cannot solve. */
int32_t bepucuda_type_info(int32_t type_id, int32_t* bodies_per_constraint, int32_t* prestep_floats, int32_t* impulse_floats);

/* Optional: page-lock a host range (e.g. a BufferPool block, BepuUtilities/Memory/BufferPool.cs:L42) so the
 * per-frame copies run at full PCIe/C2C speed. */
int32_t bepucuda_host_register(bepucuda_ctx* ctx, void* ptr, int64_t bytes);
int32_t bepucuda_host_unregister(bepucuda_ctx* ctx, void* ptr);

/* Replaces: Solver.SubstepCount / VelocityIterationCount / VelocityIterationScheduler / FallbackBatchThreshold
 * (BepuPhysics/SolveDescription.cs:L21-38). The scheduler is pre-evaluated host-side into one iteration count per
 * substep (Solver_Solve.cs:L743-751). Batches with index >= fallback_batch_threshold are treated as the
 * sequential fallback batch (Solver.cs:L1878-1884). */
int32_t bepucuda_set_solve_description(bepucuda_ctx* ctx, int32_t substep_count,
                                       const int32_t* velocity_iterations_per_substep,
                                       int32_t fallback_batch_threshold);
/* Replaces: the TIntegrationCallbacks type argument of Solver<T>/PoseIntegrator<T>. */
int32_t bepucuda_set_integrator(bepucuda_ctx* ctx, const bepucuda_integrator_desc* desc);

/* Replaces: reads of Bodies.ActiveSet.DynamicsState (BepuPhysics/BodySet.cs:L33). `body_dynamics` is the raw
 * Buffer<BodyDynamics>.Memory: body_count records of 128 B (BepuPhysics/BodyProperties.cs:L11-46,L318-338). */
int32_t bepucuda_upload_bodies(bepucuda_ctx* ctx, const void* body_dynamics, int32_t body_count);

/* Replaces: iteration over Solver.ActiveSet.Batches[b].TypeBatches[t] (BepuPhysics/Solver.cs:L24-29,
 * Constraints/TypeBatch.cs:L10-27). source_bundle_width = Vector<float>.Count on the host. */
int32_t bepucuda_begin_constraints(bepucuda_ctx* ctx, int32_t source_bundle_width, int32_t batch_count);
/* body_references / prestep / accumulated_impulses are TypeBatch.BodyReferences / PrestepData / AccumulatedImpulses
 * .Memory in the reference's AOSOA layout (row = Vector<T>; bundle k lane i = constraint k*W+i,
 * BepuUtilities/BundleIndexing.cs:L50). constraint_count = TypeBatch.ConstraintCount (includes interior empty
 * lanes in the fallback batch). The accumulated_impulses pointer is retained until the next
 * bepucuda_begin_constraints so bepucuda_download_impulses can write results back in place. */
int32_t bepucuda_upload_type_batch(bepucuda_ctx* ctx, int32_t batch_index, int32_t type_batch_index, int32_t type_id,
                                   int32_t constraint_count,
                                   const int32_t* body_references, const float* prestep, float* accumulated_impulses);
/* Replaces: Solver.ConstrainedKinematicHandles (Solver.cs:L68), already mapped handle->index through
 * Bodies.HandleToLocation. */
int32_t bepucuda_set_constrained_kinematics(bepucuda_ctx* ctx, const int32_t* body_indices, int32_t count);
/* Replaces: Solver.PrepareConstraintIntegrationResponsibilities (Solver_Solve.cs:L1072-1388): validates the batch
 * invariant, levelises the fallback batch, computes which constraint lane owns each body's integration, builds the
 * stage program and (re)captures the CUDA graph when topology changed. */
int32_t bepucuda_end_constraints(bepucuda_ctx* ctx);

/* Refresh only the per-frame contact data of an already-uploaded type batch (same topology): what the narrow phase
 * rewrites every frame (CollisionDetection/NarrowPhaseConstraintUpdate.cs:L81-135). */
int32_t bepucuda_update_type_batch(bepucuda_ctx* ctx, int32_t batch_index, int32_t type_batch_index,
                                   const float* prestep, float* accumulated_impulses);

/* Device-side contact constraint update, first slice (SURVEY.md §8 f2): the accumulated impulses of contact type batches STAY on the device between
 * frames. Replaces, for a manifold whose constraint type did not change, the impulse half of NarrowPhase.UpdateConstraint
 * (CollisionDetection/NarrowPhaseConstraintUpdate.cs:L147-196): GatherOldImpulses -> RedistributeImpulses (L81-135) -> ScatterNewImpulses
 * (ContactConstraintAccessor.cs:L36-78). The host keeps writing the new description into TypeBatch.PrestepData
 * (Solver.ApplyDescriptionWithoutWaking) and passes that buffer as before.
 *   feature ids: ConstraintCache.FeatureId0.. of the pair (CollisionDetection/PairCache.cs), one int32 per contact: [constraint][contact], contact
 *   count given by the type id (convex 1-4, nonconvex 2-4). Only contact type ids (0-10, 15-17) are accepted.
 * bepucuda_set_contact_features stores the ids that belong to the impulses uploaded with bepucuda_upload_type_batch (call it between
 * begin/end_constraints or any time after). bepucuda_update_contacts uploads the frame's prestep data and NEW feature ids; at the next solve the
 * penetration impulses are redistributed from the old to the new ids on the device (matched ids keep their impulse, the unmatched share the
 * remainder equally); friction impulses are kept, as in the reference. No impulse bytes cross the bus in either direction. */
int32_t bepucuda_set_contact_features(bepucuda_ctx* ctx, int32_t batch_index, int32_t type_batch_index, const int32_t* feature_ids);
int32_t bepucuda_update_contacts(bepucuda_ctx* ctx, int32_t batch_index, int32_t type_batch_index, const float* prestep, const int32_t* new_feature_ids);
/* The motion half of BodyDynamics only: floats 0-15 of every 128-B record (pose + velocity, BodyProperties.cs:L318-338); the inertia half does not
 * change from frame to frame (local inertia) or is recomputed by the solve (world inertia). 64 B per body over the bus instead of 128. The body
 * count must equal the one of the last bepucuda_upload_bodies. */
int32_t bepucuda_upload_body_motion(bepucuda_ctx* ctx, const void* body_dynamics, int32_t body_count);
int32_t bepucuda_download_body_motion(bepucuda_ctx* ctx, void* body_dynamics_out, int32_t body_count);

/* Replaces: Solver.Solve (Solver_Solve.cs:L1415-1484) + PoseIntegrator.IntegrateAfterSubstepping
 * (PoseIntegrator.cs:L707-726). Asynchronous on the context stream. */
int32_t bepucuda_solve(bepucuda_ctx* ctx, float dt);
/* Blocks until prior work is done. */
int32_t bepucuda_synchronize(bepucuda_ctx* ctx);

/* Replaces: the in-place writes to Bodies.ActiveSet.DynamicsState done by ScatterVelocities/ScatterPose/ScatterInertia
 * (Bodies_GatherScatter.cs:L484-753). Writes pose, velocity and world inertia into 128-B records; local inertia and
 * padding floats of the destination are left untouched. Blocks until done. */
int32_t bepucuda_download_bodies(bepucuda_ctx* ctx, void* body_dynamics_out, int32_t body_count);
/* Replaces: in-place accumulated impulse updates in TypeBatch.AccumulatedImpulses. Writes every registered host
 * impulse buffer (the narrow phase reads them next frame). Blocks until done. */
int32_t bepucuda_download_impulses(bepucuda_ctx* ctx);
/* Replaces: in-place prestep mutation by IncrementallyUpdateForSubstep (contact depths). Test/diagnostic use. */
int32_t bepucuda_download_prestep(bepucuda_ctx* ctx, int32_t batch_index, int32_t type_batch_index, float* prestep_out);

int32_t bepucuda_get_timings(bepucuda_ctx* ctx, bepucuda_timings* out);

/* Replaces SimulationProfiler.Start/End (SimulationProfiler.cs:L25-60): CUDA events on the context stream, 16 slots. */
int32_t bepucuda_event_record(bepucuda_ctx* ctx, int32_t slot);
int32_t bepucuda_event_elapsed_ms(bepucuda_ctx* ctx, int32_t slot_begin, int32_t slot_end, float* ms);

/* Per-stage-kind device time of ONE frame, measured with a CUDA event pair around every stage launch (plain stream launches, no graph).
 * Index by stage kind: 0 WarmStart(first substep), 1 WarmStart, 2 Solve, 3 IncrementallyUpdateForSubstep, 4/5 kinematic prepasses, 6 final pose pass.
 * algorithmic_bytes follows SURVEY.md §8d. Advances the simulation exactly like bepucuda_solve(ctx, dt). */
typedef struct bepucuda_stage_profile {
    float ms[8];
    int64_t launches[8];
    int64_t algorithmic_bytes[8];
} bepucuda_stage_profile;
int32_t bepucuda_profile_stages(bepucuda_ctx* ctx, float dt, bepucuda_stage_profile* out);

/* PredictBoundingBoxes on the device (SURVEY.md §8 f4): the stage DefaultTimestepper runs right before collision detection
 * (PoseIntegrator.PredictBoundingBoxes, PoseIntegrator.cs:L307-370, L424-444), over the body state the solver keeps resident. Per active body:
 * the sleep-candidacy update (UpdateSleepCandidacy, L286-304: |v|^2 + |w|^2 of the CURRENT velocity against BodyActivity.SleepThreshold), the
 * velocity callback with PrepareForIntegration(dt) applied to a copy of the velocity (the integrated velocity is used for the prediction only and
 * is not stored, L339; kinematics only when IntegrateVelocityForKinematics), and for the convex primitive shapes the bounding box and speculative
 * margin BoundingBoxBatcher.ExecuteConvexBatch computes (Collidables/BoundingBoxBatcher.cs:L142-222; IConvexShape.GetBounds of Sphere.cs:L149-160,
 * Capsule.cs:L226-239, Box.cs:L211-222, Cylinder.cs:L222-235; BoundingBoxHelpers.cs:L12-58).
 *   bepucuda_body_shape.type: the reference's shape type id -- 0 sphere (a = radius), 1 capsule (a = radius, b = half length), 2 box (a, b, c = half
 *   width, height, length), 4 cylinder (a = radius, b = half length). Any other value (no shape; triangle, hull, compound, mesh) yields valid = 0
 *   for that body; its activity is still updated. bepucuda_set_shape_library + bepucuda_set_body_collidables below cover every built-in type.
 *   bepucuda_body_activity = BodyActivity (BodyProperties.cs:L386-416), updated in place.
 *   bounds_out: 8 floats per body {min.x, min.y, min.z, speculative margin, max.x, max.y, max.z, valid (1 or 0)}.
 * Uses the body arrays as they are on the device (after bepucuda_upload_bodies / bepucuda_solve) and the integrator set by bepucuda_set_integrator.
 * Results are bit-identical to a non-contracting fp32 evaluation of the reference's expressions. Blocks until the outputs are written. */
typedef struct bepucuda_body_shape {
    int32_t type;
    float a, b, c;
    float minimum_speculative_margin;   /* Collidable.MinimumSpeculativeMargin */
    float maximum_speculative_margin;   /* Collidable.MaximumSpeculativeMargin */
    int32_t allow_expansion_beyond_speculative_margin;  /* Collidable.Continuity.AllowExpansionBeyondSpeculativeMargin */
    int32_t reserved;
} bepucuda_body_shape;
typedef struct bepucuda_body_activity {
    float sleep_threshold;
    uint8_t minimum_timesteps_under_threshold;
    uint8_t timesteps_under_threshold_count;
    uint8_t sleep_candidate;
    uint8_t reserved;
} bepucuda_body_activity;
int32_t bepucuda_set_body_shapes(bepucuda_ctx* ctx, const bepucuda_body_shape* shapes, int32_t body_count);
int32_t bepucuda_predict_bounding_boxes(bepucuda_ctx* ctx, float dt, bepucuda_body_activity* activities, float* bounds_out);

/* PredictBoundingBoxes for every built-in shape type: the reference's Shapes batches are uploaded once as a library, and each active body names its
 * shape with the reference's TypedIndex. Whichever of bepucuda_set_body_shapes / bepucuda_set_body_collidables was called last decides what
 * bepucuda_predict_bounding_boxes computes; its signature, its activity update and its output format are the same for both.
 *   Sphere (0), Capsule (1), Box (2), Cylinder (4) and Triangle (3, TriangleWide.GetBounds, Collidables/Triangle.cs:L203-221) and ConvexHull (5,
 *   ConvexHullWide.GetBounds, ConvexHull.cs:L319-364) go through ExecuteConvexBatch (Collidables/BoundingBoxBatcher.cs:L142-223). Compound (6) and
 *   BigCompound (7) go through ExecuteCompoundBatch (L268-287) and Compound.AddChildBoundsToBatcher (Compound.cs:L198-221): every child is bounded
 *   like a convex body with the parent's margins and the child's pose and velocity, and the children's boxes and margins are merged. Mesh (8)
 *   goes through ExecuteHomogeneousCompoundBatch (L225-266) and Mesh.ComputeBounds (Mesh.cs:L232-255).
 *   Results are bit-identical to a non-contracting fp32 evaluation of the reference's expressions, including the sign of a zero that ties in a
 *   min / max fold, with one documented exception: the reference merges a compound's children in the order its batcher flushes them (grouped by
 *   child type, 16 per flush, shared across bodies), which depends on the other bodies of the frame; this library merges them in child order. The
 *   two agree except for the sign of a zero coordinate on which two children tie.
 *   A body whose shape does not exist (bit 31 of the TypedIndex clear) or has a type id above 8 (a user-registered shape) gets valid = 0; its
 *   activity is still updated. */
typedef struct bepucuda_hull {
    int32_t first_bundle;   /* into hull_points, in bundles */
    int32_t bundle_count;   /* ConvexHull.Points.Length, >= 1 */
} bepucuda_hull;
typedef struct bepucuda_compound {
    int32_t first_child;    /* into compound_children */
    int32_t child_count;    /* Compound.Children.Length / BigCompound.Children.Length, >= 1 */
} bepucuda_compound;
typedef struct bepucuda_compound_child {  /* CompoundChild (Compound.cs:L18-31), 32 B */
    float local_orientation[4];           /* Quaternion x, y, z, w */
    float local_position[3];
    uint32_t shape;                       /* TypedIndex.Packed; types 0-5 only */
} bepucuda_compound_child;
typedef struct bepucuda_mesh {
    int64_t first_triangle;   /* into mesh_triangles, in triangles */
    int32_t triangle_count;   /* Mesh.Triangles.Length, >= 1 */
    float scale[3];           /* Mesh.Scale */
} bepucuda_mesh;
/* The shape library. Primitive batches are the reference's ShapeBatch<T>.shapes memory as it is: Sphere {Radius}, Capsule {Radius, HalfLength},
 * Box {HalfWidth, HalfHeight, HalfLength}, Triangle {A, B, C} (36 B), Cylinder {Radius, HalfLength}; index i of a batch is TypedIndex.Index.
 * hull_points: the Vector3Wide bundles of every hull back to back (ConvexHull.Points memory: per bundle W x floats, W y floats, W z floats; the
 * last bundle padded by repeating the last point, ConvexHullHelper.cs:L1050-1062), hull_bundle_width = W = Vector<float>.Count of the process that
 * built them (4, 8 or 16). compound_children: the children of every compound and big compound back to back. mesh_triangles: the Triangle records
 * of every mesh back to back. A pointer may be NULL when its count is 0. Host buffers are only read during the call. */
typedef struct bepucuda_shape_library {
    const float* spheres;
    const float* capsules;
    const float* boxes;
    const float* triangles;
    const float* cylinders;
    const float* hull_points;
    const bepucuda_hull* hulls;
    const bepucuda_compound_child* compound_children;
    const bepucuda_compound* compounds;
    const bepucuda_compound* big_compounds;
    const float* mesh_triangles;
    const bepucuda_mesh* meshes;
    int64_t sphere_count, capsule_count, box_count, triangle_count, cylinder_count;
    int64_t hull_bundle_width, hull_bundle_total, hull_count;
    int64_t compound_child_total, compound_count, big_compound_count;
    int64_t mesh_triangle_total, mesh_count;
} bepucuda_shape_library;
/* One per active body: the reference's Collidable (Collidable.cs:L115-152). */
typedef struct bepucuda_body_collidable {
    uint32_t shape;                                     /* TypedIndex.Packed: bit 31 exists, bits 24-30 type, bits 0-23 index */
    float minimum_speculative_margin;                   /* Collidable.MinimumSpeculativeMargin */
    float maximum_speculative_margin;                   /* Collidable.MaximumSpeculativeMargin */
    int32_t allow_expansion_beyond_speculative_margin;  /* Collidable.Continuity.AllowExpansionBeyondSpeculativeMargin */
} bepucuda_body_collidable;
/* Validates and uploads the library (index ranges of every hull, compound, child and mesh inside their pools, no empty hull / compound / mesh,
 * compound children of types 0-5 with indices in range, W in {4, 8, 16} when there are hulls). Call again when shapes change; the body
 * collidables must then be set again before the next prediction. */
int32_t bepucuda_set_shape_library(bepucuda_ctx* ctx, const bepucuda_shape_library* library);
/* Validates every existing built-in shape index against the library and builds the per-class work lists (hulls, compounds, meshes and the
 * chunks of large meshes). body_count must equal the uploaded body count when bepucuda_predict_bounding_boxes runs. */
int32_t bepucuda_set_body_collidables(bepucuda_ctx* ctx, const bepucuda_body_collidable* collidables, int32_t body_count);

/* Device-side batch colouring (SURVEY.md §8 f3). Replaces, for a whole constraint set at once, the batch search Solver.Add runs per constraint
 * (Solver.cs:L1182-1199: the first batch whose referenced-handle set holds none of the constraint's dynamic bodies; kinematic references never
 * block, GetBlockingBodyHandles L1058-1078; index == fallback_batch_threshold is the fallback batch and accepts everything, TryAllocateInBatch
 * L1093-1140; the narrow phase's FindCandidateBatch L984-1014 is the same search). The result is IDENTICAL to running that first-fit search
 * sequentially over the constraints in ascending key order:
 *   BEPUCUDA_COLOR_INSERTION_ORDER  key = constraint index: the batches the reference's Solver.Add sequence produces from an empty solver;
 *   BEPUCUDA_COLOR_HASHED_ORDER     key = (bepucuda_color_hash(index) << 32) | index: a fixed pseudo-random order, which bounds the number of
 *                                   dependent device rounds by O(log n) on bounded-degree constraint graphs (insertion order can chain);
 *   BEPUCUDA_COLOR_BY_PRIORITY      key = (priorities[index] << 32) | index. With priorities = the constraints' CURRENT batch indices no
 *                                   constraint moves to a higher batch and none could move lower afterwards: the fixed point the reference's
 *                                   BatchCompressor (BatchCompressor.cs:L233) approaches a few constraints per frame.
 * encoded_body_references: [constraint][slot] with `bodies_per_constraint` (1..4) slots per constraint: active-set body index, bit 30 set for a
 * kinematic body (Bodies_GatherScatter.cs:L107-139), -1 for an unused slot. body_count bounds the indices. batch_indices_out[i] receives the batch
 * of constraint i (0 .. fallback_batch_threshold), *batch_count_out the number of batches, *rounds_out the dependent device rounds it took
 * (both optional). Host buffers are caller-owned and only used during the call, which blocks until the result is written. */
#define BEPUCUDA_COLOR_INSERTION_ORDER 0
#define BEPUCUDA_COLOR_HASHED_ORDER 1
#define BEPUCUDA_COLOR_BY_PRIORITY 2
int32_t bepucuda_color_constraints(bepucuda_ctx* ctx, int32_t constraint_count, int32_t bodies_per_constraint, const int32_t* encoded_body_references,
                                   int32_t body_count, int32_t fallback_batch_threshold, int32_t order, const uint32_t* priorities,
                                   int32_t* batch_indices_out, int32_t* batch_count_out, int32_t* rounds_out);
/* The hash behind BEPUCUDA_COLOR_HASHED_ORDER: h = i * 0x9E3779B1; h ^= h >> 15; h *= 0x85EBCA77; h ^= h >> 13; h *= 0xC2B2AE3D; h ^= h >> 16 (uint32). */
uint32_t bepucuda_color_hash(uint32_t constraint_index);

/* Multi-GPU, one constraint graph over several contexts (SURVEY.md §8e; replaces the reference's multithreaded batch dispatch,
 * Solver_Solve.cs:L458-654, where workers split the constraints of a batch). Every participating context ("rank": one per GPU, normally one per
 * process) is given the WHOLE body set and the same batch layout, but only its share of the constraints (lanes of other ranks are empty, body
 * reference -1). Within a batch no dynamic body is referenced twice, so exactly one rank writes a given body in a given (batch, stage); after every
 * WarmStart / Solve stage the library packs the records this rank wrote (velocity; pose and world inertia too when the lane integrated) into a
 * zero-initialised staging buffer with a "valid" word, calls `exchange` to all-reduce it, and writes every valid record back, which keeps all
 * ranks' body arrays bit-identical to a single-context solve. At bepucuda_end_constraints the per-body integration owner (lowest batch referencing
 * the body) and the constrained-body mask are combined the same way.
 *   exchange(user, device_words, count, op, cuda_stream): combine `count` int32 words at `device_words` element-wise across all ranks, in place, as
 *   stream-ordered work on `cuda_stream` (e.g. ncclAllReduce with ncclInt32 and ncclSum for op 0 / ncclMin for op 1); return 0, or non-zero to fail
 *   the call that invoked it. With op 0 at most one rank contributes a non-zero word, so an integer sum transports bit patterns exactly.
 * Requirements: BEPUCUDA_EXEC_STREAM, AngularIntegrationMode.Nonconserving; call before bepucuda_begin_constraints. `body_indices` / `count` name the
 * bodies other ranks may also reference; NULL / 0 means "all of them" (the only form implemented: the list is accepted and ignored).
 * Passing exchange = NULL returns the context to single-rank operation. */
typedef int32_t (*bepucuda_exchange_fn)(void* user, void* device_words, int64_t count, int32_t op, void* cuda_stream);
int32_t bepucuda_set_boundary_bodies(bepucuda_ctx* ctx, const int32_t* body_indices, int32_t count,
                                     bepucuda_exchange_fn exchange, void* user);

/* Multi-GPU, ONE constraint graph over several GPUs with direct NVLink peer stores (SURVEY.md §8e; the fast successor of the callback path above).
 * Bodies are partitioned into owner slabs by the host; every rank (one context per GPU, normally one process per GPU) uploads ALL bodies (only
 * its own slab and the halo it references are kept current) and ONLY ITS OWN constraints, compacted, under their original batch indices. After
 * every WarmStart / Solve stage a rank copies the records its stage wrote for bodies other ranks also reference straight into those ranks' body
 * arrays (peer memory opened from CUDA IPC handles) and all ranks meet at a flag barrier in peer memory: no host round trip, no collective library.
 * Within a batch no dynamic body is referenced twice, so exactly one rank writes a given body in a given stage, and every rank's copy of a body
 * it references is bit-identical to the single-GPU solve at every stage.
 *   bepucuda_shard_export: IPC handles of this context's pose / velocity / world-inertia arrays and of its flag block (call after
 *     bepucuda_upload_bodies; the arrays must not be re-allocated afterwards, i.e. keep the body count).
 *   bepucuda_shard_import: this rank's index, the rank count (<= 8) and every rank's exported handles, in rank order.
 *   bepucuda_shard_set_global: per body, the lowest batch index that references it as a dynamic body on ANY rank (INT32_MAX if none) -- the owner of
 *     its integration, Solver_Solve.cs:L951-1044 -- and whether any rank constrains it (final pose pass, PoseIntegrator.cs:L537-693).
 *   bepucuda_shard_set_pushes: for one batch, the (body, destination rank) pairs of the bodies THIS rank's constraints of that batch write and the
 *     destination rank also references; owner_flags[i] != 0 when this batch integrates the body (pose and world inertia travel too in WarmStart).
 *     These lists are copied by the one-CTA exchange kernel that follows the stage.
 *   bepucuda_shard_set_body_masks (preferred, replaces the push lists): rank_masks[body] has bit r set when rank r references the body. The stage
 *     kernels then store a written record into the other referencing ranks' arrays themselves, from the registers of the lane that computed it,
 *     and the exchange kernel is only the flag barrier. NULL returns to the push lists.
 * Call order: upload_bodies, shard_export, (exchange handles), shard_import, shard_set_global, shard_set_body_masks | (begin_constraints ...
 * shard_set_pushes ...), end_constraints. Every rank must have finished uploading a frame's bodies before any rank's bepucuda_solve can complete
 * its first stage: the solve starts with a rank barrier, so issuing upload and solve on each rank in that order is enough. The sequential fallback batch is not supported across ranks (BEPUCUDA_ERR_BAD_STATE). BEPUCUDA_EXEC_GRAPH or _STREAM. */
typedef struct bepucuda_ipc_handles {
    unsigned char bytes[4][64];
} bepucuda_ipc_handles;
int32_t bepucuda_shard_export(bepucuda_ctx* ctx, bepucuda_ipc_handles* out);
int32_t bepucuda_shard_import(bepucuda_ctx* ctx, int32_t rank, int32_t rank_count, const bepucuda_ipc_handles* all_ranks);
/* The same for ranks that live in ONE process (one host thread per context): the other ranks' arrays are taken from their contexts directly
 * (peer access is enabled between different devices) instead of through IPC handles. all_ranks[rank] must be ctx itself. */
int32_t bepucuda_shard_import_contexts(bepucuda_ctx* ctx, int32_t rank, int32_t rank_count, bepucuda_ctx* const* all_ranks);
int32_t bepucuda_shard_set_global(bepucuda_ctx* ctx, const int32_t* first_batch_per_body, const uint8_t* constrained_per_body);
int32_t bepucuda_shard_set_pushes(bepucuda_ctx* ctx, int32_t batch_index, int32_t count, const int32_t* body_indices, const int32_t* destination_ranks,
                                  const int32_t* owner_flags);
int32_t bepucuda_shard_set_body_masks(bepucuda_ctx* ctx, const uint8_t* rank_masks);

#ifdef __cplusplus
}
#endif
#endif /* BEPUCUDA_H */
