// P/Invoke surface of libbepucuda (include/bepucuda.h). Not compiled in this repository (no .NET toolchain in the build image); it is the
// binding a bepuphysics2 maintainer adds next to their application. Every entry point replaces the reference call cited in the header.
using System;
using System.Runtime.InteropServices;

namespace BepuCuda
{
    [StructLayout(LayoutKind.Sequential)] public unsafe struct IpcHandles { public fixed byte Bytes[256]; }
    [StructLayout(LayoutKind.Sequential)]
    public unsafe struct Config { public int DeviceOrdinal, StrictFp, ExecutionMode; public fixed int Reserved[5]; }

    [StructLayout(LayoutKind.Sequential)]
    public unsafe struct IntegratorDesc
    {
        public fixed float Gravity[3];
        public float LinearDamping, AngularDamping;
        public int AngularIntegrationMode, AllowSubstepsForUnconstrained, IntegrateVelocityForKinematics;
    }

    [StructLayout(LayoutKind.Sequential)]
    public struct Timings
    {
        public float SolveMs, UploadMs, DownloadMs;
        public long ConstraintCount, ConstraintIterations, StageCount, KernelLaunches, AlgorithmicBytes, H2DBytes, D2HBytes;
        public int DeviceBatchCount, FallbackLevelCount;
    }

    [StructLayout(LayoutKind.Sequential)]
    public unsafe struct StageProfile
    {
        public fixed float Ms[8];
        public fixed long Launches[8];
        public fixed long AlgorithmicBytes[8];
    }

    // bepucuda_set_shape_library / bepucuda_set_body_collidables. The pools are the reference's own memory: ShapeBatch<T>.shapes.Memory for the
    // primitive batches (Sphere, Capsule, Box, Triangle, Cylinder), ConvexHull.Points, Compound.Children / BigCompound.Children (CompoundChild, 32 B),
    // Mesh.Triangles; hulls, compounds and meshes are gathered back to back into one pool per kind.
    [StructLayout(LayoutKind.Sequential)] public struct HullRange { public int FirstBundle, BundleCount; }
    [StructLayout(LayoutKind.Sequential)] public struct CompoundRange { public int FirstChild, ChildCount; }
    [StructLayout(LayoutKind.Sequential)]
    public unsafe struct MeshRange { public long FirstTriangle; public int TriangleCount; public fixed float Scale[3]; }
    [StructLayout(LayoutKind.Sequential)]
    public unsafe struct ShapeLibrary
    {
        public float* Spheres, Capsules, Boxes, Triangles, Cylinders, HullPoints;
        public HullRange* Hulls;
        public void* CompoundChildren;  // BepuPhysics.Collidables.CompoundChild*
        public CompoundRange* Compounds, BigCompounds;
        public float* MeshTriangles;
        public MeshRange* Meshes;
        public long SphereCount, CapsuleCount, BoxCount, TriangleCount, CylinderCount, HullBundleWidth, HullBundleTotal, HullCount;
        public long CompoundChildTotal, CompoundCount, BigCompoundCount, MeshTriangleTotal, MeshCount;
    }
    [StructLayout(LayoutKind.Sequential)]
    public struct BodyCollidable { public uint Shape; public float MinimumSpeculativeMargin, MaximumSpeculativeMargin; public int AllowExpansionBeyondSpeculativeMargin; }

    [UnmanagedFunctionPointer(CallingConvention.Cdecl)]
    public unsafe delegate int ExchangeFn(void* user, void* deviceWords, long count, int op, void* cudaStream);

    public static unsafe class Native
    {
        const string Lib = "bepucuda";
        [DllImport(Lib)] public static extern int bepucuda_create(Config* cfg, IntPtr* ctx);
        [DllImport(Lib)] public static extern int bepucuda_destroy(IntPtr ctx);
        [DllImport(Lib)] public static extern IntPtr bepucuda_last_error(IntPtr ctx);
        [DllImport(Lib)] public static extern int bepucuda_type_info(int typeId, int* bodies, int* prestepFloats, int* impulseFloats);
        [DllImport(Lib)] public static extern int bepucuda_host_register(IntPtr ctx, void* ptr, long bytes);
        [DllImport(Lib)] public static extern int bepucuda_host_unregister(IntPtr ctx, void* ptr);
        [DllImport(Lib)] public static extern int bepucuda_set_solve_description(IntPtr ctx, int substepCount, int* velocityIterationsPerSubstep, int fallbackBatchThreshold);
        [DllImport(Lib)] public static extern int bepucuda_set_integrator(IntPtr ctx, IntegratorDesc* desc);
        [DllImport(Lib)] public static extern int bepucuda_upload_bodies(IntPtr ctx, void* bodyDynamics, int bodyCount);
        [DllImport(Lib)] public static extern int bepucuda_begin_constraints(IntPtr ctx, int sourceBundleWidth, int batchCount);
        [DllImport(Lib)] public static extern int bepucuda_upload_type_batch(IntPtr ctx, int batchIndex, int typeBatchIndex, int typeId, int constraintCount, void* bodyReferences, void* prestep, void* accumulatedImpulses);
        [DllImport(Lib)] public static extern int bepucuda_set_constrained_kinematics(IntPtr ctx, int* bodyIndices, int count);
        [DllImport(Lib)] public static extern int bepucuda_end_constraints(IntPtr ctx);
        [DllImport(Lib)] public static extern int bepucuda_update_type_batch(IntPtr ctx, int batchIndex, int typeBatchIndex, void* prestep, void* accumulatedImpulses);
        [DllImport(Lib)] public static extern int bepucuda_set_contact_features(IntPtr ctx, int batchIndex, int typeBatchIndex, int* featureIds);
        [DllImport(Lib)] public static extern int bepucuda_update_contacts(IntPtr ctx, int batchIndex, int typeBatchIndex, void* prestep, int* newFeatureIds);
        [DllImport(Lib)] public static extern int bepucuda_upload_body_motion(IntPtr ctx, void* bodyDynamics, int bodyCount);
        [DllImport(Lib)] public static extern int bepucuda_download_body_motion(IntPtr ctx, void* bodyDynamicsOut, int bodyCount);
        [DllImport(Lib)] public static extern int bepucuda_solve(IntPtr ctx, float dt);
        [DllImport(Lib)] public static extern int bepucuda_synchronize(IntPtr ctx);
        [DllImport(Lib)] public static extern int bepucuda_download_bodies(IntPtr ctx, void* bodyDynamicsOut, int bodyCount);
        [DllImport(Lib)] public static extern int bepucuda_download_impulses(IntPtr ctx);
        [DllImport(Lib)] public static extern int bepucuda_download_prestep(IntPtr ctx, int batchIndex, int typeBatchIndex, float* prestepOut);
        [DllImport(Lib)] public static extern int bepucuda_get_timings(IntPtr ctx, Timings* timings);
        [DllImport(Lib)] public static extern int bepucuda_event_record(IntPtr ctx, int slot);
        [DllImport(Lib)] public static extern int bepucuda_event_elapsed_ms(IntPtr ctx, int slotBegin, int slotEnd, float* ms);
        [DllImport(Lib)] public static extern int bepucuda_profile_stages(IntPtr ctx, float dt, StageProfile* profile);
        [DllImport(Lib)] public static extern int bepucuda_shard_export(IntPtr ctx, IpcHandles* handles);
        [DllImport(Lib)] public static extern int bepucuda_shard_import(IntPtr ctx, int rank, int rankCount, IpcHandles* allRanks);
        [DllImport(Lib)] public static extern int bepucuda_shard_set_global(IntPtr ctx, int* firstBatchPerBody, byte* constrainedPerBody);
        [DllImport(Lib)] public static extern int bepucuda_shard_set_pushes(IntPtr ctx, int batchIndex, int count, int* bodyIndices, int* destinationRanks, int* ownerFlags);
        [DllImport(Lib)] public static extern int bepucuda_shard_set_body_masks(IntPtr ctx, byte* rankMasks);
        [DllImport(Lib)] public static extern int bepucuda_shard_import_contexts(IntPtr ctx, int rank, int rankCount, IntPtr* allRanks);
        /// <summary>PredictBoundingBoxes on the device: sleep candidacy + bounds and speculative margins of sphere / capsule / box / cylinder bodies from the resident body state.</summary>
        [DllImport(Lib)] public static extern int bepucuda_set_body_shapes(IntPtr ctx, BodyShape* shapes, int bodyCount);
        [DllImport(Lib)] public static extern int bepucuda_predict_bounding_boxes(IntPtr ctx, float dt, BodyActivity* activities, float* boundsOut);
        [DllImport(Lib)] public static extern int bepucuda_set_shape_library(IntPtr ctx, ShapeLibrary* library);
        [DllImport(Lib)] public static extern int bepucuda_set_body_collidables(IntPtr ctx, BodyCollidable* collidables, int bodyCount);
        /// <summary>Device-side batch colouring: the batch Solver.Add's first-fit search would pick for every constraint of a list (order 0 = add order, 1 = hashed, 2 = priorities).</summary>
        [DllImport(Lib)] public static extern int bepucuda_color_constraints(IntPtr ctx, int constraintCount, int bodiesPerConstraint, int* encodedBodyReferences, int bodyCount, int fallbackBatchThreshold, int order, uint* priorities, int* batchIndicesOut, int* batchCountOut, int* roundsOut);
        [DllImport(Lib)] public static extern uint bepucuda_color_hash(uint constraintIndex);
        [DllImport(Lib)] public static extern int bepucuda_set_boundary_bodies(IntPtr ctx, int* bodyIndices, int count, ExchangeFn exchange, void* user);
    }
}
