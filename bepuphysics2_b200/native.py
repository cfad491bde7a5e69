"""ctypes view of the C ABI (include/bepucuda.h) and of the C++ host mirror (csrc/host/bepu_host.cpp).

Class names follow the reference: `Simulation` (BepuPhysics/Simulation.cs) owns `Bodies` + `Solver` state in the reference's own
buffer layouts; `CudaTimestepper` is the ITimestepper (BepuPhysics/ITimestepper.cs:L15-34) whose Solve slot runs on the GPU.
"""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_LIBS = None


class BepuCudaError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("bepucuda error %d: %s" % (code, message))
        self.code = code


class IntegratorDesc(C.Structure):
    """bepucuda_integrator_desc — declarative IPoseIntegratorCallbacks (Demos/DemoCallbacks.cs:L12-105)."""

    _fields_ = [
        ("gravity", C.c_float * 3),
        ("linear_damping", C.c_float),
        ("angular_damping", C.c_float),
        ("angular_integration_mode", C.c_int32),
        ("allow_substeps_for_unconstrained", C.c_int32),
        ("integrate_velocity_for_kinematics", C.c_int32),
    ]

    @staticmethod
    def default():
        d = IntegratorDesc()
        d.gravity[0], d.gravity[1], d.gravity[2] = 0.0, -10.0, 0.0
        d.linear_damping = 0.03
        d.angular_damping = 0.03
        return d


class Config(C.Structure):
    _fields_ = [("device_ordinal", C.c_int32), ("strict_fp", C.c_int32), ("execution_mode", C.c_int32), ("reserved", C.c_int32 * 5)]


class Timings(C.Structure):
    _fields_ = [
        ("solve_ms", C.c_float),
        ("upload_ms", C.c_float),
        ("download_ms", C.c_float),
        ("constraint_count", C.c_int64),
        ("constraint_iterations", C.c_int64),
        ("stage_count", C.c_int64),
        ("kernel_launches", C.c_int64),
        ("algorithmic_bytes", C.c_int64),
        ("h2d_bytes", C.c_int64),
        ("d2h_bytes", C.c_int64),
        ("device_batch_count", C.c_int32),
        ("fallback_level_count", C.c_int32),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


class TypeBatchView(C.Structure):
    _fields_ = [
        ("type_id", C.c_int32),
        ("constraint_count", C.c_int32),
        ("bodies", C.c_int32),
        ("prestep_rows", C.c_int32),
        ("impulse_rows", C.c_int32),
        ("bundle_count", C.c_int32),
        ("body_references", C.POINTER(C.c_int32)),
        ("prestep", C.POINTER(C.c_float)),
        ("accumulated_impulses", C.POINTER(C.c_float)),
    ]


class StageProfile(C.Structure):
    _fields_ = [("ms", C.c_float * 8), ("launches", C.c_int64 * 8), ("algorithmic_bytes", C.c_int64 * 8)]

    STAGE_NAMES = ["warm_start_first", "warm_start", "solve", "incremental_update", "kinematic_first", "kinematic", "final_pose", "unused"]

    def as_dict(self):
        return {n: {"ms": self.ms[i], "launches": self.launches[i], "algorithmic_bytes": self.algorithmic_bytes[i]} for i, n in enumerate(self.STAGE_NAMES) if self.launches[i]}


EXEC_GRAPH, EXEC_STREAM = 0, 2  # 1 and 3 (persistent / dataflow kernels) were removed: slower than the graph on every configuration

# Every symbol include/bepucuda.h declares (checked by the CPU test-suite).
C_ABI_SYMBOLS = [
    "bepucuda_create", "bepucuda_destroy", "bepucuda_last_error", "bepucuda_type_info", "bepucuda_host_register", "bepucuda_host_unregister",
    "bepucuda_set_solve_description", "bepucuda_set_integrator", "bepucuda_upload_bodies", "bepucuda_begin_constraints", "bepucuda_upload_type_batch",
    "bepucuda_set_constrained_kinematics", "bepucuda_end_constraints", "bepucuda_update_type_batch", "bepucuda_solve", "bepucuda_synchronize",
    "bepucuda_download_bodies", "bepucuda_download_impulses", "bepucuda_download_prestep", "bepucuda_get_timings", "bepucuda_set_boundary_bodies",
    "bepucuda_event_record", "bepucuda_event_elapsed_ms", "bepucuda_profile_stages",
    "bepucuda_set_contact_features", "bepucuda_update_contacts", "bepucuda_upload_body_motion", "bepucuda_download_body_motion",
    "bepucuda_shard_export", "bepucuda_shard_import", "bepucuda_shard_set_global", "bepucuda_shard_set_pushes", "bepucuda_shard_set_body_masks", "bepucuda_shard_import_contexts",
    "bepucuda_color_constraints", "bepucuda_color_hash", "bepucuda_set_body_shapes", "bepucuda_predict_bounding_boxes",
    "bepucuda_set_shape_library", "bepucuda_set_body_collidables",
]


# bepucuda_body_shape / bepucuda_body_activity (include/bepucuda.h) as numpy record types
BODY_SHAPE_DTYPE = np.dtype([("type", "<i4"), ("a", "<f4"), ("b", "<f4"), ("c", "<f4"), ("minimum_speculative_margin", "<f4"), ("maximum_speculative_margin", "<f4"),
                             ("allow_expansion_beyond_speculative_margin", "<i4"), ("reserved", "<i4")])
BODY_ACTIVITY_DTYPE = np.dtype([("sleep_threshold", "<f4"), ("minimum_timesteps_under_threshold", "u1"), ("timesteps_under_threshold_count", "u1"), ("sleep_candidate", "u1"),
                                ("reserved", "u1")])
SHAPE_SPHERE, SHAPE_CAPSULE, SHAPE_BOX, SHAPE_CYLINDER = 0, 1, 2, 4  # Sphere.Id, Capsule.Id, Box.Id, Cylinder.Id of the reference
SHAPE_TRIANGLE, SHAPE_CONVEX_HULL, SHAPE_COMPOUND, SHAPE_BIG_COMPOUND, SHAPE_MESH = 3, 5, 6, 7, 8

# bepucuda_shape_library's record types and bepucuda_body_collidable (include/bepucuda.h)
HULL_DTYPE = np.dtype([("first_bundle", "<i4"), ("bundle_count", "<i4")])
COMPOUND_DTYPE = np.dtype([("first_child", "<i4"), ("child_count", "<i4")])
COMPOUND_CHILD_DTYPE = np.dtype([("local_orientation", "<f4", 4), ("local_position", "<f4", 3), ("shape", "<u4")])  # CompoundChild, 32 B
MESH_DTYPE = np.dtype([("first_triangle", "<i8"), ("triangle_count", "<i4"), ("scale", "<f4", 3)])
BODY_COLLIDABLE_DTYPE = np.dtype([("shape", "<u4"), ("minimum_speculative_margin", "<f4"), ("maximum_speculative_margin", "<f4"),
                                  ("allow_expansion_beyond_speculative_margin", "<i4")])


def typed_index(shape_type, index):
    """TypedIndex.Packed (TypedIndex.cs:L45-51): bit 31 set, type in bits 24-30, index in bits 0-23. Works elementwise on arrays."""
    return ((np.asarray(shape_type, dtype=np.uint32) << np.uint32(24)) | np.asarray(index, dtype=np.uint32) | np.uint32(1 << 31)).astype(np.uint32)


class ShapeLibraryDesc(C.Structure):
    """bepucuda_shape_library."""
    _fields_ = [(n, C.c_void_p) for n in ("spheres", "capsules", "boxes", "triangles", "cylinders", "hull_points", "hulls", "compound_children", "compounds", "big_compounds",
                                          "mesh_triangles", "meshes")] + \
               [(n, C.c_int64) for n in ("sphere_count", "capsule_count", "box_count", "triangle_count", "cylinder_count", "hull_bundle_width", "hull_bundle_total", "hull_count",
                                         "compound_child_total", "compound_count", "big_compound_count", "mesh_triangle_total", "mesh_count")]


class ShapeLibrary:
    """The reference's Shapes batches, flattened as bepucuda_set_shape_library takes them. Primitive batches are float arrays of one record per
    shape: spheres [n] (Radius), capsules [n, 2] (Radius, HalfLength), boxes [n, 3], triangles [n, 9] (A, B, C), cylinders [n, 2]. hull_points
    [bundles, 3, W] holds the Vector3Wide bundles of every hull (ConvexHull.Points), hulls / compounds / big_compounds / meshes are HULL_DTYPE /
    COMPOUND_DTYPE / MESH_DTYPE records indexing hull_points / compound_children (COMPOUND_CHILD_DTYPE) / mesh_triangles [n, 9]."""

    def __init__(self, spheres=(), capsules=(), boxes=(), triangles=(), cylinders=(), hull_points=None, hull_bundle_width=8, hulls=(), compound_children=(),
                 compounds=(), big_compounds=(), mesh_triangles=(), meshes=()):
        f = lambda a, k: np.ascontiguousarray(np.asarray(a, dtype=np.float32).reshape(-1, k) if k > 1 else np.asarray(a, dtype=np.float32).reshape(-1))
        self.spheres, self.capsules, self.boxes, self.triangles, self.cylinders = f(spheres, 1), f(capsules, 2), f(boxes, 3), f(triangles, 9), f(cylinders, 2)
        self.hull_bundle_width = int(hull_bundle_width)
        self.hull_points = np.ascontiguousarray(np.zeros((0, 3, self.hull_bundle_width), np.float32) if hull_points is None else np.asarray(hull_points, dtype=np.float32))
        r = lambda a, dtype: np.ascontiguousarray(np.zeros(0, dtype) if len(a) == 0 else a.astype(dtype) if isinstance(a, np.ndarray) else np.array(list(a), dtype=dtype)).reshape(-1)
        self.hulls = r(hulls, HULL_DTYPE)
        self.compound_children = r(compound_children, COMPOUND_CHILD_DTYPE)
        self.compounds, self.big_compounds = r(compounds, COMPOUND_DTYPE), r(big_compounds, COMPOUND_DTYPE)
        self.mesh_triangles = f(mesh_triangles, 9)
        self.meshes = r(meshes, MESH_DTYPE)

    def desc(self):
        """The bepucuda_shape_library pointing into this object's arrays (valid while the object lives)."""
        d = ShapeLibraryDesc()
        for name in ("spheres", "capsules", "boxes", "triangles", "cylinders", "hull_points", "hulls", "compound_children", "compounds", "big_compounds", "mesh_triangles", "meshes"):
            a = getattr(self, name)
            setattr(d, name, a.ctypes.data if a.size else None)
        d.sphere_count, d.capsule_count, d.box_count = len(self.spheres), len(self.capsules), len(self.boxes)
        d.triangle_count, d.cylinder_count = len(self.triangles), len(self.cylinders)
        d.hull_bundle_width, d.hull_bundle_total, d.hull_count = self.hull_bundle_width, self.hull_points.shape[0], len(self.hulls)
        d.compound_child_total, d.compound_count, d.big_compound_count = len(self.compound_children), len(self.compounds), len(self.big_compounds)
        d.mesh_triangle_total, d.mesh_count = len(self.mesh_triangles), len(self.meshes)
        return d

    def count(self, shape_type):
        return len([self.spheres, self.capsules, self.boxes, self.triangles, self.cylinders, self.hulls, self.compounds, self.big_compounds, self.meshes][shape_type])

EXCHANGE_FN = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p)


def load_libraries():
    """Loads libbepucuda.so and libbepuhost.so from the package directory. Fails loudly if they are missing: there is no fallback."""
    global _LIBS
    if _LIBS is not None:
        return _LIBS
    variant = os.environ.get("BEPUCUDA_VARIANT")  # development A/B builds only (see _build.py)
    cuda_path = os.path.join(HERE, "libbepucuda_%s.so" % variant if variant else "libbepucuda.so")
    host_path = os.path.join(HERE, "libbepuhost.so")
    for p in (cuda_path, host_path):
        if not os.path.exists(p):
            raise ImportError("%s is missing: run `python -m bepuphysics2_b200._build` (or __graft_entry__.build()); there is no CPU fallback" % p)
    if not variant:
        from . import _build

        if _build.binary_matches_stamp(cuda_path) is False:
            raise ImportError("%s does not match the hash recorded in its stamp (a stale or foreign binary): rebuild with `python -m bepuphysics2_b200._build --force`" % cuda_path)
    cuda = C.CDLL(cuda_path, mode=C.RTLD_GLOBAL)
    host = C.CDLL(host_path)
    vp, i32, f32 = C.c_void_p, C.c_int32, C.c_float
    cuda.bepucuda_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    cuda.bepucuda_destroy.argtypes = [vp]
    cuda.bepucuda_last_error.argtypes = [vp]
    cuda.bepucuda_last_error.restype = C.c_char_p
    cuda.bepucuda_type_info.argtypes = [i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    cuda.bepucuda_get_timings.argtypes = [vp, C.POINTER(Timings)]
    cuda.bepucuda_solve.argtypes = [vp, f32]
    cuda.bepucuda_set_boundary_bodies.argtypes = [vp, vp, i32, EXCHANGE_FN, vp]
    cuda.bepucuda_synchronize.argtypes = [vp]
    cuda.bepucuda_set_solve_description.argtypes = [vp, i32, C.POINTER(i32), i32]
    cuda.bepucuda_set_integrator.argtypes = [vp, C.POINTER(IntegratorDesc)]
    cuda.bepucuda_upload_bodies.argtypes = [vp, vp, i32]
    cuda.bepucuda_begin_constraints.argtypes = [vp, i32, i32]
    cuda.bepucuda_upload_type_batch.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp]
    cuda.bepucuda_set_constrained_kinematics.argtypes = [vp, vp, i32]
    cuda.bepucuda_end_constraints.argtypes = [vp]
    cuda.bepucuda_update_type_batch.argtypes = [vp, i32, i32, vp, vp]
    cuda.bepucuda_set_contact_features.argtypes = [vp, i32, i32, vp]
    cuda.bepucuda_update_contacts.argtypes = [vp, i32, i32, vp, vp]
    cuda.bepucuda_upload_body_motion.argtypes = [vp, vp, i32]
    cuda.bepucuda_download_body_motion.argtypes = [vp, vp, i32]
    cuda.bepucuda_download_bodies.argtypes = [vp, vp, i32]
    cuda.bepucuda_download_impulses.argtypes = [vp]
    cuda.bepucuda_download_prestep.argtypes = [vp, i32, i32, vp]
    cuda.bepucuda_event_record.argtypes = [vp, i32]
    cuda.bepucuda_event_elapsed_ms.argtypes = [vp, i32, i32, C.POINTER(f32)]
    cuda.bepucuda_profile_stages.argtypes = [vp, f32, C.POINTER(StageProfile)]
    cuda.bepucuda_host_register.argtypes = [vp, vp, C.c_int64]
    cuda.bepucuda_host_unregister.argtypes = [vp, vp]
    cuda.bepucuda_color_constraints.argtypes = [vp, i32, i32, vp, i32, i32, i32, vp, vp, C.POINTER(i32), C.POINTER(i32)]
    cuda.bepucuda_color_hash.argtypes = [C.c_uint32]
    cuda.bepucuda_set_body_shapes.argtypes = [vp, vp, i32]
    cuda.bepucuda_predict_bounding_boxes.argtypes = [vp, f32, vp, vp]
    cuda.bepucuda_set_shape_library.argtypes = [vp, C.POINTER(ShapeLibraryDesc)]
    cuda.bepucuda_set_body_collidables.argtypes = [vp, vp, i32]
    cuda.bepucuda_color_hash.restype = C.c_uint32

    host.bepuhost_create.restype = vp
    host.bepuhost_create.argtypes = [i32, i32]
    host.bepuhost_destroy.argtypes = [vp]
    host.bepuhost_last_error.argtypes = [vp]
    host.bepuhost_last_error.restype = C.c_char_p
    host.bepuhost_set_solve_description.argtypes = [vp, i32, C.POINTER(i32)]
    host.bepuhost_set_integrator.argtypes = [vp, C.POINTER(IntegratorDesc)]
    host.bepuhost_add_bodies.argtypes = [vp, vp, i32]
    host.bepuhost_body_dynamics.argtypes = [vp]
    host.bepuhost_body_dynamics.restype = C.POINTER(C.c_float)
    host.bepuhost_body_count.argtypes = [vp]
    host.bepuhost_add_constraints.argtypes = [vp, i32, i32, vp, vp]
    host.bepuhost_add_constraints_in_batches.argtypes = [vp, i32, i32, vp, vp, vp]
    host.bepuhost_export_constraint_references.argtypes = [vp, vp, vp]
    host.bepuhost_constraint_location.argtypes = [vp, i32, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    host.bepuhost_constraint_count.argtypes = [vp]
    host.bepuhost_batch_count.argtypes = [vp]
    host.bepuhost_type_batch_count.argtypes = [vp, i32]
    host.bepuhost_get_type_batch.argtypes = [vp, i32, i32, C.POINTER(TypeBatchView)]
    host.bepuhost_constrained_kinematic_count.argtypes = [vp]
    host.bepuhost_constrained_kinematics.argtypes = [vp]
    host.bepuhost_constrained_kinematics.restype = C.POINTER(i32)
    host.bepuhost_substep_count.argtypes = [vp]
    host.bepuhost_velocity_iterations.argtypes = [vp]
    host.bepuhost_velocity_iterations.restype = C.POINTER(i32)
    host.bepuhost_cuda_update_contacts.argtypes = [vp, vp, vp, i32]
    for name in ("bepuhost_cuda_describe", "bepuhost_cuda_refresh", "bepuhost_cuda_download_prestep", "bepuhost_cuda_register_buffers", "bepuhost_cuda_unregister_buffers"):
        getattr(host, name).argtypes = [vp, vp]
    host.bepuhost_cuda_solve.argtypes = [vp, vp, f32, i32]
    _LIBS = (cuda, host)
    return _LIBS


def type_info(type_id):
    """(bodies per constraint, prestep floats, accumulated impulse floats) of a constraint type id, or None if unsupported."""
    cuda, _ = load_libraries()
    b, p, d = C.c_int32(), C.c_int32(), C.c_int32()
    if cuda.bepucuda_type_info(type_id, C.byref(b), C.byref(p), C.byref(d)) != 0:
        return None
    return b.value, p.value, d.value


class TypeBatch:
    """A numpy view of one reference-layout type batch (Constraints/TypeBatch.cs:L10-27). Arrays alias the host mirror's memory."""

    def __init__(self, batch_index, type_batch_index, view, W):
        self.batch_index, self.type_batch_index = batch_index, type_batch_index
        self.type_id, self.constraint_count = view.type_id, view.constraint_count
        self.bodies, self.prestep_rows, self.impulse_rows, self.bundle_count = view.bodies, view.prestep_rows, view.impulse_rows, view.bundle_count
        n = view.bundle_count
        self.body_references = np.ctypeslib.as_array(view.body_references, shape=(n, view.bodies, W))
        self.prestep = np.ctypeslib.as_array(view.prestep, shape=(n, view.prestep_rows, W))
        self.accumulated_impulses = np.ctypeslib.as_array(view.accumulated_impulses, shape=(n, view.impulse_rows, W))
        self.view = view


class Simulation:
    """Host-side state in the reference's layouts: `bodies` is Bodies.ActiveSet.DynamicsState (n x 32 floats, BodyProperties.cs:L318-338),
    `type_batches()` walks Solver.ActiveSet.Batches[b].TypeBatches[t]. Constraint adds follow Solver.Add's greedy batch assignment."""

    def __init__(self, bundle_width=8, fallback_batch_threshold=64, substeps=1, velocity_iterations=1, integrator=None):
        _, self._host = load_libraries()
        self._sim = self._host.bepuhost_create(bundle_width, fallback_batch_threshold)
        if not self._sim:
            raise ValueError("bad bundle width / fallback threshold")
        self.bundle_width = bundle_width
        self.fallback_batch_threshold = fallback_batch_threshold
        self.set_solve_description(substeps, velocity_iterations)
        self.integrator = integrator or IntegratorDesc.default()
        self._host.bepuhost_set_integrator(self._sim, C.byref(self.integrator))

    def __del__(self):
        if getattr(self, "_sim", None):
            self._host.bepuhost_destroy(self._sim)
            self._sim = None

    def set_solve_description(self, substeps, velocity_iterations, velocity_iteration_scheduler=None):
        """SolveDescription(velocityIterationCount, substepCount); `velocity_iterations` may be a per-substep list (SolveDescription.cs:L21-38).
        With a `velocity_iteration_scheduler` (SubstepVelocityIterationScheduler) the per-substep counts are evaluated here, host-side, with the
        reference's rule: a scheduled count below 1 falls back to VelocityIterationCount (Solver_Solve.cs:L743-751)."""
        if velocity_iteration_scheduler is not None:
            assert np.isscalar(velocity_iterations)
            scheduled = [int(velocity_iteration_scheduler(i)) for i in range(substeps)]
            velocity_iterations = [velocity_iterations if n < 1 else n for n in scheduled]
        its = [velocity_iterations] * substeps if np.isscalar(velocity_iterations) else list(velocity_iterations)
        assert len(its) == substeps
        self.velocity_iterations = its
        arr = (C.c_int32 * substeps)(*its)
        self._host.bepuhost_set_solve_description(self._sim, substeps, arr)

    def set_integrator(self, integrator):
        self.integrator = integrator
        self._host.bepuhost_set_integrator(self._sim, C.byref(integrator))

    def add_bodies(self, dynamics):
        d = np.ascontiguousarray(dynamics, dtype=np.float32).reshape(-1, 32)
        return self._host.bepuhost_add_bodies(self._sim, d.ctypes.data, d.shape[0])

    @property
    def body_count(self):
        return self._host.bepuhost_body_count(self._sim)

    @property
    def bodies(self):
        n = self.body_count
        return np.ctypeslib.as_array(self._host.bepuhost_body_dynamics(self._sim), shape=(max(n, 1), 32))[:n]

    def add_constraints(self, type_id, body_handles, prestep):
        info = type_info(type_id)
        if info is None:
            raise ValueError("unsupported constraint type %d" % type_id)
        nb, p, _ = info
        h = np.ascontiguousarray(body_handles, dtype=np.int32).reshape(-1, nb)
        pre = np.ascontiguousarray(prestep, dtype=np.float32).reshape(-1, p)
        assert h.shape[0] == pre.shape[0]
        if h.shape[0] == 0:
            return -1
        first = self._host.bepuhost_add_constraints(self._sim, type_id, h.shape[0], h.ctypes.data, pre.ctypes.data)
        if first < 0:
            raise ValueError(self._host.bepuhost_last_error(self._sim).decode())
        return first

    def add_constraints_in_batches(self, type_id, body_handles, prestep, batch_indices):
        """Solver.Add for callers that already know each constraint's batch (computed by CudaTimestepper.color_constraints): the narrow phase's
        FindCandidateBatch -> TryAllocateInBatch path (Solver.cs:L984-1014, L1093-1140). Raises if a batch cannot hold its constraint."""
        nb, p, _ = type_info(type_id)
        h = np.ascontiguousarray(body_handles, dtype=np.int32).reshape(-1, nb)
        pre = np.ascontiguousarray(prestep, dtype=np.float32).reshape(-1, p)
        b = np.ascontiguousarray(batch_indices, dtype=np.int32).reshape(-1)
        assert h.shape[0] == pre.shape[0] == b.shape[0]
        if h.shape[0] == 0:
            return -1
        first = self._host.bepuhost_add_constraints_in_batches(self._sim, type_id, h.shape[0], h.ctypes.data, pre.ctypes.data, b.ctypes.data)
        if first < 0:
            raise ValueError(self._host.bepuhost_last_error(self._sim).decode())
        return first

    def constraint_references(self):
        """(references[n, 4], batch[n]) in handle (= add) order: encoded body references (kinematic flag in bit 30, -1 = unused slot) and batch indices."""
        n = self.constraint_count
        refs = np.full((max(n, 1), 4), -1, dtype=np.int32)
        batches = np.zeros(max(n, 1), dtype=np.int32)
        self._host.bepuhost_export_constraint_references(self._sim, refs.ctypes.data, batches.ctypes.data)
        return refs[:n], batches[:n]

    @property
    def constraint_count(self):
        return self._host.bepuhost_constraint_count(self._sim)

    @property
    def batch_count(self):
        return self._host.bepuhost_batch_count(self._sim)

    def constraint_location(self, handle):
        b, t, i = C.c_int32(), C.c_int32(), C.c_int32()
        if self._host.bepuhost_constraint_location(self._sim, handle, C.byref(b), C.byref(t), C.byref(i)) != 0:
            raise IndexError(handle)
        return b.value, t.value, i.value

    def type_batches(self):
        out = []
        for b in range(self.batch_count):
            for t in range(self._host.bepuhost_type_batch_count(self._sim, b)):
                v = TypeBatchView()
                self._host.bepuhost_get_type_batch(self._sim, b, t, C.byref(v))
                out.append(TypeBatch(b, t, v, self.bundle_width))
        return out

    @property
    def constrained_kinematics(self):
        n = self._host.bepuhost_constrained_kinematic_count(self._sim)
        if n == 0:
            return np.zeros(0, dtype=np.int32)
        return np.ctypeslib.as_array(self._host.bepuhost_constrained_kinematics(self._sim), shape=(n,)).copy()


class CudaTimestepper:
    """The Solve slot of DefaultTimestepper.Timestep (DefaultTimestepper.cs:L28-43) on the GPU, through the C ABI only."""

    def __init__(self, simulation, device=0, strict_fp=False, execution_mode=EXEC_GRAPH, disable_pdl=False):
        self._cuda, self._host = load_libraries()
        self.sim = simulation
        cfg = Config()
        cfg.device_ordinal, cfg.strict_fp, cfg.execution_mode = device, int(bool(strict_fp)), execution_mode
        cfg.reserved[1] = int(bool(disable_pdl))
        ctx = C.c_void_p()
        rc = self._cuda.bepucuda_create(C.byref(cfg), C.byref(ctx))
        if rc != 0:
            raise BepuCudaError(rc, "bepucuda_create failed (no usable CUDA device? there is no CPU fallback)")
        self._ctx = ctx
        self._registered = False

    def close(self):
        if getattr(self, "_ctx", None):
            for array in getattr(self, "_arrays", []):
                self._cuda.bepucuda_host_unregister(self._ctx, array.ctypes.data)
            self._arrays = []
            if self._registered:
                self._host.bepuhost_cuda_unregister_buffers(self.sim._sim, self._ctx)
            self._cuda.bepucuda_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise BepuCudaError(rc, self._cuda.bepucuda_last_error(self._ctx).decode())

    def color_constraints(self, references, body_count, fallback_batch_threshold=64, order=0, priorities=None):
        """bepucuda_color_constraints: batch index per constraint for references[n, slots] (encoded body references). Returns (batches, batch_count, rounds)."""
        refs = np.ascontiguousarray(references, dtype=np.int32)
        n, slots = refs.shape
        out = np.full(max(n, 1), -1, dtype=np.int32)
        pr = None if priorities is None else np.ascontiguousarray(priorities, dtype=np.uint32)
        count, rounds = C.c_int32(), C.c_int32()
        self._check(self._cuda.bepucuda_color_constraints(self._ctx, n, slots, refs.ctypes.data, body_count, fallback_batch_threshold, order, None if pr is None else pr.ctypes.data,
                                                          out.ctypes.data, C.byref(count), C.byref(rounds)))
        return out[:n], count.value, rounds.value

    def set_body_shapes(self, shapes):
        """bepucuda_set_body_shapes: one BODY_SHAPE_DTYPE record per body (static between frames unless a shape changes)."""
        shapes = np.ascontiguousarray(shapes, dtype=BODY_SHAPE_DTYPE)
        self._check(self._cuda.bepucuda_set_body_shapes(self._ctx, shapes.ctypes.data, shapes.shape[0]))

    def set_shape_library(self, library):
        """bepucuda_set_shape_library: uploads a ShapeLibrary (once; again when shapes change, followed by set_body_collidables)."""
        desc = library.desc()
        self._check(self._cuda.bepucuda_set_shape_library(self._ctx, C.byref(desc)))

    def set_body_collidables(self, collidables):
        """bepucuda_set_body_collidables: one BODY_COLLIDABLE_DTYPE record per body; from now on predict_bounding_boxes covers every built-in shape type."""
        collidables = np.ascontiguousarray(collidables, dtype=BODY_COLLIDABLE_DTYPE)
        self._check(self._cuda.bepucuda_set_body_collidables(self._ctx, collidables.ctypes.data if collidables.size else None, collidables.shape[0]))

    def predict_bounding_boxes(self, dt, activities):
        """bepucuda_predict_bounding_boxes on the body state resident on the device. `activities` (BODY_ACTIVITY_DTYPE) is updated in place.
        Returns bounds[n, 8] = {min.xyz, speculative margin, max.xyz, valid}."""
        assert activities.dtype == BODY_ACTIVITY_DTYPE and activities.flags["C_CONTIGUOUS"]
        bounds = np.zeros((max(activities.shape[0], 1), 8), dtype=np.float32)
        self._check(self._cuda.bepucuda_predict_bounding_boxes(self._ctx, dt, activities.ctypes.data, bounds.ctypes.data))
        return bounds[:activities.shape[0]]

    def register_host_buffers(self):
        """Page-locks the simulation's buffers (a C# host would register its BufferPool blocks once)."""
        self._check(self._host.bepuhost_cuda_register_buffers(self.sim._sim, self._ctx))
        self._registered = True

    def set_exchange(self, callback):
        """Sharded batches (bepucuda_set_boundary_bodies): `callback(device_pointer, word_count, op, cuda_stream) -> int` must combine `word_count` int32
        words at `device_pointer` across all ranks in place (op 0 = sum, 1 = min) as stream-ordered work on `cuda_stream`. None switches it off.
        Call before describe()."""
        if callback is None:
            self._exchange_cb = None
            self._check(self._cuda.bepucuda_set_boundary_bodies(self._ctx, None, 0, None, None))
            return

        def trampoline(user, words, count, op, stream):
            try:
                return int(callback(words, count, op, stream) or 0)
            except Exception:  # never unwind through the C frame
                import traceback

                traceback.print_exc()
                return -1

        self._exchange_cb = EXCHANGE_FN(trampoline)  # keep the thunk alive
        self._check(self._cuda.bepucuda_set_boundary_bodies(self._ctx, None, 0, self._exchange_cb, None))

    def describe(self):
        """Uploads bodies + every type batch and rebuilds device topology (call after any add/remove)."""
        self._check(self._host.bepuhost_cuda_describe(self.sim._sim, self._ctx))

    def refresh(self):
        """Per-frame upload with unchanged topology: body state + prestep/impulse data."""
        self._check(self._host.bepuhost_cuda_refresh(self.sim._sim, self._ctx))

    def solve(self, dt, download=True):
        self._check(self._host.bepuhost_cuda_solve(self.sim._sim, self._ctx, dt, 1 if download else 0))

    # ---- device-side contact update (SURVEY.md §8 f2, first slice): accumulated impulses stay on the device between frames --------------------
    def register_array(self, array):
        """Page-locks + maps a host array the per-frame calls read from (contact feature ids), like register_host_buffers does for the simulation's.
        The array is kept alive until close()."""
        nbytes = array.nbytes if array.ctypes.data % 4096 else ((array.nbytes + 4095) // 4096) * 4096  # page-aligned blocks are registered in whole pages
        self._check(self._cuda.bepucuda_host_register(self._ctx, array.ctypes.data, nbytes))
        self._arrays = getattr(self, "_arrays", []) + [array]

    def contact_feature_pool(self, rng=None):
        """One int32 block with the feature ids of every contact type batch back to back in (batch, type batch) order (the layout
        bepuhost_cuda_update_contacts walks), plus {(batch, type batch): view}. Filled with random ids when an rng is given."""
        count = lambda tid: (tid & 3) + 1 if tid <= 7 else (tid - 6 if tid <= 10 else tid - 13)
        tbs = [tb for tb in self.sim.type_batches() if tb.type_id <= 17]
        total = max(1, sum(tb.constraint_count * count(tb.type_id) for tb in tbs))
        backing = np.zeros(total + 2048, dtype=np.int32)  # page-aligned start and a whole number of pages, like a pinned pool block
        skip = (-backing.ctypes.data % 4096) // 4
        pool = backing[skip:skip + ((total + 1023) // 1024) * 1024][:total]
        if rng is not None:
            pool[:] = rng.integers(0, 1 << 20, size=pool.size, dtype=np.int32)
        views, at = {}, 0
        for tb in tbs:
            n = tb.constraint_count * count(tb.type_id)
            views[(tb.batch_index, tb.type_batch_index)] = pool[at:at + n].reshape(tb.constraint_count, count(tb.type_id))
            at += n
        return pool, views

    def set_contact_feature_pool(self, pool):
        self._check(self._host.bepuhost_cuda_update_contacts(self.sim._sim, self._ctx, pool.ctypes.data, 1))

    def update_contacts_from_pool(self, pool):
        """The whole per-frame refresh of the resident path in one native call: body motion + prestep + feature ids of every contact type batch."""
        self._check(self._host.bepuhost_cuda_update_contacts(self.sim._sim, self._ctx, pool.ctypes.data, 0))

    def set_contact_features(self, features):
        """features: {(batch_index, type_batch_index): int32[constraints, contacts]} = the feature ids the uploaded impulses belong to."""
        for (b, t), ids in features.items():
            ids = np.ascontiguousarray(ids, dtype=np.int32)
            self._check(self._cuda.bepucuda_set_contact_features(self._ctx, b, t, ids.ctypes.data))

    def update_contacts(self, features):
        """Per frame, same topology: the host's new prestep data + the new feature ids of every contact type batch; impulses are redistributed on the
        device (NarrowPhaseConstraintUpdate.cs:L81-135). Type batches not named in `features` keep their device rows."""
        by_key = {(tb.batch_index, tb.type_batch_index): tb for tb in self.sim.type_batches()}
        for (b, t), ids in features.items():
            ids = np.ascontiguousarray(ids, dtype=np.int32)
            self._check(self._cuda.bepucuda_update_contacts(self._ctx, b, t, by_key[(b, t)].prestep.ctypes.data, ids.ctypes.data))

    def upload_body_motion(self):
        """Pose + velocity halves of every BodyDynamics record only (64 of 128 bytes per body)."""
        self._check(self._cuda.bepucuda_upload_body_motion(self._ctx, self.sim.bodies.ctypes.data, self.sim.body_count))

    def download_bodies(self):
        """Full 128-B records: pose, velocity and world inertia."""
        self._check(self._cuda.bepucuda_download_bodies(self._ctx, self.sim.bodies.ctypes.data, self.sim.body_count))

    def download_body_motion(self):
        self._check(self._cuda.bepucuda_download_body_motion(self._ctx, self.sim.bodies.ctypes.data, self.sim.body_count))

    def download_impulses(self):
        self._check(self._cuda.bepucuda_download_impulses(self._ctx))

    def synchronize(self):
        self._check(self._cuda.bepucuda_synchronize(self._ctx))

    def download_prestep(self):
        self._check(self._host.bepuhost_cuda_download_prestep(self.sim._sim, self._ctx))

    def event_record(self, slot):
        self._check(self._cuda.bepucuda_event_record(self._ctx, slot))

    def event_elapsed_ms(self, slot_begin, slot_end):
        ms = C.c_float()
        self._check(self._cuda.bepucuda_event_elapsed_ms(self._ctx, slot_begin, slot_end, C.byref(ms)))
        return ms.value

    def profile_stages(self, dt):
        """One frame as plain stream launches with a CUDA event pair around every stage launch; returns per-stage-kind ms / launches / algorithmic bytes."""
        p = StageProfile()
        self._check(self._cuda.bepucuda_profile_stages(self._ctx, dt, C.byref(p)))
        return p

    def solve_device_only(self, dt):
        """bepucuda_solve without downloads (state stays resident in HBM)."""
        self._check(self._cuda.bepucuda_solve(self._ctx, dt))

    def timings(self):
        t = Timings()
        self._check(self._cuda.bepucuda_get_timings(self._ctx, C.byref(t)))
        return t
