// libbepucuda host side: context, device memory, uploads/downloads, topology analysis, stage program, CUDA graph.
// C ABI declared in include/bepucuda.h. No CPU fallback lives here: without a usable CUDA device bepucuda_create fails.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../include/bepucuda.h"
#include "bepu_layout_kernels.h"
#include "bepu_coloring.h"
#include "bepu_bounds.h"
#include "bepu_shape_bounds.h"

using namespace bepucuda;

namespace bepucuda {

// ---- type registry -------------------------------------------------------------------------------------------------------
// bodies / prestep floats / impulse floats per BatchTypeId, and SURVEY.md §8d algorithmic bytes:
//   solve       = 4 * (P + 2D + n + sum(R_i + W_i))        R/W from the type's Solve access filters
//   warm start  = 4 * (P + D + n + sum(R'_i + W'_i))       (non-integrating lane, WarmStart filters)
//   incremental = 4 * (P_read + contacts_written + n + 6n)
// Filters (IBodyAccessFilter.cs:L38-126): pos 3, orientation 4, lin 3, ang 3, inertia tensor 6, mass 1.
static TypeInfo make_contact(int bodies, int prestep, int impulses, int contacts, const char* name) {
    TypeInfo t{};
    t.bodies = bodies; t.prestep_rows = prestep; t.impulse_rows = impulses; t.incremental = 1; t.name = name;
    const int body_rw = 13 + 6;  // AccessNoPose: velocity 6 + inertia 7 read, velocity 6 written
    t.solve_bytes = 4 * (prestep + 2 * impulses + bodies + bodies * body_rw);
    t.warm_start_bytes = 4 * (prestep + impulses + bodies + bodies * body_rw);
    t.incremental_bytes = 4 * (prestep + contacts + bodies + 6 * bodies);
    return t;
}
static TypeInfo make_joint(int bodies, int prestep, int impulses, int solve_r, int solve_w, int ws_r, int ws_w, const char* name) {
    TypeInfo t{};
    t.bodies = bodies; t.prestep_rows = prestep; t.impulse_rows = impulses; t.incremental = 0; t.name = name;
    t.solve_bytes = 4 * (prestep + 2 * impulses + bodies + solve_r + solve_w);
    t.warm_start_bytes = 4 * (prestep + impulses + bodies + ws_r + ws_w);
    t.incremental_bytes = 0;
    return t;
}
struct Registry {
    TypeInfo types[64];
    bool present[64];
    Registry() {
        std::memset(present, 0, sizeof(present));
        auto add = [&](int id, TypeInfo t) { types[id] = t; present[id] = true; };
        add(0, make_contact(1, 11, 4, 1, "Contact1OneBody")); add(1, make_contact(1, 15, 5, 2, "Contact2OneBody"));
        add(2, make_contact(1, 19, 6, 3, "Contact3OneBody")); add(3, make_contact(1, 23, 7, 4, "Contact4OneBody"));
        add(4, make_contact(2, 14, 4, 1, "Contact1")); add(5, make_contact(2, 18, 5, 2, "Contact2"));
        add(6, make_contact(2, 22, 6, 3, "Contact3")); add(7, make_contact(2, 26, 7, 4, "Contact4"));
        add(8, make_contact(1, 18, 6, 2, "Contact2NonconvexOneBody")); add(9, make_contact(1, 25, 9, 3, "Contact3NonconvexOneBody"));
        add(10, make_contact(1, 32, 12, 4, "Contact4NonconvexOneBody"));
        add(15, make_contact(2, 21, 6, 2, "Contact2Nonconvex")); add(16, make_contact(2, 28, 9, 3, "Contact3Nonconvex"));
        add(17, make_contact(2, 35, 12, 4, "Contact4Nonconvex"));
#define BEPU_REGISTER_JOINTS
#include "bepu_joint_registry.inc"
#undef BEPU_REGISTER_JOINTS
    }
};
static const Registry& registry() {
    static Registry r;
    return r;
}
const TypeInfo* get_type_info(int type_id) {
    if (type_id < 0 || type_id >= 64 || !registry().present[type_id]) return nullptr;
    return &registry().types[type_id];
}

// ---- small RAII helpers ------------------------------------------------------------------------------------------------------
struct DeviceBuffer {
    void* ptr = nullptr;
    size_t capacity = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= capacity) return cudaSuccess;
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        capacity = 0;
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&ptr, want);
        if (e == cudaSuccess) capacity = want;
        return e;
    }
    void release() {
        if (ptr) cudaFree(ptr);
        ptr = nullptr;
        capacity = 0;
    }
    template <class T> T* as() const { return (T*)ptr; }
};

// Bump allocator over chunks that are never reallocated (uploads are enqueued against their addresses).
struct ChunkArena {
    struct Chunk { char* base; size_t size, used; };
    std::vector<Chunk> chunks;
    bool pinned_host = false;
    size_t min_chunk = (size_t)64 << 20;
    void reset() { for (auto& c : chunks) c.used = 0; }
    void* alloc(size_t bytes, cudaError_t* err) {
        bytes = (bytes + 255) & ~(size_t)255;
        for (auto& c : chunks)
            if (c.size - c.used >= bytes) {
                void* p = c.base + c.used;
                c.used += bytes;
                return p;
            }
        Chunk c{};
        c.size = std::max(bytes, min_chunk);
        cudaError_t e = pinned_host ? cudaMallocHost((void**)&c.base, c.size) : cudaMalloc((void**)&c.base, c.size);
        if (e != cudaSuccess) { if (err) *err = e; return nullptr; }
        c.used = bytes;
        chunks.push_back(c);
        return chunks.back().base;
    }
    void release() {
        for (auto& c : chunks) { if (pinned_host) cudaFreeHost(c.base); else cudaFree(c.base); }
        chunks.clear();
    }
};

struct SourceTypeBatch {
    int batch_index, type_batch_index, type_id, count;
    int live = 0;          // constraints actually present (fallback type batches may contain holes)
    float* host_impulses;
    int32_t* raw_refs;     // device, reference AOSOA-W layout
    float* raw_prestep;
    float* raw_impulses;
    size_t refs_bytes, prestep_bytes, impulse_bytes;
    std::vector<int32_t> host_refs;  // retained only for fallback batches (levelisation)
    std::vector<int> device_tbs;
    // device-side contact update (bepucuda_update_contacts): feature ids of the resident impulses / of the frame being uploaded
    int32_t* raw_features_old = nullptr;
    int32_t* raw_features_new = nullptr;
    size_t feature_bytes = 0;
    bool resident_impulses = false, redistribute = false;
};

}  // namespace bepucuda

struct bepucuda_ctx {
    bepucuda_config cfg{};
    int32_t tune[4] = {0, 0, 0, 0};
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev_solve_begin = nullptr, ev_solve_end = nullptr, ev_up_begin = nullptr, ev_up_end = nullptr, ev_down_begin = nullptr, ev_down_end = nullptr;
    bool up_open = false, have_solve = false, have_down = false, have_up = false;
    std::string error;
    const SolverLaunchers* launchers = nullptr;

    // solve description / integrator
    std::vector<int32_t> iterations{1};
    int fallback_threshold = 64;
    bepucuda_integrator_desc integ{};
    bool integ_set = false;

    // bodies
    int body_count = 0;
    DeviceBuffer raw_bodies, pose, velocity, inertia_local, inertia_world, constrained, first_batch, sync_refcount, sync_mask;
    BodyBuffers B{};

    // constraints
    int W = 8;
    int batch_count = 0;
    bool constraints_open = false, constraints_ready = false, data_dirty = false, descs_dirty = false;
    std::vector<SourceTypeBatch> sources;
    ChunkArena raw_arena, pinned_arena;
    DeviceBuffer record_table, ref_rows, source_bundle_flags, refs32, prestep32, impulses32, tb_table, tdesc_table, work_table, map_table, bodies_per_type, kinematics_dev, program_dev, frame_params_dev, error_dev;
    std::vector<DeviceTypeBatch> tbs;
    std::vector<TransposeDesc> tdescs;
    std::vector<WorkItem> work;                 // grouped by device batch, then the incremental list
    std::vector<int32_t> bundle_live;           // live constraints per work item (parallel to `work`)
    std::vector<WorkRecord> records;            // what the solver kernels read (parallel to `work`)
    std::vector<std::pair<int, int>> batch_work; // per device batch: (begin, count) into work
    bool exchange_failed = false;
    bepucuda_exchange_fn exchange = nullptr;    // sharded batches (bepucuda_set_boundary_bodies): all-reduce callback, its user pointer, staging planes
    void* exchange_user = nullptr;
    DeviceBuffer exchange_staging;
    // peer sharding (bepucuda_shard_*): one constraint graph over several GPUs with NVLink peer stores and a flag barrier per stage
    bool peer_mode = false;
    ShardPeers peers{};
    DeviceBuffer shard_flags, pushes_dev, peer32, body_masks_dev, boundary_flags_dev;
    uint32_t shard_solve_index = 0;                                 // solves since the arrival targets were last published
    std::vector<int> boundary_count;                                // per device batch: bundles that touch a body another rank references
    std::vector<uint8_t> body_masks;                                // bepucuda_shard_set_body_masks: fused pushes from the stage kernels
    size_t refs_words = 0;
    std::vector<void*> opened_ipc;
    std::vector<int32_t> global_first_batch;
    std::vector<uint8_t> global_constrained;
    std::map<int, std::vector<uint32_t>> pushes_by_batch;          // host batch index -> packed (body | rank << 28 | owner << 31)
    std::vector<std::pair<size_t, int>> push_range;                // per device batch: (offset, count) into pushes_dev
    uint32_t exchange_counter = 0;                                  // exchange points executed so far (flag barrier sequence)
    uint32_t exchanges_per_solve = 0;
    int inc_work_begin = 0, inc_work_count = 0;
    int all_work_count = 0;                     // work[0 .. all_work_count) covers every bundle once
    int sync_batch_count = 0, fallback_levels = 0;
    std::vector<int32_t> kinematics;
    std::vector<StageOp> program;
    FrameParams* frame_params_host = nullptr;   // pinned

    cudaGraph_t graph = nullptr;
    cudaGraphExec_t graph_exec = nullptr;
    bool graph_valid = false;

    bepucuda_timings timings{};
    int64_t h2d_accum = 0;
    struct HostRange { char* host; size_t bytes; char* dev; };
    std::vector<HostRange> host_ranges;    // page-locked + device-mapped host memory registered through bepucuda_host_register
    std::vector<CopyChunk> pending_h2d;    // batched copies waiting for the next flush
    DeviceBuffer chunk_table;
    struct ChunkStage { void* host = nullptr; size_t capacity = 0; cudaEvent_t done = nullptr; };
    ChunkStage chunk_stage[4];             // pinned ring for chunk tables (a table must outlive its H2D copy)
    int chunk_stage_next = 0;
    cudaEvent_t user_events[16] = {};
    DeviceBuffer body_shapes, body_activities, body_bounds;  // bepucuda_set_body_shapes / bepucuda_predict_bounding_boxes
    int shape_count = -1;
    // bepucuda_set_shape_library / bepucuda_set_body_collidables
    struct ShapeBounds {
        DeviceBuffer library[12];  // the arrays of bepucuda_shape_library, in its field order
        ShapeLibraryView view{};
        bool library_set = false;
        bepucuda_shape_library counts{};  // counts only (pointers cleared)
        std::vector<bepucuda_mesh> meshes;
        DeviceBuffer collidables, hull_bodies, compound_bodies, mesh_bodies, mesh_chunks, mesh_partials;
        ShapeBoundsWork work{};
        int collidable_count = -1;
        bool active = false;  // set_body_collidables was called after set_body_shapes
        void release() {
            for (auto& b : library) b.release();
            for (DeviceBuffer* b : {&collidables, &hull_bodies, &compound_bodies, &mesh_bodies, &mesh_chunks, &mesh_partials}) b->release();
        }
    } shape_bounds;
    DeviceBuffer color_refs, color_priorities, color_body_min, color_body_mask, color_out, color_lists, color_counts;  // bepucuda_color_constraints
    std::vector<cudaEvent_t> profile_events;
};

namespace {

int fail(bepucuda_ctx* c, int code, const std::string& msg) {
    if (c) c->error = msg;
    return code;
}
int cuda_fail(bepucuda_ctx* c, cudaError_t e, const char* what) {
    return fail(c, e == cudaErrorMemoryAllocation ? BEPUCUDA_ERR_OUT_OF_MEMORY : BEPUCUDA_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}
#define CK(call)                                                  \
    do {                                                          \
        cudaError_t _e = (call);                                  \
        if (_e != cudaSuccess) return cuda_fail(ctx, _e, #call);  \
    } while (0)

void open_upload_window(bepucuda_ctx* ctx) {
    if (!ctx->up_open) {
        cudaEventRecord(ctx->ev_up_begin, ctx->stream);
        ctx->up_open = true;
    }
}

// Device alias of a host pointer if [ptr, ptr + bytes) lies inside a registered (mapped) range, else nullptr.
char* map_host(bepucuda_ctx* ctx, const void* ptr, size_t bytes) {
    const char* p = (const char*)ptr;
    for (auto& r : ctx->host_ranges)
        if (p >= r.host && p + bytes <= r.host + r.bytes) return r.dev + (p - r.host);
    return nullptr;
}
void queue_chunks(std::vector<CopyChunk>& list, void* dst, const void* src, size_t bytes) {
    const size_t kChunk = (size_t)64 << 10;
    for (size_t off = 0; off < bytes; off += kChunk) list.push_back({(char*)dst + off, (const char*)src + off, std::min(kChunk, bytes - off)});
}
// Runs the queued chunks as one kernel. The chunk table travels through the pinned staging arena (recycled at begin_constraints / per flush).
int flush_chunks(bepucuda_ctx* ctx, std::vector<CopyChunk>& list) {
    if (list.empty()) return BEPUCUDA_OK;
    const size_t bytes = list.size() * sizeof(CopyChunk);
    CK(ctx->chunk_table.reserve(bytes));
    auto& st = ctx->chunk_stage[ctx->chunk_stage_next];
    ctx->chunk_stage_next = (ctx->chunk_stage_next + 1) & 3;
    if (!st.done) CK(cudaEventCreateWithFlags(&st.done, cudaEventDisableTiming));
    CK(cudaEventSynchronize(st.done));  // its previous use (4 flushes ago) is long finished
    if (st.capacity < bytes) {
        if (st.host) cudaFreeHost(st.host);
        st.host = nullptr;
        st.capacity = 0;
        CK(cudaMallocHost(&st.host, bytes * 2));
        st.capacity = bytes * 2;
    }
    std::memcpy(st.host, list.data(), bytes);
    // The device-side table is reused by every flush: stream order keeps the previous batched copy ahead of this overwrite.
    CK(cudaMemcpyAsync(ctx->chunk_table.ptr, st.host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    launch_batched_copy(ctx->chunk_table.as<CopyChunk>(), (int)list.size(), ctx->stream);
    CK(cudaGetLastError());
    CK(cudaEventRecord(st.done, ctx->stream));
    list.clear();
    return BEPUCUDA_OK;
}

// H2D copy of one host buffer into the raw arena. Small buffers are packed through pinned staging so that hundreds of
// tiny type batches do not each pay a pageable-memory DMA setup; large ones go directly (fast when the host registered them).
int copy_in(bepucuda_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (bytes == 0) return BEPUCUDA_OK;
    if (char* alias = map_host(ctx, src, bytes)) {
        queue_chunks(ctx->pending_h2d, dst, alias, bytes);  // read straight from the mapped host buffer by the batched copy kernel at the next flush
        ctx->h2d_accum += (int64_t)bytes;
        return BEPUCUDA_OK;
    }
    if (bytes < ((size_t)256 << 10)) {
        cudaError_t e = cudaSuccess;
        void* stage = ctx->pinned_arena.alloc(bytes, &e);
        if (!stage) return cuda_fail(ctx, e, "pinned staging");
        std::memcpy(stage, src, bytes);
        CK(cudaMemcpyAsync(dst, stage, bytes, cudaMemcpyHostToDevice, ctx->stream));
    } else {
        CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    ctx->h2d_accum += (int64_t)bytes;
    return BEPUCUDA_OK;
}

void invalidate_graph(bepucuda_ctx* ctx) {
    if (ctx->graph_exec) cudaGraphExecDestroy(ctx->graph_exec);
    if (ctx->graph) cudaGraphDestroy(ctx->graph);
    ctx->graph_exec = nullptr;
    ctx->graph = nullptr;
    ctx->graph_valid = false;
}

// Issues the whole stage sequence of one frame as individual launches on `s` (used directly in STREAM mode and under
// capture in GRAPH mode). Order: Solver_Solve.cs:L1419-1479, then PoseIntegrator.IntegrateAfterSubstepping.
void issue_stage_sequence(bepucuda_ctx* ctx, cudaStream_t s, int64_t* launches) {
    const WorkRecord* records = ctx->record_table.as<WorkRecord>();
    const int32_t* ref_rows = ctx->ref_rows.as<int32_t>();
    const FrameParams* fp = ctx->frame_params_dev.as<FrameParams>();
    const int32_t* kin = ctx->kinematics_dev.as<int32_t>();
    int64_t n = 0;
    const bool pdl = ctx->cfg.reserved[1] == 0;
    // Row prefetch in the PDL prologue (see constraint_stage_kernel): allowed when the kernel launched immediately before neither rewrites this
    // batch's prestep rows (the incremental contact update does) nor its impulses (a stage of the same batch does: single-batch scenes).
    const StageOp* previous = nullptr;  // last launched op
    uint32_t exchange_index = 0;
    const bool fused_pushes = ctx->peer_mode && !ctx->body_masks.empty();
    for (const StageOp& op : ctx->program) {
        if (ctx->peer_mode && op.pad == -1) {
            // all ranks meet (nothing to push): before the first stage of a solve; around the incremental contact update, which reads the velocities
            // of shared bodies -- after every peer's last Solve stage has completed, before any peer's WarmStart stage stores into this rank's
            // arrays; and before the final pose pass
            launch_shard_exchange(nullptr, 0, 1, ctx->B, ctx->peers, fp, exchange_index++, ctx->error_dev.as<int32_t>(), s);
            ++n;
            continue;
        }
        if (ctx->peer_mode && op.pad >= 2 && op.stage <= kStageSolve) {
            // peer sharding: the stage on this rank's constraints of the batch, then records written for shared bodies go to the ranks that
            // reference them and all ranks meet at the flag barrier
            if (op.work_count > 0) {
                // row prefetch in the prologue: the exchange kernel between two stages writes no rows, so the rule of the single-GPU sequence applies
                bool prefetch = previous != nullptr && previous->stage != kStageIncremental && !(previous->stage <= kStageSolve && previous->work_begin == op.work_begin && previous->work_count > 0);
                const int launch_flags = (pdl ? kLaunchPdl : 0) | (prefetch ? kLaunchPrefetchRows : 0);
                if (fused_pushes) {
                    // the stage pushes, signals and (in its boundary bundles) waits itself: no exchange kernel
                    const ShardStage shard{exchange_index, ctx->error_dev.as<int32_t>()};
                    ctx->launchers->constraint_stage_sharded(op.stage, records + op.work_begin, ref_rows + (size_t)op.work_begin * 64, op.work_count, ctx->B, fp, launch_flags, ctx->peers,
                                                             (long long)(ctx->peer32.as<int32_t>() - ctx->refs32.as<int32_t>()), shard, s);
                    ++exchange_index;
                    ++n;
                    previous = &op;
                    continue;
                }
                ctx->launchers->constraint_stage(op.stage, records + op.work_begin, ref_rows + (size_t)op.work_begin * 64, op.work_count, ctx->B, fp, launch_flags, s);
                ++n;
            }
            if (fused_pushes) { ++exchange_index; continue; }  // no constraint of this batch here: nothing arrives from this rank, its targets say so
            const auto& range = ctx->push_range[op.pad - 2];
            launch_shard_exchange(ctx->pushes_dev.as<uint32_t>() + range.first, range.second, op.stage == kStageSolve ? 1 : (op.stage == kStageWarmStart ? 3 : 2), ctx->B, ctx->peers, fp,
                                  exchange_index++, ctx->error_dev.as<int32_t>(), s);
            ++n;
            if (op.work_count > 0) previous = &op;
            continue;
        }
        switch (op.stage) {
            case kStageWarmStartFirst: case kStageWarmStart: case kStageSolve: case kStageIncremental:
                if (op.work_count > 0) {
                    bool prefetch = op.stage != kStageIncremental && previous != nullptr && previous->stage != kStageIncremental;
                    if (prefetch && previous->stage <= kStageSolve && previous->work_begin == op.work_begin) prefetch = false;
                    if (ctx->exchange) {
                        // sharded batches: plain launches, then all ranks learn what this rank's constraints wrote in this stage
                        ctx->launchers->constraint_stage(op.stage, records + op.work_begin, ref_rows + (size_t)op.work_begin * 64, op.work_count, ctx->B, fp, 0, s);
                        ++n;
                        if (op.stage != kStageIncremental) {
                            const int planes = op.stage == kStageSolve ? 1 : (op.stage == kStageWarmStart ? 3 : 2);
                            const size_t words = (size_t)ctx->body_count * 8 * planes;
                            cudaMemsetAsync(ctx->exchange_staging.ptr, 0, words * 4, s);
                            launch_collect_stage(ctx->tb_table.as<DeviceTypeBatch>(), ctx->work_table.as<WorkItem>() + op.work_begin, op.work_count, ctx->bodies_per_type.as<int32_t>(), op.stage,
                                                 ctx->B, ctx->exchange_staging.as<int32_t>(), s);
                            if (ctx->exchange(ctx->exchange_user, ctx->exchange_staging.ptr, (int64_t)words, 0, (void*)s) != 0) ctx->exchange_failed = true;
                            launch_apply_stage(ctx->exchange_staging.as<int32_t>(), planes, ctx->B, s);
                            n += 2;
                        }
                        previous = &op;
                        break;
                    }
                    ctx->launchers->constraint_stage(op.stage, records + op.work_begin, ref_rows + (size_t)op.work_begin * 64, op.work_count, ctx->B, fp, (pdl ? kLaunchPdl : 0) | (prefetch ? kLaunchPrefetchRows : 0), s);
                    previous = &op;
                    ++n;
                }
                break;
            case kStageKinematicFirst: case kStageKinematic:
                if (op.work_count > 0) { ctx->launchers->kinematic_stage(op.stage, kin, op.work_count, ctx->B, fp, s); previous = &op; ++n; }
                break;
            case kStageFinalPose:
                if (ctx->B.count > 0) { ctx->launchers->final_pose(ctx->B, fp, s); previous = &op; ++n; }
                break;
        }
    }
    if (launches) *launches = n;
    ctx->exchanges_per_solve = exchange_index;
}

// Builds the flat stage program for the current topology + solve description.
void build_program(bepucuda_ctx* ctx) {
    ctx->program.clear();
    const int substeps = (int)ctx->iterations.size();
    const int kin = (int)ctx->kinematics.size();
    for (int s = 0; s < substeps; ++s) {
        if (s > 0) {
            // peer sharding: what peers pushed in the last Solve stages must have arrived before the contact update reads velocities (rank barrier)
            if (ctx->peer_mode) ctx->program.push_back({kStageKinematic, 0, 0, -1});
            if (ctx->inc_work_count > 0) ctx->program.push_back({kStageIncremental, ctx->inc_work_begin, ctx->inc_work_count, 0});
            if (kin > 0) ctx->program.push_back({kStageKinematic, 0, kin, 0});
        } else if (ctx->integ.integrate_velocity_for_kinematics && kin > 0) {
            ctx->program.push_back({kStageKinematicFirst, 0, kin, 0});
        }
        if (ctx->peer_mode) ctx->program.push_back({kStageKinematic, 0, 0, -1});  // rank barrier (see issue_stage_sequence)
        // pad carries the device batch index + 2 in peer mode (every rank runs the exchange of every batch, also of one it has no constraint in)
        for (size_t b = 0; b < ctx->batch_work.size(); ++b) {
            auto& bw = ctx->batch_work[b];
            if (bw.second > 0 || (ctx->peer_mode && (int)b < ctx->sync_batch_count)) ctx->program.push_back({s == 0 ? kStageWarmStartFirst : kStageWarmStart, bw.first, bw.second, ctx->peer_mode ? (int)b + 2 : 0});
        }
        for (int it = 0; it < ctx->iterations[s]; ++it)
            for (size_t b = 0; b < ctx->batch_work.size(); ++b) {
                auto& bw = ctx->batch_work[b];
                if (bw.second > 0 || (ctx->peer_mode && (int)b < ctx->sync_batch_count)) ctx->program.push_back({kStageSolve, bw.first, bw.second, ctx->peer_mode ? (int)b + 2 : 0});
            }
    }
    if (ctx->peer_mode) ctx->program.push_back({kStageKinematic, 0, 0, -1});  // ... and before the final pose pass reads them
    ctx->program.push_back({kStageFinalPose, 0, ctx->body_count, 0});
}

int upload_program(bepucuda_ctx* ctx) {
    build_program(ctx);
    if (ctx->peer_mode && !ctx->body_masks.empty() && ctx->boundary_count.size() == ctx->batch_work.size()) {
        // fused pushes: publish, to every peer, how many boundary bundles of this rank arrive through each exchange point of one solve (ShardStage),
        // and restart the arrival counters other ranks increment here. Every rank does this for the same program, between solves.
        std::vector<unsigned long long> targets((size_t)kShardMaxExchanges, 0ull);
        unsigned long long arrived = 0;
        size_t e = 0;
        for (const StageOp& op : ctx->program) {
            if (op.pad != -1 && !(op.pad >= 2 && op.stage <= kStageSolve)) continue;
            if (e + 1 >= (size_t)kShardMaxExchanges) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "peer sharding: more than 4095 exchange points per solve");
            if (op.pad >= 2 && op.work_count > 0) arrived += (unsigned long long)ctx->boundary_count[(size_t)(op.pad - 2)];
            targets[e++] = arrived;
        }
        targets[(size_t)kShardMaxExchanges - 1] = arrived;
        CK(cudaStreamSynchronize(ctx->stream));
        for (int q = 0; q < ctx->peers.rank_count; ++q)
            if (q != ctx->peers.rank)
                CK(cudaMemcpy(ctx->peers.flags[q] + kShardTargetSlot + (size_t)ctx->peers.rank * kShardMaxExchanges, targets.data(), targets.size() * 8, cudaMemcpyDefault));
        CK(cudaMemset((unsigned long long*)ctx->shard_flags.ptr + kShardCounterSlot, 0, kMaxShardRanks * 8));
        ctx->shard_solve_index = 0;
    }
    CK(ctx->program_dev.reserve(ctx->program.size() * sizeof(StageOp)));
    CK(cudaMemcpyAsync(ctx->program_dev.ptr, ctx->program.data(), ctx->program.size() * sizeof(StageOp), cudaMemcpyHostToDevice, ctx->stream));
    // The copy source is a std::vector: make sure the DMA read it before anyone mutates it.
    CK(cudaStreamSynchronize(ctx->stream));
    invalidate_graph(ctx);
    // stage statistics
    int64_t stages = 0;
    for (auto& op : ctx->program) stages += (op.work_count > 0 || op.stage == kStageFinalPose) ? 1 : 0;
    ctx->timings.stage_count = stages;
    return BEPUCUDA_OK;
}

void compute_frame_params(bepucuda_ctx* ctx, float dt, FrameParams* fp) {
    const int substeps = (int)ctx->iterations.size();
    const float substepDt = dt / substeps;  // Solver_Solve.cs:L1417
    auto clamp01 = [](float v) { return v < 0.f ? 0.f : (v > 1.f ? 1.f : v); };
    const bepucuda_integrator_desc& d = ctx->integ;
    fp->dt = substepDt;
    fp->inverse_dt = 1.0f / substepDt;
    // PrepareForIntegration(substepDt): Demos/DemoCallbacks.cs:L79-86
    fp->linear_damping_dt = powf(clamp01(1 - d.linear_damping), substepDt);
    fp->angular_damping_dt = powf(clamp01(1 - d.angular_damping), substepDt);
    for (int i = 0; i < 3; ++i) fp->gravity_dt[i] = d.gravity[i] * substepDt;
    // IntegrateAfterSubstepping: PoseIntegrator.cs:L707-712
    const float finalDt = d.allow_substeps_for_unconstrained ? substepDt : dt;
    fp->final_dt = finalDt;
    fp->final_linear_damping_dt = powf(clamp01(1 - d.linear_damping), finalDt);
    fp->final_angular_damping_dt = powf(clamp01(1 - d.angular_damping), finalDt);
    for (int i = 0; i < 3; ++i) fp->final_gravity_dt[i] = d.gravity[i] * finalDt;
    fp->final_steps = d.allow_substeps_for_unconstrained ? substeps : 1;
    fp->angular_mode = d.angular_integration_mode;
    fp->integrate_velocity_for_kinematics = d.integrate_velocity_for_kinematics;
    for (int i = 0; i < 4; ++i) fp->tune[i] = ctx->tune[i];
}

// Brings the device AOSOA-32 rows up to date with what the host queued since the last solve (bepucuda_update_type_batch / bepucuda_update_contacts):
// flushes the batched copies, re-uploads the transposition descriptors when a type batch switched to resident impulses, transposes, and
// redistributes the resident penetration impulses of updated contact type batches from the old to the new feature ids.
int refresh_device_rows(bepucuda_ctx* ctx) {
    if (!ctx->data_dirty) return BEPUCUDA_OK;
    { int rc = flush_chunks(ctx, ctx->pending_h2d); if (rc != BEPUCUDA_OK) return rc; }
    bool any_redistribute = false;
    if (ctx->descs_dirty) {
        for (SourceTypeBatch& s : ctx->sources)
            for (int tb : s.device_tbs) {
                TransposeDesc& d = ctx->tdescs[tb];
                d.flags = (s.resident_impulses ? kDescResidentImpulses : 0) | (s.redistribute ? kDescRedistribute : 0);
                d.features_old = s.raw_features_old;
                d.features_new = s.raw_features_new;
                any_redistribute |= s.redistribute;
            }
        CK(cudaMemcpyAsync(ctx->tdesc_table.ptr, ctx->tdescs.data(), ctx->tdescs.size() * sizeof(TransposeDesc), cudaMemcpyHostToDevice, ctx->stream));
    }
    launch_transpose_in_all(ctx->tb_table.as<DeviceTypeBatch>(), ctx->tdesc_table.as<TransposeDesc>(), ctx->work_table.as<WorkItem>(), ctx->all_work_count, ctx->W,
                            kTransposePrestep | kTransposeImpulses, ctx->stream);
    if (any_redistribute) {
        launch_redistribute_impulses(ctx->tb_table.as<DeviceTypeBatch>(), ctx->tdesc_table.as<TransposeDesc>(), ctx->work_table.as<WorkItem>(), ctx->all_work_count, ctx->stream);
        for (SourceTypeBatch& s : ctx->sources)
            if (s.redistribute) {
                std::swap(s.raw_features_old, s.raw_features_new);  // the resident impulses now belong to the new ids
                s.redistribute = false;
            }
        // descriptors still carry kDescRedistribute and the pre-swap pointers: they are rewritten by the next update (descs_dirty stays set)
    } else {
        ctx->descs_dirty = false;
    }
    CK(cudaGetLastError());
    ctx->data_dirty = false;
    return BEPUCUDA_OK;
}

}  // namespace

extern "C" {

int32_t bepucuda_type_info(int32_t type_id, int32_t* bodies_per_constraint, int32_t* prestep_floats, int32_t* impulse_floats) {
    const TypeInfo* t = get_type_info(type_id);
    if (!t) return BEPUCUDA_ERR_UNSUPPORTED_TYPE;
    if (bodies_per_constraint) *bodies_per_constraint = t->bodies;
    if (prestep_floats) *prestep_floats = t->prestep_rows;
    if (impulse_floats) *impulse_floats = t->impulse_rows;
    return BEPUCUDA_OK;
}

int32_t bepucuda_create(const bepucuda_config* cfg, bepucuda_ctx** out) {
    if (!cfg || !out) return BEPUCUDA_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) return BEPUCUDA_ERR_NO_DEVICE;  // no CPU fallback, by design
    if (cfg->device_ordinal < 0 || cfg->device_ordinal >= count) return BEPUCUDA_ERR_INVALID_ARGUMENT;
    if (cfg->execution_mode != BEPUCUDA_EXEC_GRAPH && cfg->execution_mode != BEPUCUDA_EXEC_STREAM) return BEPUCUDA_ERR_INVALID_ARGUMENT;  // 1 and 3 are retired modes
    bepucuda_ctx* ctx = new bepucuda_ctx();
    ctx->cfg = *cfg;
    if (const char* tune = getenv("BEPUCUDA_TUNE")) sscanf(tune, "%d,%d,%d,%d", &ctx->tune[0], &ctx->tune[1], &ctx->tune[2], &ctx->tune[3]);
    ctx->device = cfg->device_ordinal;
    ctx->launchers = cfg->strict_fp ? get_launchers_bepu_strict() : get_launchers_bepu_fast();
    ctx->pinned_arena.pinned_host = true;
    ctx->pinned_arena.min_chunk = (size_t)16 << 20;
    cudaError_t e = cudaSetDevice(ctx->device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
    cudaEvent_t* evs[] = {&ctx->ev_solve_begin, &ctx->ev_solve_end, &ctx->ev_up_begin, &ctx->ev_up_end, &ctx->ev_down_begin, &ctx->ev_down_end};
    for (auto ev : evs)
        if (e == cudaSuccess) e = cudaEventCreate(ev);
    if (e == cudaSuccess) e = cudaMallocHost((void**)&ctx->frame_params_host, sizeof(FrameParams));
    if (e == cudaSuccess) e = ctx->frame_params_dev.reserve(sizeof(FrameParams));
    if (e == cudaSuccess) e = ctx->error_dev.reserve(8 * sizeof(int32_t));
    if (e != cudaSuccess) {
        bepucuda_destroy(ctx);
        return e == cudaErrorMemoryAllocation ? BEPUCUDA_ERR_OUT_OF_MEMORY : BEPUCUDA_ERR_CUDA;
    }
    // DemoPoseIntegratorCallbacks defaults (Demos/DemoCallbacks.cs:L60)
    ctx->integ.gravity[0] = 0; ctx->integ.gravity[1] = -10; ctx->integ.gravity[2] = 0;
    ctx->integ.linear_damping = 0.03f;
    ctx->integ.angular_damping = 0.03f;
    *out = ctx;
    return BEPUCUDA_OK;
}

int32_t bepucuda_destroy(bepucuda_ctx* ctx) {
    if (!ctx) return BEPUCUDA_OK;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    invalidate_graph(ctx);
    for (void* p : ctx->opened_ipc) cudaIpcCloseMemHandle(p);
    DeviceBuffer* bufs[] = {&ctx->shard_flags, &ctx->pushes_dev, &ctx->peer32, &ctx->body_masks_dev, &ctx->boundary_flags_dev, &ctx->raw_bodies, &ctx->pose, &ctx->velocity, &ctx->inertia_local, &ctx->inertia_world, &ctx->constrained, &ctx->first_batch, &ctx->sync_refcount,
                            &ctx->sync_mask, &ctx->chunk_table, &ctx->record_table, &ctx->ref_rows, &ctx->body_shapes, &ctx->body_activities, &ctx->body_bounds, &ctx->color_refs, &ctx->color_priorities, &ctx->color_body_min, &ctx->color_body_mask, &ctx->color_out, &ctx->color_lists, &ctx->color_counts, &ctx->source_bundle_flags, &ctx->refs32, &ctx->prestep32, &ctx->impulses32, &ctx->tb_table, &ctx->tdesc_table, &ctx->work_table, &ctx->map_table,
                            &ctx->bodies_per_type, &ctx->kinematics_dev, &ctx->program_dev, &ctx->frame_params_dev, &ctx->error_dev, &ctx->exchange_staging};
    for (auto b : bufs) b->release();
    ctx->shape_bounds.release();
    ctx->raw_arena.release();
    ctx->pinned_arena.release();
    if (ctx->frame_params_host) cudaFreeHost(ctx->frame_params_host);
    for (auto ev : ctx->user_events)
        if (ev) cudaEventDestroy(ev);
    for (auto& st : ctx->chunk_stage) {
        if (st.host) cudaFreeHost(st.host);
        if (st.done) cudaEventDestroy(st.done);
    }
    for (auto ev : ctx->profile_events) cudaEventDestroy(ev);
    cudaEvent_t evs[] = {ctx->ev_solve_begin, ctx->ev_solve_end, ctx->ev_up_begin, ctx->ev_up_end, ctx->ev_down_begin, ctx->ev_down_end};
    for (auto ev : evs)
        if (ev) cudaEventDestroy(ev);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return BEPUCUDA_OK;
}

const char* bepucuda_last_error(bepucuda_ctx* ctx) { return ctx ? ctx->error.c_str() : "null context"; }

int32_t bepucuda_host_register(bepucuda_ctx* ctx, void* ptr, int64_t bytes) {
    if (!ctx || !ptr || bytes <= 0) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "host_register: bad arguments");
    CK(cudaSetDevice(ctx->device));
    CK(cudaHostRegister(ptr, (size_t)bytes, cudaHostRegisterMapped | cudaHostRegisterPortable));
    void* dev = nullptr;
    CK(cudaHostGetDevicePointer(&dev, ptr, 0));
    ctx->host_ranges.push_back({(char*)ptr, (size_t)bytes, (char*)dev});
    return BEPUCUDA_OK;
}
int32_t bepucuda_host_unregister(bepucuda_ctx* ctx, void* ptr) {
    if (!ctx || !ptr) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "host_unregister: bad arguments");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaHostUnregister(ptr));
    for (size_t i = 0; i < ctx->host_ranges.size(); ++i)
        if (ctx->host_ranges[i].host == (char*)ptr) { ctx->host_ranges.erase(ctx->host_ranges.begin() + i); break; }
    return BEPUCUDA_OK;
}

int32_t bepucuda_set_solve_description(bepucuda_ctx* ctx, int32_t substep_count, const int32_t* its, int32_t fallback_batch_threshold) {
    if (!ctx || substep_count < 1 || !its || fallback_batch_threshold < 1) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "set_solve_description: bad arguments");
    for (int i = 0; i < substep_count; ++i)
        if (its[i] < 0) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "set_solve_description: negative iteration count");
    std::vector<int32_t> v(its, its + substep_count);
    const bool threshold_changed = fallback_batch_threshold != ctx->fallback_threshold;
    const bool changed = v != ctx->iterations || threshold_changed;
    ctx->iterations = v;
    ctx->fallback_threshold = fallback_batch_threshold;
    if (threshold_changed && ctx->constraints_ready) ctx->constraints_ready = false;  // fallback split must be redone
    if (changed && ctx->constraints_ready) {
        CK(cudaSetDevice(ctx->device));
        return upload_program(ctx);
    }
    return BEPUCUDA_OK;
}

int32_t bepucuda_set_integrator(bepucuda_ctx* ctx, const bepucuda_integrator_desc* desc) {
    if (!ctx || !desc) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "set_integrator: bad arguments");
    if (desc->angular_integration_mode < 0 || desc->angular_integration_mode > 2) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "set_integrator: unknown AngularIntegrationMode");
    const bool kin_changed = (desc->integrate_velocity_for_kinematics != 0) != (ctx->integ.integrate_velocity_for_kinematics != 0);
    ctx->integ = *desc;
    ctx->integ_set = true;
    if (kin_changed && ctx->constraints_ready) {
        CK(cudaSetDevice(ctx->device));
        return upload_program(ctx);
    }
    return BEPUCUDA_OK;
}

int32_t bepucuda_upload_bodies(bepucuda_ctx* ctx, const void* body_dynamics, int32_t body_count) {
    if (!ctx || body_count < 0 || (body_count > 0 && !body_dynamics)) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "upload_bodies: bad arguments");
    if ((uint32_t)body_count > kRefIndexMask) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "upload_bodies: too many bodies");
    CK(cudaSetDevice(ctx->device));
    open_upload_window(ctx);
    const size_t n = (size_t)body_count;
    if (body_count != ctx->body_count) {
        // constrained flags / ownership depend on the body count; force a rebuild of topology products.
        if (ctx->constraints_ready) ctx->constraints_ready = false;
        invalidate_graph(ctx);
    }
    CK(ctx->raw_bodies.reserve(n * 128));
    CK(ctx->pose.reserve(n * 32));
    CK(ctx->velocity.reserve(n * 32));
    CK(ctx->inertia_local.reserve(n * 32));
    CK(ctx->inertia_world.reserve(n * 32));
    const size_t old_constrained_cap = ctx->constrained.capacity;
    CK(ctx->constrained.reserve(n + 1));
    if (ctx->constrained.capacity != old_constrained_cap) CK(cudaMemsetAsync(ctx->constrained.ptr, 0, ctx->constrained.capacity, ctx->stream));
    ctx->body_count = body_count;
    BodyBuffers B{};
    B.pose = ctx->pose.as<float4>();
    B.velocity = ctx->velocity.as<float4>();
    B.inertia_local = ctx->inertia_local.as<float4>();
    B.inertia_world = ctx->inertia_world.as<float4>();
    B.constrained = ctx->constrained.as<uint8_t>();
    B.count = body_count;
    if (B.pose != ctx->B.pose || B.velocity != ctx->B.velocity || B.inertia_local != ctx->B.inertia_local || B.inertia_world != ctx->B.inertia_world ||
        B.constrained != ctx->B.constrained || B.count != ctx->B.count)
        invalidate_graph(ctx);  // kernel arguments are baked into graph nodes
    ctx->B = B;
    if (body_count > 0) {
        CK(cudaMemcpyAsync(ctx->raw_bodies.ptr, body_dynamics, n * 128, cudaMemcpyHostToDevice, ctx->stream));
        ctx->h2d_accum += (int64_t)n * 128;
        launch_split_bodies(ctx->raw_bodies.ptr, body_count, ctx->B, ctx->stream);
        CK(cudaGetLastError());
    }
    return BEPUCUDA_OK;
}

int32_t bepucuda_begin_constraints(bepucuda_ctx* ctx, int32_t source_bundle_width, int32_t batch_count) {
    if (!ctx || source_bundle_width < 1 || source_bundle_width > 64 || batch_count < 0) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "begin_constraints: bad arguments");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));  // staging arenas are recycled below
    open_upload_window(ctx);
    ctx->W = source_bundle_width;
    ctx->batch_count = batch_count;
    ctx->sources.clear();
    ctx->pending_h2d.clear();  // queued refreshes target raw-arena addresses that are recycled below; a re-describe uploads everything anyway
    ctx->raw_arena.reset();
    ctx->pinned_arena.reset();
    ctx->constraints_open = true;
    ctx->constraints_ready = false;
    invalidate_graph(ctx);
    return BEPUCUDA_OK;
}

int32_t bepucuda_upload_type_batch(bepucuda_ctx* ctx, int32_t batch_index, int32_t type_batch_index, int32_t type_id, int32_t constraint_count,
                                   const int32_t* body_references, const float* prestep, float* accumulated_impulses) {
    if (!ctx) return BEPUCUDA_ERR_INVALID_ARGUMENT;
    if (!ctx->constraints_open) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "upload_type_batch outside begin/end_constraints");
    if (batch_index < 0 || batch_index >= ctx->batch_count || type_batch_index < 0 || constraint_count < 0)
        return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "upload_type_batch: bad indices");
    const TypeInfo* t = get_type_info(type_id);
    if (!t) return fail(ctx, BEPUCUDA_ERR_UNSUPPORTED_TYPE, "upload_type_batch: unsupported constraint type id " + std::to_string(type_id));
    if (constraint_count == 0) return BEPUCUDA_OK;
    if (!body_references || !prestep || !accumulated_impulses) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "upload_type_batch: null buffer");
    CK(cudaSetDevice(ctx->device));
    const int W = ctx->W;
    const size_t bundles = ((size_t)constraint_count + W - 1) / W;
    SourceTypeBatch s{};
    s.batch_index = batch_index; s.type_batch_index = type_batch_index; s.type_id = type_id; s.count = constraint_count;
    s.host_impulses = accumulated_impulses;
    s.refs_bytes = bundles * t->bodies * W * 4;
    s.prestep_bytes = bundles * t->prestep_rows * W * 4;
    s.impulse_bytes = bundles * t->impulse_rows * W * 4;
    cudaError_t e = cudaSuccess;
    s.raw_refs = (int32_t*)ctx->raw_arena.alloc(s.refs_bytes, &e);
    s.raw_prestep = (float*)ctx->raw_arena.alloc(s.prestep_bytes, &e);
    s.raw_impulses = (float*)ctx->raw_arena.alloc(s.impulse_bytes, &e);
    if (!s.raw_refs || !s.raw_prestep || !s.raw_impulses) return cuda_fail(ctx, e, "raw arena");
    int rc;
    if ((rc = copy_in(ctx, s.raw_refs, body_references, s.refs_bytes)) != BEPUCUDA_OK) return rc;
    if ((rc = copy_in(ctx, s.raw_prestep, prestep, s.prestep_bytes)) != BEPUCUDA_OK) return rc;
    if ((rc = copy_in(ctx, s.raw_impulses, accumulated_impulses, s.impulse_bytes)) != BEPUCUDA_OK) return rc;
    if (batch_index >= ctx->fallback_threshold) s.host_refs.assign(body_references, body_references + s.refs_bytes / 4);
    ctx->sources.push_back(std::move(s));
    return BEPUCUDA_OK;
}

int32_t bepucuda_set_constrained_kinematics(bepucuda_ctx* ctx, const int32_t* body_indices, int32_t count) {
    if (!ctx || count < 0 || (count > 0 && !body_indices)) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "set_constrained_kinematics: bad arguments");
    ctx->kinematics.assign(body_indices, body_indices + count);
    if (ctx->constraints_ready) ctx->constraints_ready = false;
    return BEPUCUDA_OK;
}

int32_t bepucuda_end_constraints(bepucuda_ctx* ctx) {
    if (!ctx) return BEPUCUDA_ERR_INVALID_ARGUMENT;
    if (!ctx->constraints_open) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "end_constraints without begin_constraints");
    CK(cudaSetDevice(ctx->device));
    const int W = ctx->W;
    std::stable_sort(ctx->sources.begin(), ctx->sources.end(), [](const SourceTypeBatch& a, const SourceTypeBatch& b) {
        return a.batch_index != b.batch_index ? a.batch_index < b.batch_index : a.type_batch_index < b.type_batch_index;
    });

    std::vector<int32_t> source_bundle_base(ctx->sources.size());
    int32_t total_source_bundles = 0;
    for (size_t si = 0; si < ctx->sources.size(); ++si) {
        source_bundle_base[si] = total_source_bundles;
        total_source_bundles += (ctx->sources[si].count + W - 1) / W;
    }

    // ---- device batches: synchronized batches in order, then dependency levels of the sequential fallback batch ----
    ctx->tbs.clear();
    ctx->tdescs.clear();
    std::vector<int32_t> maps;                       // concatenated slot->source maps for fallback-level type batches
    std::vector<size_t> map_offset;                  // per device tb: offset into maps or SIZE_MAX
    std::vector<std::vector<int>> batch_tbs;         // device batch -> device tb indices
    int64_t constraint_count = 0;
    ctx->sync_batch_count = 0;
    ctx->fallback_levels = 0;
    {
        int current_batch = -1;
        for (size_t si = 0; si < ctx->sources.size(); ++si) {
            SourceTypeBatch& s = ctx->sources[si];
            s.device_tbs.clear();
            if (s.batch_index >= ctx->fallback_threshold) continue;
            // device batch index == host batch index (empty batches stay as empty slots): ranks of a sharded graph then agree on batch numbers
            while ((int)batch_tbs.size() <= s.batch_index) batch_tbs.emplace_back();
            current_batch = s.batch_index;
            const TypeInfo* t = get_type_info(s.type_id);
            DeviceTypeBatch d{};
            d.type_id = s.type_id;
            d.bundle_count = (s.count + 31) / 32;
            d.device_batch = s.batch_index;
            TransposeDesc td{s.raw_refs, s.raw_prestep, s.raw_impulses, nullptr, s.count, t->bodies, t->prestep_rows, t->impulse_rows, source_bundle_base[si], 0, nullptr, nullptr};
            s.device_tbs.push_back((int)ctx->tbs.size());
            batch_tbs[s.batch_index].push_back((int)ctx->tbs.size());
            ctx->tbs.push_back(d);
            ctx->tdescs.push_back(td);
            map_offset.push_back(SIZE_MAX);
            s.live = s.count;
            constraint_count += s.count;
        }
        if (ctx->peer_mode) {
            // every rank runs the exchange of every batch, also of batches it has no constraint in
            while ((int)batch_tbs.size() < std::min(ctx->batch_count, ctx->fallback_threshold)) batch_tbs.emplace_back();
            for (const SourceTypeBatch& src : ctx->sources)
                if (src.batch_index >= ctx->fallback_threshold) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "end_constraints: the sequential fallback batch is not supported across ranks");
        }
        if (ctx->exchange && !ctx->peer_mode) {
            // sharded batches through the exchange callback: levels computed from one rank's constraints differ between ranks, so would the number of
            // collectives per step (a hang), and level indices are not comparable across ranks
            for (const SourceTypeBatch& src : ctx->sources)
                if (src.batch_index >= ctx->fallback_threshold) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "end_constraints: the sequential fallback batch is not supported with an exchange callback");
        }
        (void)current_batch;
        ctx->sync_batch_count = (int)batch_tbs.size();
    }
    {
        // Fallback levelisation. The reference executes fallback bundles one after another on a single thread
        // (Solver_Solve.cs:L546-583); within a bundle no dynamic body repeats (TypeProcessor.cs:L338-359). A constraint's
        // level is 1 + the highest level of any earlier-bundle constraint sharing a dynamic body with it: executing levels in
        // order with a barrier in between preserves every read-after-write of the sequential loop, so results are identical.
        std::vector<int32_t> last_level;  // per body: highest level assigned so far (0 = none)
        struct Slot { int level; int source; int constraint; };
        std::vector<Slot> slots;
        bool any = false;
        for (size_t si = 0; si < ctx->sources.size(); ++si) {
            SourceTypeBatch& s = ctx->sources[si];
            if (s.batch_index < ctx->fallback_threshold) continue;
            if (!any) { last_level.assign((size_t)ctx->body_count, 0); any = true; }
            s.live = 0;
            const TypeInfo* t = get_type_info(s.type_id);
            const int nb = t->bodies;
            const int bundles = (s.count + W - 1) / W;
            std::vector<int> lane_level(W);
            for (int k = 0; k < bundles; ++k) {
                // all lanes of a bundle read the state left by earlier bundles
                for (int l = 0; l < W; ++l) {
                    lane_level[l] = 0;
                    const int c = k * W + l;
                    if (c >= s.count) continue;
                    const int32_t first = s.host_refs[((size_t)k * nb) * W + l];
                    if (first < 0) continue;  // hole
                    int lvl = 0;
                    for (int b = 0; b < nb; ++b) {
                        const int32_t enc = s.host_refs[((size_t)k * nb + b) * W + l];
                        if (enc < 0 || ((uint32_t)enc & kRefKinematicBit)) continue;
                        const uint32_t idx = (uint32_t)enc & kRefIndexMask;
                        if ((int)idx >= ctx->body_count) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "end_constraints: body reference out of range");
                        lvl = std::max(lvl, last_level[idx]);
                    }
                    lane_level[l] = lvl + 1;
                }
                for (int l = 0; l < W; ++l) {
                    if (lane_level[l] == 0) continue;
                    for (int b = 0; b < nb; ++b) {
                        const int32_t enc = s.host_refs[((size_t)k * nb + b) * W + l];
                        if (enc < 0 || ((uint32_t)enc & kRefKinematicBit)) continue;
                        last_level[(uint32_t)enc & kRefIndexMask] = lane_level[l];
                    }
                    // TypeProcessor.cs:L338-359: a fallback bundle never holds a dynamic body twice (two lanes of one level would race on its record)
                    for (int l2 = 0; l2 < l; ++l2) {
                        if (lane_level[l2] == 0) continue;
                        for (int b = 0; b < nb; ++b) {
                            const int32_t e1 = s.host_refs[((size_t)k * nb + b) * W + l];
                            if (e1 < 0 || ((uint32_t)e1 & kRefKinematicBit)) continue;
                            for (int b2 = 0; b2 < nb; ++b2) {
                                const int32_t e2 = s.host_refs[((size_t)k * nb + b2) * W + l2];
                                if (e2 >= 0 && !((uint32_t)e2 & kRefKinematicBit) && (((uint32_t)e1 ^ (uint32_t)e2) & kRefIndexMask) == 0)
                                    return fail(ctx, BEPUCUDA_ERR_BATCH_INVARIANT, "end_constraints: a fallback bundle references the same dynamic body more than once");
                            }
                        }
                    }
                    slots.push_back({lane_level[l], (int)si, k * W + l});
                    ++s.live;
                    ++constraint_count;
                }
            }
        }
        if (any) {
            std::stable_sort(slots.begin(), slots.end(), [](const Slot& a, const Slot& b) { return a.level != b.level ? a.level < b.level : a.source < b.source; });
            size_t i = 0;
            while (i < slots.size()) {
                const int level = slots[i].level;
                batch_tbs.emplace_back();
                ++ctx->fallback_levels;
                while (i < slots.size() && slots[i].level == level) {
                    const int source = slots[i].source;
                    size_t j = i;
                    while (j < slots.size() && slots[j].level == level && slots[j].source == source) ++j;
                    SourceTypeBatch& s = ctx->sources[source];
                    const TypeInfo* t = get_type_info(s.type_id);
                    const int n = (int)(j - i);
                    DeviceTypeBatch d{};
                    d.type_id = s.type_id;
                    d.bundle_count = (n + 31) / 32;
                    d.device_batch = (int)batch_tbs.size() - 1;
                    map_offset.push_back(maps.size());
                    for (size_t q = i; q < j; ++q) maps.push_back(slots[q].constraint);
                    for (int q = n; q < d.bundle_count * 32; ++q) maps.push_back(-1);
                    TransposeDesc td{s.raw_refs, s.raw_prestep, s.raw_impulses, nullptr, s.count, t->bodies, t->prestep_rows, t->impulse_rows, source_bundle_base[source], 0, nullptr, nullptr};
                    s.device_tbs.push_back((int)ctx->tbs.size());
                    batch_tbs.back().push_back((int)ctx->tbs.size());
                    ctx->tbs.push_back(d);
                    ctx->tdescs.push_back(td);
                    i = j;
                }
            }
        }
    }

    // ---- device arenas for the AOSOA-32 image ----
    size_t refs_floats = 0, prestep_floats = 0, impulse_floats = 0;
    std::vector<size_t> ro(ctx->tbs.size()), po(ctx->tbs.size()), io(ctx->tbs.size());
    for (size_t i = 0; i < ctx->tbs.size(); ++i) {
        const TypeInfo* t = get_type_info(ctx->tbs[i].type_id);
        ro[i] = refs_floats; po[i] = prestep_floats; io[i] = impulse_floats;
        refs_floats += (size_t)ctx->tbs[i].bundle_count * t->bodies * 32;
        prestep_floats += (size_t)ctx->tbs[i].bundle_count * t->prestep_rows * 32;
        impulse_floats += (size_t)ctx->tbs[i].bundle_count * t->impulse_rows * 32;
    }
    CK(ctx->refs32.reserve(refs_floats * 4 + 1024));  // slack: solver warps always read two body-reference rows
    ctx->refs_words = refs_floats;
    CK(ctx->prestep32.reserve(prestep_floats * 4 + 4));
    CK(ctx->impulses32.reserve(impulse_floats * 4 + 4));
    CK(ctx->map_table.reserve(maps.size() * 4 + 4));
    for (size_t i = 0; i < ctx->tbs.size(); ++i) {
        ctx->tbs[i].refs = ctx->refs32.as<int32_t>() + ro[i];
        ctx->tbs[i].prestep = ctx->prestep32.as<float>() + po[i];
        ctx->tbs[i].impulses = ctx->impulses32.as<float>() + io[i];
        ctx->tdescs[i].map = map_offset[i] == SIZE_MAX ? nullptr : ctx->map_table.as<int32_t>() + map_offset[i];
    }

    // ---- work lists: per device batch (one warp per bundle), then the incremental-update list over all contact bundles ----
    ctx->work.clear();
    ctx->bundle_live.clear();
    ctx->batch_work.clear();
    auto live_in_bundle = [&](int tb, int k) {
        // identity-mapped type batches: lanes beyond the source count are padding; mapped (fallback level) ones: -1 entries are padding
        if (map_offset[tb] == SIZE_MAX) return std::max(0, std::min(32, ctx->tdescs[tb].src_count - k * 32));
        int n = 0;
        for (int l = 0; l < 32; ++l) n += maps[map_offset[tb] + (size_t)k * 32 + l] >= 0;
        return n;
    };
    for (auto& list : batch_tbs) {
        const int begin = (int)ctx->work.size();
        for (int tb : list)
            for (int k = 0; k < ctx->tbs[tb].bundle_count; ++k) { ctx->work.push_back({tb, k}); ctx->bundle_live.push_back(live_in_bundle(tb, k)); }
        ctx->batch_work.push_back({begin, (int)ctx->work.size() - begin});
    }
    ctx->all_work_count = (int)ctx->work.size();
    ctx->inc_work_begin = (int)ctx->work.size();
    for (size_t tb = 0; tb < ctx->tbs.size(); ++tb)
        if (get_type_info(ctx->tbs[tb].type_id)->incremental)
            for (int k = 0; k < ctx->tbs[tb].bundle_count; ++k) { ctx->work.push_back({(int)tb, k}); ctx->bundle_live.push_back(live_in_bundle((int)tb, k)); }
    ctx->inc_work_count = (int)ctx->work.size() - ctx->inc_work_begin;

    ctx->records.resize(ctx->work.size());
    for (size_t i = 0; i < ctx->work.size(); ++i) {
        const WorkItem& w = ctx->work[i];
        const DeviceTypeBatch& tb = ctx->tbs[w.type_batch];
        const TypeInfo* t = get_type_info(tb.type_id);
        WorkRecord r{};
        r.refs = tb.refs + (size_t)w.bundle * t->bodies * 32;
        r.prestep = tb.prestep + (size_t)w.bundle * t->prestep_rows * 32;
        r.impulses = tb.impulses + (size_t)w.bundle * t->impulse_rows * 32;
        r.type_id = tb.type_id;
        r.live_lanes = ctx->bundle_live[i];
        ctx->records[i] = r;
    }

    // ---- upload tables ----
    int32_t bodies_per_type[64];
    for (int i = 0; i < 64; ++i) bodies_per_type[i] = get_type_info(i) ? get_type_info(i)->bodies : 0;
    CK(ctx->tb_table.reserve(ctx->tbs.size() * sizeof(DeviceTypeBatch) + 16));
    CK(ctx->tdesc_table.reserve(ctx->tdescs.size() * sizeof(TransposeDesc) + 16));
    CK(ctx->work_table.reserve(ctx->work.size() * sizeof(WorkItem) + 16));
    CK(ctx->record_table.reserve(ctx->records.size() * sizeof(WorkRecord) + 64));
    CK(ctx->bodies_per_type.reserve(sizeof(bodies_per_type)));
    CK(ctx->kinematics_dev.reserve(ctx->kinematics.size() * 4 + 4));
    if (!ctx->tbs.empty()) CK(cudaMemcpyAsync(ctx->tb_table.ptr, ctx->tbs.data(), ctx->tbs.size() * sizeof(DeviceTypeBatch), cudaMemcpyHostToDevice, ctx->stream));
    if (!ctx->tdescs.empty()) CK(cudaMemcpyAsync(ctx->tdesc_table.ptr, ctx->tdescs.data(), ctx->tdescs.size() * sizeof(TransposeDesc), cudaMemcpyHostToDevice, ctx->stream));
    if (!ctx->work.empty()) CK(cudaMemcpyAsync(ctx->work_table.ptr, ctx->work.data(), ctx->work.size() * sizeof(WorkItem), cudaMemcpyHostToDevice, ctx->stream));
    if (!ctx->records.empty()) CK(cudaMemcpyAsync(ctx->record_table.ptr, ctx->records.data(), ctx->records.size() * sizeof(WorkRecord), cudaMemcpyHostToDevice, ctx->stream));
    if (!maps.empty()) CK(cudaMemcpyAsync(ctx->map_table.ptr, maps.data(), maps.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->bodies_per_type.ptr, bodies_per_type, sizeof(bodies_per_type), cudaMemcpyHostToDevice, ctx->stream));
    if (!ctx->kinematics.empty()) CK(cudaMemcpyAsync(ctx->kinematics_dev.ptr, ctx->kinematics.data(), ctx->kinematics.size() * 4, cudaMemcpyHostToDevice, ctx->stream));

    // ---- transposition into AOSOA-32 + ownership analysis ----
    { int rc = flush_chunks(ctx, ctx->pending_h2d); if (rc != BEPUCUDA_OK) return rc; }
    launch_transpose_in_all(ctx->tb_table.as<DeviceTypeBatch>(), ctx->tdesc_table.as<TransposeDesc>(), ctx->work_table.as<WorkItem>(), ctx->all_work_count, W,
                            kTransposeRefs | kTransposePrestep | kTransposeImpulses, ctx->stream);
    const size_t nb = (size_t)std::max(ctx->body_count, 1);
    CK(ctx->first_batch.reserve(nb * 4));
    CK(ctx->sync_refcount.reserve(nb * 4));
    CK(ctx->sync_mask.reserve(nb * 8));
    launch_fill_i32(ctx->first_batch.as<int32_t>(), nb, 0x7fffffff, ctx->stream);
    CK(cudaMemsetAsync(ctx->sync_refcount.ptr, 0, nb * 4, ctx->stream));
    CK(cudaMemsetAsync(ctx->sync_mask.ptr, 0, nb * 8, ctx->stream));
    CK(cudaMemsetAsync(ctx->constrained.ptr, 0, nb, ctx->stream));
    CK(cudaMemsetAsync(ctx->error_dev.ptr, 0, 32, ctx->stream));
    CK(ctx->source_bundle_flags.reserve((size_t)std::max(total_source_bundles, 1) * 16));
    CK(cudaMemsetAsync(ctx->source_bundle_flags.ptr, 0, (size_t)std::max(total_source_bundles, 1) * 16, ctx->stream));
    launch_ownership_pass1(ctx->tb_table.as<DeviceTypeBatch>(), ctx->work_table.as<WorkItem>(), ctx->all_work_count, ctx->bodies_per_type.as<int32_t>(), ctx->sync_batch_count,
                           ctx->body_count, ctx->first_batch.as<int32_t>(), ctx->sync_refcount.as<int32_t>(), (unsigned long long*)ctx->sync_mask.ptr, ctx->error_dev.as<int32_t>(),
                           ctx->stream);
    if (ctx->peer_mode && nb > 0) {
        // peer sharding: the integration owner of a body is the lowest batch referencing it on ANY rank (computed by the host over the whole graph)
        if ((int)ctx->global_first_batch.size() != ctx->body_count) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "end_constraints: bepucuda_shard_set_global was not called for this body count");
        CK(cudaMemcpyAsync(ctx->first_batch.ptr, ctx->global_first_batch.data(), (size_t)ctx->body_count * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    if (ctx->exchange && !ctx->peer_mode && nb > 0) {
        // sharded batches: the integration owner of a body is the lowest batch referencing it on ANY rank
        if (ctx->exchange(ctx->exchange_user, ctx->first_batch.ptr, (int64_t)ctx->body_count, 1, (void*)ctx->stream) != 0)
            return fail(ctx, BEPUCUDA_ERR_CUDA, "end_constraints: the exchange callback failed (first-batch minimum)");
    }
    launch_ownership_rest(ctx->tb_table.as<DeviceTypeBatch>(), ctx->work_table.as<WorkItem>(), ctx->all_work_count, ctx->bodies_per_type.as<int32_t>(), ctx->body_count,
                          ctx->first_batch.as<int32_t>(), ctx->sync_refcount.as<int32_t>(), (const unsigned long long*)ctx->sync_mask.ptr, ctx->constrained.as<uint8_t>(),
                          ctx->kinematics_dev.as<int32_t>(), (int)ctx->kinematics.size(), ctx->error_dev.as<int32_t>(), ctx->tdesc_table.as<TransposeDesc>(), W,
                          ctx->source_bundle_flags.as<int32_t>(), ctx->stream);
    if (ctx->peer_mode && nb > 0) {
        CK(cudaMemcpyAsync(ctx->constrained.ptr, ctx->global_constrained.data(), (size_t)ctx->body_count, cudaMemcpyHostToDevice, ctx->stream));
        // the (body, destination rank) lists of every batch, back to back
        std::vector<uint32_t> all;
        ctx->push_range.assign(ctx->sync_batch_count, {0, 0});
        for (int b = 0; b < ctx->sync_batch_count; ++b) {
            auto it = ctx->pushes_by_batch.find(b);
            if (it == ctx->pushes_by_batch.end()) continue;
            ctx->push_range[b] = {all.size(), (int)it->second.size()};
            all.insert(all.end(), it->second.begin(), it->second.end());
        }
        CK(ctx->pushes_dev.reserve(all.size() * 4 + 16));
        if (!all.empty()) CK(cudaMemcpy(ctx->pushes_dev.ptr, all.data(), all.size() * 4, cudaMemcpyHostToDevice));
    }
    if (ctx->exchange && !ctx->peer_mode && nb > 0) {
        // ... and a body is "constrained" (final pose pass) if any rank constrains it
        CK(ctx->exchange_staging.reserve((size_t)nb * 24 * 4));
        launch_widen_u8(ctx->constrained.as<uint8_t>(), ctx->exchange_staging.as<int32_t>(), (size_t)ctx->body_count, ctx->stream);
        if (ctx->exchange(ctx->exchange_user, ctx->exchange_staging.ptr, (int64_t)ctx->body_count, 0, (void*)ctx->stream) != 0)
            return fail(ctx, BEPUCUDA_ERR_CUDA, "end_constraints: the exchange callback failed (constrained mask)");
        launch_narrow_i32(ctx->exchange_staging.as<int32_t>(), ctx->constrained.as<uint8_t>(), (size_t)ctx->body_count, ctx->stream);
    }
    if (ctx->peer_mode && !ctx->body_masks.empty()) {
        // fused pushes: per body reference, the other ranks that need what this rank's constraint writes
        if ((int)ctx->body_masks.size() != ctx->body_count) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "end_constraints: bepucuda_shard_set_body_masks was called for another body count");
        CK(ctx->peer32.reserve(ctx->refs_words * 4 + 1024));
        CK(ctx->body_masks_dev.reserve((size_t)ctx->body_count + 16));
        CK(cudaMemcpyAsync(ctx->body_masks_dev.ptr, ctx->body_masks.data(), (size_t)ctx->body_count, cudaMemcpyHostToDevice, ctx->stream));
        launch_fill_peer_masks(ctx->refs32.as<int32_t>(), ctx->peer32.as<uint32_t>(), ctx->refs_words, ctx->body_masks_dev.as<uint8_t>(), ctx->peers.rank, ctx->stream);
        // boundary bundles (any lane writes a shared body) go to the front of their batch and carry kRecordBoundaryBit: they are scheduled first, and
        // the flag barrier of the stage involves only them (ShardStage)
        const int n_rec = ctx->all_work_count;
        CK(ctx->boundary_flags_dev.reserve((size_t)n_rec + 16));
        launch_boundary_flags(ctx->record_table.as<WorkRecord>(), n_rec, ctx->bodies_per_type.as<int32_t>(), (long long)(ctx->peer32.as<int32_t>() - ctx->refs32.as<int32_t>()),
                              ctx->boundary_flags_dev.as<uint8_t>(), ctx->stream);
        std::vector<uint8_t> is_boundary((size_t)n_rec);
        if (n_rec > 0) CK(cudaMemcpyAsync(is_boundary.data(), ctx->boundary_flags_dev.ptr, (size_t)n_rec, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->boundary_count.assign(ctx->batch_work.size(), 0);
        std::vector<WorkRecord> sorted;
        for (size_t b = 0; b < ctx->batch_work.size(); ++b) {
            const int begin = ctx->batch_work[b].first, count = ctx->batch_work[b].second;
            sorted.clear();
            for (int pass = 0; pass < 2; ++pass)
                for (int i = begin; i < begin + count; ++i)
                    if ((is_boundary[(size_t)i] != 0) == (pass == 0)) {
                        WorkRecord r = ctx->records[(size_t)i];
                        r.live_lanes = (r.live_lanes & ~kRecordBoundaryBit) | (pass == 0 ? kRecordBoundaryBit : 0);
                        sorted.push_back(r);
                        ctx->boundary_count[b] += pass == 0;
                    }
            std::copy(sorted.begin(), sorted.end(), ctx->records.begin() + begin);
        }
        if (n_rec > 0) CK(cudaMemcpyAsync(ctx->record_table.ptr, ctx->records.data(), (size_t)n_rec * sizeof(WorkRecord), cudaMemcpyHostToDevice, ctx->stream));
    }
    // the first two body-reference rows of every work record, packed in work-list order (they carry the ownership bits set above)
    CK(ctx->ref_rows.reserve((size_t)std::max<size_t>(ctx->records.size(), 1) * 64 * 4));
    launch_pack_ref_rows(ctx->record_table.as<WorkRecord>(), (int)ctx->records.size(), ctx->ref_rows.as<int32_t>(), ctx->stream);
    CK(cudaGetLastError());
    int32_t err = 0;
    CK(cudaMemcpyAsync(&err, ctx->error_dev.ptr, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));  // also guarantees the std::vector sources of the copies above were consumed
    if (err == 1) return fail(ctx, BEPUCUDA_ERR_BATCH_INVARIANT, "end_constraints: a synchronized batch references the same dynamic body more than once");
    if (err == 2) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "end_constraints: body reference out of range");

    ctx->timings.constraint_count = constraint_count;
    ctx->timings.device_batch_count = (int)batch_tbs.size();
    ctx->timings.fallback_level_count = ctx->fallback_levels;
    ctx->constraints_open = false;
    ctx->constraints_ready = true;
    ctx->data_dirty = false;
    return upload_program(ctx);
}

int32_t bepucuda_update_type_batch(bepucuda_ctx* ctx, int32_t batch_index, int32_t type_batch_index, const float* prestep, float* accumulated_impulses) {
    if (!ctx || !prestep || !accumulated_impulses) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "update_type_batch: bad arguments");
    if (!ctx->constraints_ready) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "update_type_batch before end_constraints");
    CK(cudaSetDevice(ctx->device));
    open_upload_window(ctx);
    for (auto& s : ctx->sources)
        if (s.batch_index == batch_index && s.type_batch_index == type_batch_index) {
            char* alias_p = map_host(ctx, prestep, s.prestep_bytes);
            char* alias_i = map_host(ctx, accumulated_impulses, s.impulse_bytes);
            if (alias_p && alias_i) {
                queue_chunks(ctx->pending_h2d, s.raw_prestep, alias_p, s.prestep_bytes);
                queue_chunks(ctx->pending_h2d, s.raw_impulses, alias_i, s.impulse_bytes);
            } else {
                // Direct copies only: the pinned staging arena is recycled per begin_constraints, not per frame.
                CK(cudaMemcpyAsync(s.raw_prestep, prestep, s.prestep_bytes, cudaMemcpyHostToDevice, ctx->stream));
                CK(cudaMemcpyAsync(s.raw_impulses, accumulated_impulses, s.impulse_bytes, cudaMemcpyHostToDevice, ctx->stream));
            }
            ctx->h2d_accum += (int64_t)(s.prestep_bytes + s.impulse_bytes);
            s.host_impulses = accumulated_impulses;
            if (s.resident_impulses) { s.resident_impulses = false; s.redistribute = false; ctx->descs_dirty = true; }  // the host took the impulses back
            ctx->data_dirty = true;
            return BEPUCUDA_OK;
        }
    return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "update_type_batch: unknown type batch");
}

static int contact_count_of_type(int type_id) {
    if (type_id >= 0 && type_id <= 7) return (type_id & 3) + 1;
    if (type_id >= 8 && type_id <= 10) return type_id - 6;
    if (type_id >= 15 && type_id <= 17) return type_id - 13;
    return 0;
}
static SourceTypeBatch* find_source(bepucuda_ctx* ctx, int32_t batch_index, int32_t type_batch_index) {
    for (auto& s : ctx->sources)
        if (s.batch_index == batch_index && s.type_batch_index == type_batch_index) return &s;
    return nullptr;
}
static int ensure_feature_arrays(bepucuda_ctx* ctx, SourceTypeBatch& s) {
    if (s.raw_features_old) return BEPUCUDA_OK;
    s.feature_bytes = (size_t)s.count * contact_count_of_type(s.type_id) * sizeof(int32_t);
    cudaError_t e = cudaSuccess;
    s.raw_features_old = (int32_t*)ctx->raw_arena.alloc(s.feature_bytes, &e);
    s.raw_features_new = (int32_t*)ctx->raw_arena.alloc(s.feature_bytes, &e);
    if (!s.raw_features_old || !s.raw_features_new) return cuda_fail(ctx, e, "raw arena (contact feature ids)");
    return BEPUCUDA_OK;
}

int32_t bepucuda_set_contact_features(bepucuda_ctx* ctx, int32_t batch_index, int32_t type_batch_index, const int32_t* feature_ids) {
    if (!ctx || !feature_ids) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "set_contact_features: bad arguments");
    if (!ctx->constraints_open && !ctx->constraints_ready) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "set_contact_features before the type batch was uploaded");
    SourceTypeBatch* s = find_source(ctx, batch_index, type_batch_index);
    if (!s) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "set_contact_features: unknown type batch");
    if (contact_count_of_type(s->type_id) == 0) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "set_contact_features: not a contact constraint type");
    CK(cudaSetDevice(ctx->device));
    { int rc = ensure_feature_arrays(ctx, *s); if (rc != BEPUCUDA_OK) return rc; }
    return copy_in(ctx, s->raw_features_old, feature_ids, s->feature_bytes);
}

int32_t bepucuda_update_contacts(bepucuda_ctx* ctx, int32_t batch_index, int32_t type_batch_index, const float* prestep, const int32_t* new_feature_ids) {
    if (!ctx || !prestep || !new_feature_ids) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "update_contacts: bad arguments");
    if (!ctx->constraints_ready) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "update_contacts before end_constraints");
    SourceTypeBatch* s = find_source(ctx, batch_index, type_batch_index);
    if (!s) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "update_contacts: unknown type batch");
    if (!s->raw_features_old) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "update_contacts: bepucuda_set_contact_features was never called for this type batch");
    if (s->redistribute) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "update_contacts: called twice for the same type batch without a solve in between");
    CK(cudaSetDevice(ctx->device));
    open_upload_window(ctx);
    // per-frame path: mapped (registered) host buffers go through the batched zero-copy kernel, anything else is copied directly -- never through the
    // pinned staging arena, which is only recycled by bepucuda_begin_constraints
    const void* srcs[2] = {prestep, new_feature_ids};
    void* dsts[2] = {s->raw_prestep, s->raw_features_new};
    const size_t sizes[2] = {s->prestep_bytes, s->feature_bytes};
    for (int i = 0; i < 2; ++i) {
        if (char* alias = map_host(ctx, srcs[i], sizes[i])) queue_chunks(ctx->pending_h2d, dsts[i], alias, sizes[i]);
        else CK(cudaMemcpyAsync(dsts[i], srcs[i], sizes[i], cudaMemcpyHostToDevice, ctx->stream));
        ctx->h2d_accum += (int64_t)sizes[i];
    }
    s->resident_impulses = true;
    s->redistribute = true;
    ctx->descs_dirty = true;
    ctx->data_dirty = true;
    return BEPUCUDA_OK;
}

int32_t bepucuda_upload_body_motion(bepucuda_ctx* ctx, const void* body_dynamics, int32_t body_count) {
    if (!ctx || !body_dynamics || body_count != ctx->body_count) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "upload_body_motion: bad arguments (the body count must match the last upload_bodies)");
    if (body_count == 0) return BEPUCUDA_OK;
    CK(cudaSetDevice(ctx->device));
    open_upload_window(ctx);
    const size_t n = (size_t)body_count;
    if (char* alias = map_host(ctx, body_dynamics, n * 128)) {
        launch_scatter_body_motion(alias, body_count, ctx->B, ctx->stream);  // 64 of every 128 bytes read straight from the mapped host buffer
    } else {
        CK(cudaMemcpy2DAsync(ctx->raw_bodies.ptr, 128, body_dynamics, 128, 64, n, cudaMemcpyHostToDevice, ctx->stream));
        launch_scatter_body_motion(ctx->raw_bodies.ptr, body_count, ctx->B, ctx->stream);
    }
    CK(cudaGetLastError());
    ctx->h2d_accum += (int64_t)n * 64;
    return BEPUCUDA_OK;
}

int32_t bepucuda_download_body_motion(bepucuda_ctx* ctx, void* out, int32_t body_count) {
    if (!ctx || !out || body_count < 0 || body_count > ctx->body_count) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "download_body_motion: bad arguments");
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventRecord(ctx->ev_down_begin, ctx->stream));
    const size_t n = (size_t)body_count;
    if (char* alias = map_host(ctx, out, n * 128)) {
        launch_gather_body_motion(alias, body_count, ctx->B, ctx->stream);
    } else {
        launch_gather_body_motion(ctx->raw_bodies.ptr, body_count, ctx->B, ctx->stream);
        CK(cudaMemcpy2DAsync(out, 128, ctx->raw_bodies.ptr, 128, 64, n, cudaMemcpyDeviceToHost, ctx->stream));
    }
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev_down_end, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->have_down = true;
    ctx->timings.d2h_bytes = (int64_t)n * 64;
    return BEPUCUDA_OK;
}

int32_t bepucuda_solve(bepucuda_ctx* ctx, float dt) {
    if (!ctx || !(dt > 0)) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "solve: bad arguments");
    CK(cudaSetDevice(ctx->device));
    if (!ctx->constraints_ready) {
        // No constraints were ever described (or the description was invalidated): only legal when nothing was uploaded.
        if (ctx->constraints_open) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "solve inside begin/end_constraints");
        if (!ctx->sources.empty()) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "solve: constraint description is stale; re-run begin/upload/end_constraints");
        int rc = bepucuda_begin_constraints(ctx, ctx->W, 0);
        if (rc == BEPUCUDA_OK) rc = bepucuda_end_constraints(ctx);
        if (rc != BEPUCUDA_OK) return rc;
    }
    { int rc = refresh_device_rows(ctx); if (rc != BEPUCUDA_OK) return rc; }
    if (ctx->up_open) {
        cudaEventRecord(ctx->ev_up_end, ctx->stream);
        ctx->up_open = false;
        ctx->have_up = true;
    }
    ctx->timings.h2d_bytes = ctx->h2d_accum;
    ctx->h2d_accum = 0;
    // frame parameters (previous frame's copy has completed by stream order only after its graph; wait for it before reusing the pinned struct)
    CK(cudaEventSynchronize(ctx->ev_solve_end));
    compute_frame_params(ctx, dt, ctx->frame_params_host);
    ctx->frame_params_host->exchange_base = ctx->exchange_counter;
    ctx->frame_params_host->shard_solve_index = ctx->shard_solve_index;
    CK(cudaMemcpyAsync(ctx->frame_params_dev.ptr, ctx->frame_params_host, sizeof(FrameParams), cudaMemcpyHostToDevice, ctx->stream));

    if (ctx->peer_mode && ctx->cfg.execution_mode != BEPUCUDA_EXEC_GRAPH && ctx->cfg.execution_mode != BEPUCUDA_EXEC_STREAM)
        return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "solve: peer sharding needs BEPUCUDA_EXEC_GRAPH or BEPUCUDA_EXEC_STREAM");
    if (ctx->exchange && !ctx->peer_mode) {
        if (ctx->cfg.execution_mode != BEPUCUDA_EXEC_STREAM) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "solve: sharded batches need BEPUCUDA_EXEC_STREAM");
        if (ctx->integ.angular_integration_mode != 0) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "solve: sharded batches support AngularIntegrationMode.Nonconserving only");
        ctx->exchange_failed = false;
    }
    CK(cudaEventRecord(ctx->ev_solve_begin, ctx->stream));
    int64_t launches = 0;
    if (ctx->cfg.execution_mode == BEPUCUDA_EXEC_GRAPH) {
        if (!ctx->graph_valid) {
            ctx->exchange_failed = false;
            CK(cudaStreamBeginCapture(ctx->stream, cudaStreamCaptureModeThreadLocal));
            int64_t n = 0;
            issue_stage_sequence(ctx, ctx->stream, &n);
            cudaError_t e = cudaStreamEndCapture(ctx->stream, &ctx->graph);
            if (e == cudaSuccess && ctx->exchange_failed) e = cudaErrorUnknown;
            if (e == cudaSuccess) e = cudaGraphInstantiate(&ctx->graph_exec, ctx->graph, 0);
            if (e != cudaSuccess) return cuda_fail(ctx, e, "graph capture");
            ctx->graph_valid = true;
            ctx->timings.kernel_launches = n;
        }
        if (ctx->graph_valid) {
            CK(cudaGraphLaunch(ctx->graph_exec, ctx->stream));
            launches = ctx->timings.kernel_launches;
        }
    }
    if (ctx->cfg.execution_mode == BEPUCUDA_EXEC_STREAM) {
        issue_stage_sequence(ctx, ctx->stream, &launches);
        CK(cudaGetLastError());
        if (ctx->exchange_failed) return fail(ctx, BEPUCUDA_ERR_CUDA, "solve: the exchange callback failed");
    }
    CK(cudaEventRecord(ctx->ev_solve_end, ctx->stream));
    if (ctx->peer_mode) { ctx->exchange_counter += ctx->exchanges_per_solve; ++ctx->shard_solve_index; }  // the flag barrier and the arrival counters keep counting across solves
    ctx->have_solve = true;
    ctx->timings.kernel_launches = launches;

    // metric bookkeeping (SURVEY.md §8d)
    int64_t ci = 0, bytes = 0;
    const int substeps = (int)ctx->iterations.size();
    for (const SourceTypeBatch& s : ctx->sources) {
        const TypeInfo* t = get_type_info(s.type_id);
        const int64_t n = s.live;
        for (int sub = 0; sub < substeps; ++sub) {
            ci += n * ctx->iterations[sub];
            bytes += n * ((int64_t)t->warm_start_bytes + (int64_t)ctx->iterations[sub] * t->solve_bytes + (sub > 0 ? t->incremental_bytes : 0));
        }
    }
    bytes += (int64_t)ctx->body_count * 108;
    ctx->timings.constraint_iterations = ci;
    ctx->timings.algorithmic_bytes = bytes;
    return BEPUCUDA_OK;
}

static int check_device_error_flag(bepucuda_ctx* ctx) {
    if (ctx->peer_mode && ctx->tune[3]) {
        unsigned long long acc[4] = {};
        cudaMemcpy(acc, (unsigned long long*)ctx->shard_flags.ptr + kMaxShardRanks, sizeof(acc), cudaMemcpyDeviceToHost);
        if (acc[3]) fprintf(stderr, "[bepucuda shard rank %d] exchange phases, mean over %llu: push+fence %.2f us, signal %.2f us, wait %.2f us\n", ctx->peers.rank, acc[3],
                            acc[0] / 1e3 / acc[3], acc[1] / 1e3 / acc[3], acc[2] / 1e3 / acc[3]);
    }
    if (ctx->peer_mode) {
        int32_t e = 0;
        CK(cudaMemcpyAsync(&e, ctx->error_dev.ptr, 4, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        if (e == 5) return fail(ctx, BEPUCUDA_ERR_CUDA, "sharded solve: a peer rank never reached an exchange point (flag barrier timed out); results are invalid");
    }
    return BEPUCUDA_OK;
}

int32_t bepucuda_synchronize(bepucuda_ctx* ctx) {
    if (!ctx) return BEPUCUDA_ERR_INVALID_ARGUMENT;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    return check_device_error_flag(ctx);
}

int32_t bepucuda_download_bodies(bepucuda_ctx* ctx, void* out, int32_t body_count) {
    if (!ctx || !out || body_count < 0 || body_count > ctx->body_count) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "download_bodies: bad arguments");
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventRecord(ctx->ev_down_begin, ctx->stream));
    launch_merge_bodies(ctx->raw_bodies.ptr, body_count, ctx->B, ctx->stream);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, ctx->raw_bodies.ptr, (size_t)body_count * 128, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaEventRecord(ctx->ev_down_end, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->have_down = true;
    ctx->timings.d2h_bytes = (int64_t)body_count * 128;
    return BEPUCUDA_OK;
}

int32_t bepucuda_download_impulses(bepucuda_ctx* ctx) {
    if (!ctx) return BEPUCUDA_ERR_INVALID_ARGUMENT;
    if (!ctx->constraints_ready) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "download_impulses before end_constraints");
    CK(cudaSetDevice(ctx->device));
    launch_transpose_out_all(ctx->tb_table.as<DeviceTypeBatch>(), ctx->tdesc_table.as<TransposeDesc>(), ctx->work_table.as<WorkItem>(), ctx->all_work_count, ctx->W,
                             kTransposeImpulses, ctx->stream);
    CK(cudaGetLastError());
    int64_t bytes = 0;
    std::vector<CopyChunk> d2h;
    for (auto& s : ctx->sources) {
        if (char* alias = map_host(ctx, s.host_impulses, s.impulse_bytes)) queue_chunks(d2h, alias, s.raw_impulses, s.impulse_bytes);
        else CK(cudaMemcpyAsync(s.host_impulses, s.raw_impulses, s.impulse_bytes, cudaMemcpyDeviceToHost, ctx->stream));
        bytes += (int64_t)s.impulse_bytes;
    }
    { int rc = flush_chunks(ctx, d2h); if (rc != BEPUCUDA_OK) return rc; }
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->timings.d2h_bytes += bytes;
    return BEPUCUDA_OK;
}

int32_t bepucuda_download_prestep(bepucuda_ctx* ctx, int32_t batch_index, int32_t type_batch_index, float* prestep_out) {
    if (!ctx || !prestep_out) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "download_prestep: bad arguments");
    if (!ctx->constraints_ready) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "download_prestep before end_constraints");
    CK(cudaSetDevice(ctx->device));
    for (auto& s : ctx->sources)
        if (s.batch_index == batch_index && s.type_batch_index == type_batch_index) {
            launch_transpose_out_all(ctx->tb_table.as<DeviceTypeBatch>(), ctx->tdesc_table.as<TransposeDesc>(), ctx->work_table.as<WorkItem>(), ctx->all_work_count, ctx->W,
                                     kTransposePrestep, ctx->stream);
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(prestep_out, s.raw_prestep, s.prestep_bytes, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            return BEPUCUDA_OK;
        }
    return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "download_prestep: unknown type batch");
}

int32_t bepucuda_get_timings(bepucuda_ctx* ctx, bepucuda_timings* out) {
    if (!ctx || !out) return BEPUCUDA_ERR_INVALID_ARGUMENT;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    { int rc = check_device_error_flag(ctx); if (rc != BEPUCUDA_OK) return rc; }
    if (ctx->have_solve) cudaEventElapsedTime(&ctx->timings.solve_ms, ctx->ev_solve_begin, ctx->ev_solve_end);
    if (ctx->have_up && !ctx->up_open) cudaEventElapsedTime(&ctx->timings.upload_ms, ctx->ev_up_begin, ctx->ev_up_end);
    if (ctx->have_down) cudaEventElapsedTime(&ctx->timings.download_ms, ctx->ev_down_begin, ctx->ev_down_end);
    *out = ctx->timings;
    return BEPUCUDA_OK;
}

int32_t bepucuda_event_record(bepucuda_ctx* ctx, int32_t slot) {
    if (!ctx || slot < 0 || slot >= 16) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "event_record: bad slot");
    CK(cudaSetDevice(ctx->device));
    if (!ctx->user_events[slot]) CK(cudaEventCreate(&ctx->user_events[slot]));
    CK(cudaEventRecord(ctx->user_events[slot], ctx->stream));
    return BEPUCUDA_OK;
}
int32_t bepucuda_event_elapsed_ms(bepucuda_ctx* ctx, int32_t a, int32_t b, float* ms) {
    if (!ctx || !ms || a < 0 || a >= 16 || b < 0 || b >= 16 || !ctx->user_events[a] || !ctx->user_events[b]) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "event_elapsed_ms: bad slots");
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventSynchronize(ctx->user_events[b]));
    CK(cudaEventElapsedTime(ms, ctx->user_events[a], ctx->user_events[b]));
    return BEPUCUDA_OK;
}

int32_t bepucuda_profile_stages(bepucuda_ctx* ctx, float dt, bepucuda_stage_profile* out) {
    if (ctx && ctx->exchange) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "profile_stages: not available with sharded batches");
    if (!ctx || !out || !(dt > 0)) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "profile_stages: bad arguments");
    if (!ctx->constraints_ready) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "profile_stages before end_constraints");
    CK(cudaSetDevice(ctx->device));
    std::memset(out, 0, sizeof(*out));
    { int rc = refresh_device_rows(ctx); if (rc != BEPUCUDA_OK) return rc; }
    CK(cudaStreamSynchronize(ctx->stream));
    compute_frame_params(ctx, dt, ctx->frame_params_host);
    CK(cudaMemcpyAsync(ctx->frame_params_dev.ptr, ctx->frame_params_host, sizeof(FrameParams), cudaMemcpyHostToDevice, ctx->stream));
    const size_t need = ctx->program.size() * 2;
    while (ctx->profile_events.size() < need) {
        cudaEvent_t ev;
        CK(cudaEventCreate(&ev));
        ctx->profile_events.push_back(ev);
    }
    const WorkRecord* records = ctx->record_table.as<WorkRecord>();
    const int32_t* ref_rows = ctx->ref_rows.as<int32_t>();
    const FrameParams* fp = ctx->frame_params_dev.as<FrameParams>();
    const int32_t* kin = ctx->kinematics_dev.as<int32_t>();
    std::vector<int> launched(ctx->program.size(), 0);
    for (size_t i = 0; i < ctx->program.size(); ++i) {
        const StageOp& op = ctx->program[i];
        const bool has_work = op.stage == kStageFinalPose ? ctx->B.count > 0 : op.work_count > 0;
        if (!has_work) continue;
        CK(cudaEventRecord(ctx->profile_events[2 * i], ctx->stream));
        if (op.stage <= kStageIncremental) ctx->launchers->constraint_stage(op.stage, records + op.work_begin, ref_rows + (size_t)op.work_begin * 64, op.work_count, ctx->B, fp, 0, ctx->stream);
        else if (op.stage <= kStageKinematic) ctx->launchers->kinematic_stage(op.stage, kin, op.work_count, ctx->B, fp, ctx->stream);
        else ctx->launchers->final_pose(ctx->B, fp, ctx->stream);
        CK(cudaEventRecord(ctx->profile_events[2 * i + 1], ctx->stream));
        launched[i] = 1;
    }
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaGetLastError());
    for (size_t i = 0; i < ctx->program.size(); ++i) {
        if (!launched[i]) continue;
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, ctx->profile_events[2 * i], ctx->profile_events[2 * i + 1]));
        const StageOp& op = ctx->program[i];
        out->ms[op.stage] += ms;
        out->launches[op.stage] += 1;
        int64_t bytes = 0;
        if (op.stage <= kStageIncremental) {
            // live constraints per work item are not tracked per bundle; use 32 lanes per bundle minus padding via the per-type-batch totals
            for (int w = 0; w < op.work_count; ++w) {
                const WorkItem& wi = ctx->work[op.work_begin + w];
                const TypeInfo* t = get_type_info(ctx->tbs[wi.type_batch].type_id);
                const int per = op.stage == kStageSolve ? t->solve_bytes : op.stage == kStageIncremental ? t->incremental_bytes : t->warm_start_bytes;
                bytes += (int64_t)per * ctx->bundle_live[(size_t)op.work_begin + w];
            }
        } else if (op.stage == kStageFinalPose) {
            bytes = (int64_t)ctx->body_count * 108;
        } else {
            bytes = (int64_t)op.work_count * 108;
        }
        out->algorithmic_bytes[op.stage] += bytes;
    }
    return BEPUCUDA_OK;
}

static_assert(sizeof(bepucuda_body_shape) == sizeof(BodyShape) && sizeof(bepucuda_body_activity) == sizeof(BodyActivityRecord), "ABI structs mirror the device records");

int32_t bepucuda_set_body_shapes(bepucuda_ctx* ctx, const bepucuda_body_shape* shapes, int32_t body_count) {
    if (!ctx || body_count < 0 || (body_count > 0 && !shapes)) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "set_body_shapes: bad arguments");
    CK(cudaSetDevice(ctx->device));
    CK(ctx->body_shapes.reserve((size_t)std::max(body_count, 1) * sizeof(BodyShape)));
    if (body_count > 0) CK(cudaMemcpyAsync(ctx->body_shapes.ptr, shapes, (size_t)body_count * sizeof(BodyShape), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));  // the caller's buffer is only guaranteed for the duration of the call
    ctx->shape_count = body_count;
    ctx->shape_bounds.active = false;
    return BEPUCUDA_OK;
}

int32_t bepucuda_predict_bounding_boxes(bepucuda_ctx* ctx, float dt, bepucuda_body_activity* activities, float* bounds_out) {
    if (!ctx || !(dt > 0) || !activities || !bounds_out) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "predict_bounding_boxes: bad arguments");
    auto& sb = ctx->shape_bounds;
    if (sb.active && sb.collidable_count != ctx->body_count)
        return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "predict_bounding_boxes: bepucuda_set_body_collidables was not called for the current body count");
    if (!sb.active && ctx->shape_count != ctx->body_count) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "predict_bounding_boxes: bepucuda_set_body_shapes was not called for the current body count");
    const int n = ctx->body_count;
    if (n == 0) return BEPUCUDA_OK;
    CK(cudaSetDevice(ctx->device));
    CK(ctx->body_activities.reserve((size_t)n * sizeof(BodyActivityRecord)));
    CK(ctx->body_bounds.reserve((size_t)n * 32));
    CK(cudaMemcpyAsync(ctx->body_activities.ptr, activities, (size_t)n * sizeof(BodyActivityRecord), cudaMemcpyHostToDevice, ctx->stream));
    // PoseIntegrator.PredictBoundingBoxes calls Callbacks.PrepareForIntegration(dt) with the frame dt (PoseIntegrator.cs:L428)
    auto clamp01 = [](float v) { return v < 0.f ? 0.f : (v > 1.f ? 1.f : v); };
    PredictParams p{};
    p.dt = dt;
    for (int i = 0; i < 3; ++i) p.gravity_dt[i] = ctx->integ.gravity[i] * dt;
    p.linear_damping_dt = powf(clamp01(1 - ctx->integ.linear_damping), dt);
    p.angular_damping_dt = powf(clamp01(1 - ctx->integ.angular_damping), dt);
    p.integrate_velocity_for_kinematics = ctx->integ.integrate_velocity_for_kinematics;
    if (sb.active)
        launch_predict_shape_bounds(ctx->B, sb.view, sb.work, ctx->body_activities.as<BodyActivityRecord>(), ctx->body_bounds.as<float4>(), p, ctx->stream);
    else
        launch_predict_bounding_boxes(ctx->B, ctx->body_shapes.as<BodyShape>(), ctx->body_activities.as<BodyActivityRecord>(), ctx->body_bounds.as<float4>(), p, ctx->stream);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(activities, ctx->body_activities.ptr, (size_t)n * sizeof(BodyActivityRecord), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(bounds_out, ctx->body_bounds.ptr, (size_t)n * 32, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return BEPUCUDA_OK;
}

static_assert(sizeof(bepucuda_hull) == sizeof(bepu_bounds_math::HullRecord) && sizeof(bepucuda_compound) == sizeof(bepu_bounds_math::CompoundRecord) &&
                  sizeof(bepucuda_compound_child) == 32 && sizeof(bepucuda_compound_child) == sizeof(bepu_bounds_math::CompoundChildRecord) &&
                  sizeof(bepucuda_mesh) == sizeof(bepu_bounds_math::MeshRecord) && sizeof(bepucuda_body_collidable) == sizeof(BodyCollidableRecord),
              "ABI structs mirror the device records");

namespace {
// Element count of a library shape type (0 for a type the library does not hold).
int64_t library_count(const bepucuda_shape_library& l, int32_t type) {
    switch (type) {
        case 0: return l.sphere_count;
        case 1: return l.capsule_count;
        case 2: return l.box_count;
        case 3: return l.triangle_count;
        case 4: return l.cylinder_count;
        case 5: return l.hull_count;
        case 6: return l.compound_count;
        case 7: return l.big_compound_count;
        case 8: return l.mesh_count;
        default: return 0;
    }
}
// An empty string when the library is consistent, else what is wrong with it.
std::string validate_library(const bepucuda_shape_library& l) {
    char msg[256];
    const struct { const void* ptr; int64_t count; const char* name; } arrays[] = {
        {l.spheres, l.sphere_count, "spheres"}, {l.capsules, l.capsule_count, "capsules"}, {l.boxes, l.box_count, "boxes"}, {l.triangles, l.triangle_count, "triangles"},
        {l.cylinders, l.cylinder_count, "cylinders"}, {l.hull_points, l.hull_bundle_total, "hull_points"}, {l.hulls, l.hull_count, "hulls"},
        {l.compound_children, l.compound_child_total, "compound_children"}, {l.compounds, l.compound_count, "compounds"}, {l.big_compounds, l.big_compound_count, "big_compounds"},
        {l.mesh_triangles, l.mesh_triangle_total, "mesh_triangles"}, {l.meshes, l.mesh_count, "meshes"}};
    for (const auto& a : arrays) {
        if (a.count < 0) return std::string(a.name) + ": negative count";
        if (a.count > 0 && !a.ptr) return std::string(a.name) + ": null pointer with a non-zero count";
    }
    for (int t = 0; t <= 8; ++t)
        if (library_count(l, t) > (1 << 24)) return "shape type " + std::to_string(t) + ": more entries than a TypedIndex can address (2^24)";
    if ((l.hull_count > 0 || l.hull_bundle_total > 0) && !(l.hull_bundle_width == 4 || l.hull_bundle_width == 8 || l.hull_bundle_width == 16))
        return "hull_bundle_width must be 4, 8 or 16 (Vector<float>.Count)";
    for (int64_t i = 0; i < l.hull_count; ++i) {
        const bepucuda_hull h = l.hulls[i];
        if (h.bundle_count < 1) return (snprintf(msg, sizeof msg, "hull %lld is empty", (long long)i), msg);
        if (h.first_bundle < 0 || (int64_t)h.first_bundle + h.bundle_count > l.hull_bundle_total)
            return (snprintf(msg, sizeof msg, "hull %lld: bundles [%d, %lld) outside hull_points (%lld bundles)", (long long)i, h.first_bundle, (long long)h.first_bundle + h.bundle_count, (long long)l.hull_bundle_total), msg);
    }
    for (int kind = 0; kind < 2; ++kind) {
        const bepucuda_compound* list = kind ? l.big_compounds : l.compounds;
        const int64_t count = kind ? l.big_compound_count : l.compound_count;
        const char* name = kind ? "big compound" : "compound";
        for (int64_t i = 0; i < count; ++i) {
            const bepucuda_compound c = list[i];
            if (c.child_count < 1) return (snprintf(msg, sizeof msg, "%s %lld is empty", name, (long long)i), msg);
            if (c.first_child < 0 || (int64_t)c.first_child + c.child_count > l.compound_child_total)
                return (snprintf(msg, sizeof msg, "%s %lld: children [%d, %lld) outside compound_children (%lld)", name, (long long)i, c.first_child, (long long)c.first_child + c.child_count, (long long)l.compound_child_total), msg);
        }
    }
    for (int64_t i = 0; i < l.compound_child_total; ++i) {
        const uint32_t shape = l.compound_children[i].shape;
        const int32_t type = (int32_t)((shape & 0x7F000000u) >> 24), index = (int32_t)(shape & 0x00FFFFFFu);
        if (!(shape & 0x80000000u) || type > 5)
            return (snprintf(msg, sizeof msg, "compound child %lld: shape 0x%08x is not an existing convex shape (types 0-5)", (long long)i, shape), msg);
        if (index >= library_count(l, type))
            return (snprintf(msg, sizeof msg, "compound child %lld: index %d out of range for shape type %d (%lld)", (long long)i, index, type, (long long)library_count(l, type)), msg);
    }
    for (int64_t i = 0; i < l.mesh_count; ++i) {
        const bepucuda_mesh m = l.meshes[i];
        if (m.triangle_count < 1) return (snprintf(msg, sizeof msg, "mesh %lld is empty", (long long)i), msg);
        if (m.first_triangle < 0 || m.first_triangle + m.triangle_count > l.mesh_triangle_total)
            return (snprintf(msg, sizeof msg, "mesh %lld: triangles [%lld, %lld) outside mesh_triangles (%lld)", (long long)i, (long long)m.first_triangle, (long long)(m.first_triangle + m.triangle_count), (long long)l.mesh_triangle_total), msg);
    }
    return "";
}
}  // namespace

int32_t bepucuda_set_shape_library(bepucuda_ctx* ctx, const bepucuda_shape_library* library) {
    if (!ctx || !library) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "set_shape_library: bad arguments");
    const bepucuda_shape_library& l = *library;
    const std::string problem = validate_library(l);
    if (!problem.empty()) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "set_shape_library: " + problem);
    CK(cudaSetDevice(ctx->device));
    auto& sb = ctx->shape_bounds;
    sb.library_set = false;
    sb.active = false;  // the work lists index the old library
    sb.collidable_count = -1;
    const int64_t w = l.hull_bundle_width;
    const struct { const void* ptr; size_t bytes; } arrays[12] = {
        {l.spheres, (size_t)l.sphere_count * 4}, {l.capsules, (size_t)l.capsule_count * 8}, {l.boxes, (size_t)l.box_count * 12}, {l.triangles, (size_t)l.triangle_count * 36},
        {l.cylinders, (size_t)l.cylinder_count * 8}, {l.hull_points, (size_t)l.hull_bundle_total * 12 * (size_t)w}, {l.hulls, (size_t)l.hull_count * sizeof(bepucuda_hull)},
        {l.compound_children, (size_t)l.compound_child_total * sizeof(bepucuda_compound_child)}, {l.compounds, (size_t)l.compound_count * sizeof(bepucuda_compound)},
        {l.big_compounds, (size_t)l.big_compound_count * sizeof(bepucuda_compound)}, {l.mesh_triangles, (size_t)l.mesh_triangle_total * 36},
        {l.meshes, (size_t)l.mesh_count * sizeof(bepucuda_mesh)}};
    for (int k = 0; k < 12; ++k) {
        CK(sb.library[k].reserve(std::max<size_t>(arrays[k].bytes, 16)));
        if (arrays[k].bytes) CK(cudaMemcpyAsync(sb.library[k].ptr, arrays[k].ptr, arrays[k].bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));  // the caller's buffers are only guaranteed for the duration of the call
    ShapeLibraryView& v = sb.view;
    v.spheres = sb.library[0].as<float>(), v.capsules = sb.library[1].as<float>(), v.boxes = sb.library[2].as<float>(), v.triangles = sb.library[3].as<float>();
    v.cylinders = sb.library[4].as<float>(), v.hull_points = sb.library[5].as<float>(), v.hulls = sb.library[6].as<bepu_bounds_math::HullRecord>();
    v.compound_children = sb.library[7].as<bepu_bounds_math::CompoundChildRecord>(), v.compounds = sb.library[8].as<bepu_bounds_math::CompoundRecord>();
    v.big_compounds = sb.library[9].as<bepu_bounds_math::CompoundRecord>(), v.mesh_triangles = sb.library[10].as<float>(), v.meshes = sb.library[11].as<bepu_bounds_math::MeshRecord>();
    v.hull_width = (int32_t)w;
    sb.counts = l;
    sb.counts.spheres = sb.counts.capsules = sb.counts.boxes = sb.counts.triangles = sb.counts.cylinders = sb.counts.hull_points = sb.counts.mesh_triangles = nullptr;
    sb.counts.hulls = nullptr, sb.counts.compound_children = nullptr, sb.counts.compounds = sb.counts.big_compounds = nullptr, sb.counts.meshes = nullptr;
    sb.meshes.assign(l.meshes, l.meshes + l.mesh_count);
    sb.library_set = true;
    return BEPUCUDA_OK;
}

int32_t bepucuda_set_body_collidables(bepucuda_ctx* ctx, const bepucuda_body_collidable* collidables, int32_t body_count) {
    if (!ctx || body_count < 0 || (body_count > 0 && !collidables)) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "set_body_collidables: bad arguments");
    auto& sb = ctx->shape_bounds;
    if (!sb.library_set) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "set_body_collidables: bepucuda_set_shape_library was not called");
    // per-class work lists; every built-in index is checked against the library
    std::vector<int32_t> hulls, compounds;
    std::vector<MeshBody> mesh_bodies;
    std::vector<MeshChunk> chunks;
    for (int32_t i = 0; i < body_count; ++i) {
        const uint32_t shape = collidables[i].shape;
        const int32_t type = (int32_t)((shape & 0x7F000000u) >> 24), index = (int32_t)(shape & 0x00FFFFFFu);
        if (!(shape & 0x80000000u) || type > 8) continue;  // no shape / user-registered type: valid = 0
        if (index >= library_count(sb.counts, type)) {
            char msg[160];
            snprintf(msg, sizeof msg, "set_body_collidables: body %d: index %d out of range for shape type %d (%lld in the library)", i, index, type, (long long)library_count(sb.counts, type));
            return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, msg);
        }
        if (type == 5) hulls.push_back(i);
        else if (type == 6 || type == 7) compounds.push_back(i);
        else if (type == 8) {
            const bepucuda_mesh& m = sb.meshes[index];
            MeshBody mb{i, index, (int32_t)chunks.size(), 0};
            for (int64_t t = 0; t < m.triangle_count; t += kMeshChunkTriangles, ++mb.chunk_count)
                chunks.push_back(MeshChunk{m.first_triangle + t, (int32_t)std::min<int64_t>(kMeshChunkTriangles, m.triangle_count - t), (int32_t)mesh_bodies.size()});
            mesh_bodies.push_back(mb);
        }
    }
    CK(cudaSetDevice(ctx->device));
    auto upload = [&](DeviceBuffer& buf, const void* src, size_t bytes) -> cudaError_t {
        cudaError_t e = buf.reserve(std::max<size_t>(bytes, 16));
        if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(buf.ptr, src, bytes, cudaMemcpyHostToDevice, ctx->stream);
        return e;
    };
    CK(upload(sb.collidables, collidables, (size_t)body_count * sizeof(bepucuda_body_collidable)));
    CK(upload(sb.hull_bodies, hulls.data(), hulls.size() * sizeof(int32_t)));
    CK(upload(sb.compound_bodies, compounds.data(), compounds.size() * sizeof(int32_t)));
    CK(upload(sb.mesh_bodies, mesh_bodies.data(), mesh_bodies.size() * sizeof(MeshBody)));
    CK(upload(sb.mesh_chunks, chunks.data(), chunks.size() * sizeof(MeshChunk)));
    CK(sb.mesh_partials.reserve(std::max<size_t>(chunks.size() * 6 * sizeof(float), 16)));
    CK(cudaStreamSynchronize(ctx->stream));
    ShapeBoundsWork& w = sb.work;
    w.collidables = sb.collidables.as<BodyCollidableRecord>();
    w.hull_bodies = sb.hull_bodies.as<int32_t>(), w.hull_body_count = (int32_t)hulls.size();
    w.compound_bodies = sb.compound_bodies.as<int32_t>(), w.compound_body_count = (int32_t)compounds.size();
    w.mesh_bodies = sb.mesh_bodies.as<MeshBody>(), w.mesh_body_count = (int32_t)mesh_bodies.size();
    w.mesh_chunks = sb.mesh_chunks.as<MeshChunk>(), w.mesh_chunk_count = (int32_t)chunks.size();
    w.mesh_partials = sb.mesh_partials.as<float>();
    sb.collidable_count = body_count;
    sb.active = true;
    return BEPUCUDA_OK;
}

uint32_t bepucuda_color_hash(uint32_t constraint_index) { return color_hash(constraint_index); }

int32_t bepucuda_color_constraints(bepucuda_ctx* ctx, int32_t constraint_count, int32_t bodies_per_constraint, const int32_t* encoded_body_references, int32_t body_count,
                                   int32_t fallback_batch_threshold, int32_t order, const uint32_t* priorities, int32_t* batch_indices_out, int32_t* batch_count_out,
                                   int32_t* rounds_out) {
    if (!ctx) return BEPUCUDA_ERR_INVALID_ARGUMENT;
    if (constraint_count < 0 || bodies_per_constraint < 1 || bodies_per_constraint > 4 || body_count < 0 || fallback_batch_threshold < 1 || fallback_batch_threshold > 64)
        return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "color_constraints: counts out of range (1..4 body slots, fallback threshold 1..64)");
    if (order < BEPUCUDA_COLOR_INSERTION_ORDER || order > BEPUCUDA_COLOR_BY_PRIORITY || (order == BEPUCUDA_COLOR_BY_PRIORITY && !priorities))
        return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "color_constraints: unknown order, or BEPUCUDA_COLOR_BY_PRIORITY without priorities");
    if (constraint_count > 0 && (!encoded_body_references || !batch_indices_out)) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "color_constraints: null buffer");
    if (batch_count_out) *batch_count_out = 0;
    if (rounds_out) *rounds_out = 0;
    if (constraint_count == 0) return BEPUCUDA_OK;
    CK(cudaSetDevice(ctx->device));
    // body references are validated on the host while they are being staged (one pass over memory the copy touches anyway)
    const size_t words = (size_t)constraint_count * bodies_per_constraint;
    for (size_t i = 0; i < words; ++i) {
        const int32_t enc = encoded_body_references[i];
        if (enc >= 0 && (int32_t)((uint32_t)enc & ((1u << 30) - 1u)) >= body_count) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "color_constraints: body reference out of range");
    }
    constexpr int kRoundsPerChunk = 32;  // even: the ping-pong lists return to their starting roles after every chunk
    const size_t nb = (size_t)std::max(body_count, 1), nc = (size_t)constraint_count;
    CK(ctx->color_refs.reserve(words * 4));
    CK(ctx->color_priorities.reserve(nc * 4));
    CK(ctx->color_body_min.reserve(nb * 8));
    CK(ctx->color_body_mask.reserve(nb * 8));
    CK(ctx->color_out.reserve(nc * 4));
    CK(ctx->color_lists.reserve(nc * 8));
    CK(ctx->color_counts.reserve((kRoundsPerChunk + 1) * 4));
    CK(cudaMemcpyAsync(ctx->color_refs.ptr, encoded_body_references, words * 4, cudaMemcpyHostToDevice, ctx->stream));
    if (order == BEPUCUDA_COLOR_BY_PRIORITY) CK(cudaMemcpyAsync(ctx->color_priorities.ptr, priorities, nc * 4, cudaMemcpyHostToDevice, ctx->stream));
    ColoringBuffers cb{};
    cb.refs = ctx->color_refs.as<int32_t>();
    cb.priorities = ctx->color_priorities.as<uint32_t>();
    cb.body_min = ctx->color_body_min.as<unsigned long long>();
    cb.body_mask = ctx->color_body_mask.as<unsigned long long>();
    cb.batch_out = ctx->color_out.as<int32_t>();
    cb.list[0] = ctx->color_lists.as<int32_t>();
    cb.list[1] = ctx->color_lists.as<int32_t>() + nc;
    cb.counts = ctx->color_counts.as<unsigned int>();
    cb.constraint_count = constraint_count;
    cb.bodies_per_constraint = bodies_per_constraint;
    cb.body_count = body_count;
    cb.fallback_threshold = fallback_batch_threshold;
    cb.order = order;
    CK(cudaMemsetAsync(ctx->color_counts.ptr, 0, (kRoundsPerChunk + 1) * 4, ctx->stream));
    launch_color_init(cb, ctx->stream);
    unsigned int counts[kRoundsPerChunk + 1];
    int64_t rounds = 0;
    for (;;) {
        for (int r = 0; r < kRoundsPerChunk; ++r) launch_color_round(cb, r, ctx->stream);
        CK(cudaMemcpyAsync(counts, ctx->color_counts.ptr, sizeof(counts), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        CK(cudaGetLastError());
        int used = kRoundsPerChunk;
        for (int r = 0; r < kRoundsPerChunk; ++r)
            if (counts[r + 1] == 0) { used = r + 1; break; }
        rounds += used;
        if (counts[used] == 0) break;
        // every round assigns at least the constraint with the globally lowest key, so the list shrinks: the loop ends after at most constraint_count rounds
        if (counts[kRoundsPerChunk] >= counts[0]) return fail(ctx, BEPUCUDA_ERR_CUDA, "color_constraints: no progress (internal error)");
        counts[0] = counts[kRoundsPerChunk];
        for (int r = 1; r <= kRoundsPerChunk; ++r) counts[r] = 0;
        CK(cudaMemcpyAsync(ctx->color_counts.ptr, counts, sizeof(counts), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));  // `counts` is a stack array: the copy must have read it before the next chunk's download overwrites it
    }
    CK(cudaMemcpyAsync(batch_indices_out, ctx->color_out.ptr, nc * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    int32_t highest = -1;
    for (size_t i = 0; i < nc; ++i) highest = std::max(highest, batch_indices_out[i]);
    if (batch_count_out) *batch_count_out = highest + 1;
    if (rounds_out) *rounds_out = (int32_t)std::min<int64_t>(rounds, 0x7fffffff);
    return BEPUCUDA_OK;
}

int32_t bepucuda_shard_export(bepucuda_ctx* ctx, bepucuda_ipc_handles* out) {
    if (!ctx || !out) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "shard_export: bad arguments");
    if (ctx->body_count <= 0) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "shard_export before upload_bodies");
    CK(cudaSetDevice(ctx->device));
    CK(ctx->shard_flags.reserve(kShardFlagBlockWords * sizeof(unsigned long long)));  // barrier flags, arrival counters and targets (ShardStage)
    CK(cudaMemset(ctx->shard_flags.ptr, 0, kShardFlagBlockWords * sizeof(unsigned long long)));
    void* ptrs[4] = {ctx->pose.ptr, ctx->velocity.ptr, ctx->inertia_world.ptr, ctx->shard_flags.ptr};
    for (int i = 0; i < 4; ++i) {
        cudaIpcMemHandle_t h;
        CK(cudaIpcGetMemHandle(&h, ptrs[i]));
        static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
        std::memcpy(out->bytes[i], &h, 64);
    }
    return BEPUCUDA_OK;
}

int32_t bepucuda_shard_import(bepucuda_ctx* ctx, int32_t rank, int32_t rank_count, const bepucuda_ipc_handles* all) {
    if (!ctx || !all || rank_count < 1 || rank_count > kMaxShardRanks || rank < 0 || rank >= rank_count) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "shard_import: bad arguments");
    if (!ctx->shard_flags.ptr) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "shard_import before shard_export");
    CK(cudaSetDevice(ctx->device));
    ShardPeers p{};
    p.rank = rank;
    p.rank_count = rank_count;
    for (int r = 0; r < rank_count; ++r) {
        void* ptrs[4] = {ctx->pose.ptr, ctx->velocity.ptr, ctx->inertia_world.ptr, ctx->shard_flags.ptr};
        if (r != rank)
            for (int i = 0; i < 4; ++i) {
                cudaIpcMemHandle_t h;
                std::memcpy(&h, all[r].bytes[i], 64);
                CK(cudaIpcOpenMemHandle(&ptrs[i], h, cudaIpcMemLazyEnablePeerAccess));
                ctx->opened_ipc.push_back(ptrs[i]);
            }
        p.pose[r] = (float4*)ptrs[0];
        p.velocity[r] = (float4*)ptrs[1];
        p.inertia_world[r] = (float4*)ptrs[2];
        p.flags[r] = (unsigned long long*)ptrs[3];
    }
    ctx->peers = p;
    ctx->peer_mode = true;
    ctx->exchange_counter = 0;
    if (ctx->constraints_ready) ctx->constraints_ready = false;
    invalidate_graph(ctx);
    return BEPUCUDA_OK;
}

int32_t bepucuda_shard_import_contexts(bepucuda_ctx* ctx, int32_t rank, int32_t rank_count, bepucuda_ctx* const* all) {
    if (!ctx || !all || rank_count < 1 || rank_count > kMaxShardRanks || rank < 0 || rank >= rank_count || all[rank] != ctx)
        return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "shard_import_contexts: bad arguments");
    CK(cudaSetDevice(ctx->device));
    ShardPeers p{};
    p.rank = rank;
    p.rank_count = rank_count;
    for (int r = 0; r < rank_count; ++r) {
        bepucuda_ctx* o = all[r];
        if (!o || !o->shard_flags.ptr || o->body_count != ctx->body_count) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "shard_import_contexts: every context needs the same bodies and a shard_export");
        if (o->device != ctx->device) {
            int can = 0;
            CK(cudaDeviceCanAccessPeer(&can, ctx->device, o->device));
            if (!can) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "shard_import_contexts: no peer access between the devices");
            cudaError_t e = cudaDeviceEnablePeerAccess(o->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) CK(e);
            (void)cudaGetLastError();
        }
        p.pose[r] = o->pose.as<float4>();
        p.velocity[r] = o->velocity.as<float4>();
        p.inertia_world[r] = o->inertia_world.as<float4>();
        p.flags[r] = (unsigned long long*)o->shard_flags.ptr;
    }
    ctx->peers = p;
    ctx->peer_mode = true;
    ctx->exchange_counter = 0;
    if (ctx->constraints_ready) ctx->constraints_ready = false;
    invalidate_graph(ctx);
    return BEPUCUDA_OK;
}

int32_t bepucuda_shard_set_global(bepucuda_ctx* ctx, const int32_t* first_batch, const uint8_t* constrained) {
    if (!ctx || !first_batch || !constrained) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "shard_set_global: bad arguments");
    ctx->global_first_batch.assign(first_batch, first_batch + ctx->body_count);
    ctx->global_constrained.assign(constrained, constrained + ctx->body_count);
    if (ctx->constraints_ready) ctx->constraints_ready = false;
    return BEPUCUDA_OK;
}

int32_t bepucuda_shard_set_body_masks(bepucuda_ctx* ctx, const uint8_t* rank_masks) {
    if (!ctx) return BEPUCUDA_ERR_INVALID_ARGUMENT;
    if (rank_masks) ctx->body_masks.assign(rank_masks, rank_masks + ctx->body_count);
    else ctx->body_masks.clear();
    if (ctx->constraints_ready) ctx->constraints_ready = false;
    return BEPUCUDA_OK;
}

int32_t bepucuda_shard_set_pushes(bepucuda_ctx* ctx, int32_t batch_index, int32_t count, const int32_t* bodies, const int32_t* ranks, const int32_t* owner_flags) {
    if (!ctx || batch_index < 0 || count < 0 || (count > 0 && (!bodies || !ranks || !owner_flags))) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "shard_set_pushes: bad arguments");
    std::vector<uint32_t>& list = ctx->pushes_by_batch[batch_index];
    list.resize((size_t)count);
    for (int i = 0; i < count; ++i) {
        if (bodies[i] < 0 || bodies[i] >= ctx->body_count || ranks[i] < 0 || ranks[i] >= kMaxShardRanks) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "shard_set_pushes: body or rank out of range");
        list[i] = (uint32_t)bodies[i] | ((uint32_t)ranks[i] << 28) | (owner_flags[i] ? kPushOwnerBit : 0u);
    }
    if (ctx->constraints_ready) ctx->constraints_ready = false;
    return BEPUCUDA_OK;
}

int32_t bepucuda_set_boundary_bodies(bepucuda_ctx* ctx, const int32_t* body_indices, int32_t count, bepucuda_exchange_fn exchange, void* user) {
    if (!ctx || count < 0) return fail(ctx, BEPUCUDA_ERR_INVALID_ARGUMENT, "set_boundary_bodies: bad arguments");
    (void)body_indices;  // every body is treated as possibly shared (see the header)
    if (ctx->constraints_open) return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "set_boundary_bodies inside begin/end_constraints");
    if (exchange && ctx->cfg.execution_mode != BEPUCUDA_EXEC_STREAM)
        return fail(ctx, BEPUCUDA_ERR_BAD_STATE, "set_boundary_bodies: sharded batches need a context created with BEPUCUDA_EXEC_STREAM");
    ctx->exchange = exchange;
    ctx->exchange_user = user;
    // ownership and the constrained mask depend on it: the constraint description has to be (re)built
    if (ctx->constraints_ready && !ctx->sources.empty()) ctx->constraints_ready = false;
    return BEPUCUDA_OK;
}

}  // extern "C"
