// solver2d-b200 — the C ABI between the host C library and the CUDA (sm_100a) step pipeline.
//
// This is the inner drop-in boundary (SURVEY.md §8b): everything s2World_Step does to simulation state happens
// behind these entry points, on the GPU. They are plain `extern "C"` functions over an opaque handle, POD rows and
// raw pointers + sizes — no C++ or torch types — so the reference's own host C (or any FFI: cgo, JNI, ctypes) can
// bind them. Each entry point cites the reference interface it replaces.
//
// Memory model: the device owns the simulation state in SoA columns (DESIGN.md "data layout"). The host pushes
// changed objects as rows (`s2b_upload_*`), runs stages, and pulls rows back on demand (`s2b_download_*`).
// All calls on one world are ordered on that world's CUDA stream; downloads synchronise, uploads and stages do not.
// A missing/failed CUDA runtime is fatal (message + abort): there is no CPU fallback.
#pragma once

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C"
{
#endif

typedef struct s2bWorld s2bWorld;

#if defined(__GNUC__)
	#define S2B_API __attribute__((visibility("default")))
#else
	#define S2B_API
#endif

// ---- rows -----------------------------------------------------------------------------------------------------

// flags shared by all rows
#define S2B_ROW_VALID 0x1
// body rows only: the slot already holds this body on the device, so the row's force / torque are ADDED to what the device
// accumulated since the last step (bulk forces) instead of replacing it
#define S2B_BODY_ADD_FORCE 0x8

// One rigid body; mirrors the solver-relevant fields of s2Body (reference src/body.h:16-76).
typedef struct s2bBodyRow
{
	int32_t index;	 // body pool slot
	int32_t flags;	 // S2B_ROW_VALID | (s2BodyType << 1)
	float origin[2]; // body origin
	float position[2]; // centre of mass, world
	float rot[2];	   // (sin, cos)
	float linearVelocity[2];
	float angularVelocity;
	float localCenter[2];
	float mass, invMass;
	float I, invI;
	float force[2];
	float torque;
	float linearDamping, angularDamping, gravityScale;
} s2bBodyRow;

// shape kinds, numeric values of s2ShapeType (reference src/shape.h:14-21)
enum
{
	S2B_SHAPE_CAPSULE = 0,
	S2B_SHAPE_CIRCLE = 1,
	S2B_SHAPE_POLYGON = 2,
	S2B_SHAPE_SEGMENT = 3,
};

// One collision shape; mirrors s2Shape (reference src/shape.h:23-48). Geometry is always given in "polygon form":
// circle = 1 vertex + radius, capsule / segment = 2 vertices + the two side normals of s2MakeCapsule + radius,
// polygon = count vertices + normals + radius.
typedef struct s2bShapeRow
{
	int32_t index; // shape pool slot
	int32_t flags; // S2B_ROW_VALID | (type << 1) | S2B_SHAPE_MOVED | S2B_SHAPE_FRESH
	int32_t body;
	int32_t proxyKey; // reference broad-phase proxy key (decides which shape of a pair is "A", broad_phase.c:196-205)
	uint32_t categoryBits, maskBits;
	int32_t groupIndex;
	float friction;
	float aabb[4];	  // tight AABB + speculative margin
	float fatAABB[4]; // broad-phase AABB
	float radius;
	int32_t count;
	float vertices[16];
	float normals[16];
} s2bShapeRow;

#define S2B_SHAPE_MOVED 0x10
// set by the host on every (re)created shape: a contact that references such a slot belongs to a destroyed shape
#define S2B_SHAPE_FRESH 0x20

enum
{
	S2B_JOINT_REVOLUTE = 0,
	S2B_JOINT_MOUSE = 1,
};

#define S2B_JOINT_ENABLE_LIMIT 0x10
#define S2B_JOINT_ENABLE_MOTOR 0x20
#define S2B_JOINT_COLLIDE_CONNECTED 0x40

// One joint; mirrors s2Joint / s2RevoluteJoint / s2MouseJoint (reference src/joint.h:28-102).
typedef struct s2bJointRow
{
	int32_t index; // joint pool slot
	int32_t flags; // S2B_ROW_VALID | (type << 1) | S2B_JOINT_*
	int32_t bodyA, bodyB;
	float localOriginAnchorA[2], localOriginAnchorB[2];
	// revolute
	float referenceAngle, lowerAngle, upperAngle;
	float maxMotorTorque, motorSpeed;
	// mouse
	float hertz, dampingRatio;
	float target[2];
	// accumulated impulses (simulation state)
	float impulse[2];
	float motorImpulse, lowerImpulse, upperImpulse;
} s2bJointRow;

// One contact (shape pair) with its persistent manifold; mirrors s2Contact + s2Manifold + s2DistanceCache
// (reference src/contact.h:44-61, include/solver2d/manifold.h:19-46, distance.h:37-43).
typedef struct s2bContactPoint
{
	float localAnchorA[2], localAnchorB[2];
	float separation, normalImpulse, tangentImpulse;
	float frictionAnchorA[2], frictionAnchorB[2];
	float frictionNormalA[2], frictionNormalB[2];
	int32_t id;
	int32_t persisted;
} s2bContactPoint;

typedef struct s2bContactRow
{
	int32_t shapeA, shapeB;
	int32_t bodyA, bodyB;
	int32_t pointCount;
	int32_t frictionPersisted;
	float friction;
	float normal[2];
	s2bContactPoint points[2];
	int32_t cacheCount;
	uint8_t cacheIndexA[4], cacheIndexB[4];
	float cacheMetric;
} s2bContactRow;

// ---- step context ---------------------------------------------------------------------------------------------

// Mirrors s2StepContext (reference src/solvers.h:13-24) without the host body pointer.
typedef struct s2bStepContext
{
	float dt, inv_dt;
	float h, inv_h; // sub-step for the sub-stepping variants, else dt
	int32_t iterations;
	int32_t extraIterations;
	int32_t warmStart;
} s2bStepContext;

// How constraints are grouped into conflict-free sets (DESIGN.md "schedules").
enum
{
	// Graph colouring on the device: few large groups, the production path. Gauss-Seidel order = colour-major.
	S2B_SCHEDULE_COLOR = 0,
	// Order-preserving wavefront levels: reproduces the sequential constraint order exactly (joints, then contacts,
	// each in slot order, or in the order given by s2b_set_contact_order). Validation path — thousands of groups.
	S2B_SCHEDULE_WAVEFRONT = 1,
};

typedef struct s2bCounters
{
	int32_t bodyCapacity, shapeCapacity, jointCapacity;
	int32_t contactCount;	 // shape pairs with overlapping fat AABBs
	int32_t constraintCount; // manifolds with >= 1 point in the last solve
	int32_t jointCount;		 // live joints in the last solve
	int32_t groupCount;		 // colours (or wavefront levels) in the last solve
	int32_t overflowCount;	 // constraints solved serially after the coloured groups
	int32_t treeHeight;		 // box levels a pair query descends through, leaves included (broad-phase hierarchy of the last pass)
	int32_t movedCount;		 // proxies whose fat AABB changed in the last finalize
	int32_t pairPassCount;	 // number of broad-phase passes run so far
	int32_t kernelLaunches;	 // CUDA kernels launched by this world since creation (graph replays count their kernels)
	int32_t graphReplays;	 // solver stages executed as a CUDA graph replay
	int32_t graphCaptures;	 // times the solver stage was (re)captured into a graph
	int64_t scratchBytes;	 // device bytes of per-step scratch currently reserved
	int32_t regionCount;	 // region-local schedule: regions (= blocks of the persistent kernel) of the last solve, 0 = off
	int32_t cutCount;		 // constraints that straddle two regions (solved in device-wide steps)
	int32_t cutGroupCount;	 // colours of the cut set = device-wide steps per Gauss-Seidel sweep
	int32_t recolouredCount; /* constraints moved out of a sparse top colour by Kempe chains so far (colouring, DESIGN.md 3.2) */
	int32_t largeLeafCount;	 // scene-sized proxies kept out of the broad-phase hierarchy (DESIGN.md 3.3)
	int32_t pairRebuildCount; // broad-phase passes that re-sorted the proxies so far
} s2bCounters;

// ---- lifecycle ------------------------------------------------------------------------------------------------

// Replaces the device-less pools/arena of s2CreateWorld (reference src/world.c:47-103). `cudaDevice` < 0 selects the
// current device. `solverType` is the s2SolverType the world will be stepped with (selects optional columns).
S2B_API s2bWorld* s2b_world_create(int cudaDevice, int solverType);
S2B_API void s2b_world_destroy(s2bWorld* world);

S2B_API void s2b_set_gravity(s2bWorld* world, float gx, float gy);
S2B_API void s2b_set_schedule(s2bWorld* world, int schedule);
// Colour-schedule tuning: maximum number of colours (<= 64) before a constraint spills to the serial overflow set.
S2B_API void s2b_set_max_colors(s2bWorld* world, int maxColors);
// Use the single persistent cooperative kernel for the solver stage (1, default where supported) or one launch
// per group and pass (0; used for per-kernel profiling and as a cross-check).
S2B_API void s2b_set_persistent(s2bWorld* world, int enable);
// Warm start of the sub-stepping variants as a per-body gather fused with s2IntegrateVelocities (1, default) or as
// grouped constraint passes like every other pass (0; cross-check). Both give bit-identical results.
S2B_API void s2b_set_warm_gather(s2bWorld* world, int enable);
// Replay the solver stage (set-up kernels + persistent kernel, ~30 launches) as ONE CUDA graph launch while its inputs'
// shapes and addresses are unchanged (1, default) or always launch kernel by kernel (0).
S2B_API void s2b_set_graph(s2bWorld* world, int enable);
// Region-local schedule of the persistent kernel: bodies are partitioned into one region per thread block, constraints
// interior to a region run between block barriers, only the cut set needs grid barriers (DESIGN.md §3.1).
// mode 0 = never: one device-wide step per colour; 1 (default) = when the cut set needs at most 3 colours (islands,
// batched worlds, chains, anything that fits one block), decided on the device whenever the schedule is built; 2 = always.
// Whatever order results is reported by s2b_download_solve_order and replayed bit for bit by the oracle.
S2B_API void s2b_set_regions(s2bWorld* world, int mode);
// Gauss-Seidel passes of the persistent kernel synchronised by one grid barrier per colour (0, default) or by per-body
// tickets (1: a constraint waits only for the previous constraint on each of its bodies; no barrier inside a sweep).
// Same bits either way; the ticketed form measured SLOWER on B200 (75 k pollers saturate L2), kept as an experiment.
S2B_API void s2b_set_dataflow(s2bWorld* world, int enable);

// ---- host -> device -------------------------------------------------------------------------------------------

// Scatter rows into the SoA columns; capacities grow on demand (replaces pool growth, reference src/pool.c:108-159).
S2B_API void s2b_upload_bodies(s2bWorld* world, const s2bBodyRow* rows, int count, int bodyCapacity);
S2B_API void s2b_upload_shapes(s2bWorld* world, const s2bShapeRow* rows, int count, int shapeCapacity);
S2B_API void s2b_upload_joints(s2bWorld* world, const s2bJointRow* rows, int count, int jointCapacity);
// Replace the whole contact table (rows in solve order). Test / checkpoint-restore hook: on the normal path contacts
// are created and destroyed on the device by s2b_update_pairs.
S2B_API void s2b_upload_contacts(s2bWorld* world, const s2bContactRow* rows, int count);
// Sorted (bodyLo << 32 | bodyHi) keys of jointed body pairs, consulted by the pair pass:
//   blockKeys   — every live joint; no NEW contact is created between such bodies (replaces the joint-list walk of
//                 s2ShouldBodiesCollide, reference src/body.c:386-417, which ignores collideConnected);
//   destroyKeys — joints created with collideConnected == false; EXISTING contacts between such bodies are removed
//                 (replaces s2DestroyContactsBetweenBodies, reference src/joint.c:120-152, 214-217).
S2B_API void s2b_upload_joint_pairs(s2bWorld* world, const uint64_t* blockKeys, int blockCount, const uint64_t* destroyKeys,
									int destroyCount);
// Force / torque of the listed bodies (the per-frame input of s2Body_ApplyForceToCenter), ADDED to the device's
// accumulators; s2b_finalize zeroes them at the end of every step (reference src/world.c:275-276).
typedef struct s2bForceRow
{
	int32_t index;
	float force[2];
	float torque;
} s2bForceRow;
S2B_API void s2b_upload_forces(s2bWorld* world, const s2bForceRow* rows, int count);
// Bulk form of s2Body_ApplyForceToCenter (reference src/body.c:206-212): force[k] is ADDED to body bodyIndices[k]. The
// host arrays are copied into page-locked staging before the call returns; the H2D copy and the add are asynchronous.
S2B_API void s2b_add_forces(s2bWorld* world, const int32_t* bodyIndices, const float* forcesXY, int count);
// Page-locked host memory for row staging (uploads from it are asynchronous DMA).
S2B_API void* s2b_host_alloc(size_t bytes);
S2B_API void s2b_host_free(void* p);
// Force a broad-phase pass on the next s2b_update_pairs (creation/destruction of shapes or joints).
S2B_API void s2b_mark_pairs_dirty(s2bWorld* world);
// Validation hook: impose the sequential contact order for S2B_SCHEDULE_WAVEFRONT as a list of shape-pair keys
// (lo << 32 | hi), earliest first; contacts not listed follow in slot order. count == 0 clears it.
S2B_API void s2b_set_contact_order(s2bWorld* world, const uint64_t* pairKeys, int count);

// ---- the step, stage by stage (reference src/world.c:120-306) -------------------------------------------------

// Stages 1+2 and the destroy half of stage 3: s2UpdateBroadPhasePairs + s2BroadPhase_RebuildTrees (reference
// src/broad_phase.c:309-367, :381-385) and the fat-AABB overlap test of world.c:149-166. No-op when no proxy moved.
S2B_API void s2b_update_pairs(s2bWorld* world);
// Stage 3: s2UpdateContact for every contact (reference src/contact.c:296-359 -> manifold.c, distance.c).
S2B_API void s2b_update_contacts(s2bWorld* world);
// Solver dispatch: s2Solve_<variant>(world, context) (reference src/solvers.h:70-79, src/world.c:206-256).
S2B_API void s2b_solve(s2bWorld* world, int solverType, const s2bStepContext* context);
// Stage 4: transforms, force reset, AABB refit, proxy enlarge + move buffering (reference src/world.c:258-301).
S2B_API void s2b_finalize(s2bWorld* world);
// Start the pair search of the NEXT step (hierarchy refit, queries of the moved proxies, survivors of the contact table)
// behind this step's finalize, whose results are its inputs: the search's counters then reach the host together with the
// end of the step, and the next s2b_update_pairs merges the result without a host synchronisation in the middle of the pass.
// Optional (s2b_update_pairs does the whole pass itself when nothing was prefetched or rows were uploaded since); a no-op on
// scenes where nothing moved in the previous pass.
S2B_API void s2b_prefetch_pairs(s2bWorld* world);
// All four in order, then s2b_prefetch_pairs.
S2B_API void s2b_step(s2bWorld* world, int solverType, const s2bStepContext* context);

// ---- device -> host (synchronising) ---------------------------------------------------------------------------

S2B_API void s2b_sync(s2bWorld* world);
// The CUDA stream (cudaStream_t, returned as an opaque pointer) every operation of this world is enqueued on: lets a
// caller order its own work — e.g. an NCCL collective over s2b_pack_body_state's output — after the step without a host
// synchronisation.
S2B_API void* s2b_get_stream(s2bWorld* world);
// rows[i].index selects the slot to read for i < count (flags are filled in).
S2B_API void s2b_download_bodies(s2bWorld* world, s2bBodyRow* rows, int count);
// every slot 0..capacity-1 in order
S2B_API void s2b_download_all_bodies(s2bWorld* world, s2bBodyRow* rows, int capacity);
// The lazy read-back behind s2Body_GetPosition & co: 12 floats per body slot {origin.xy, position.xy, rot.sc, v.xy, w,
// force.xy, torque} gathered on the device and copied into a pinned buffer owned by the world. The pointer stays valid
// until the next call. Synchronises.
S2B_API const float* s2b_sync_body_state(s2bWorld* world, int capacity);
// Transforms only: {origin.x, origin.y, rot.s, rot.c} of body slots [0, count) into `out` (4 floats per slot, pageable or
// page-locked host memory). What a renderer reads every frame (reference src/world.c:369-412 reads them per shape).
S2B_API void s2b_download_transforms(s2bWorld* world, float* out, int count);
S2B_API void s2b_download_shape_boxes(s2bWorld* world, float* aabb4, float* fat4, int32_t* flags, int capacity);
S2B_API void s2b_download_joints(s2bWorld* world, s2bJointRow* rows, int capacity);
// returns the number of contacts written (<= maxCount), in device order (sorted by shape-pair key)
S2B_API int s2b_download_contacts(s2bWorld* world, s2bContactRow* rows, int maxCount);
// The Gauss-Seidel visiting order of the last s2b_solve, group by group: items[k] >= 0 is a contact slot, items[k] < 0
// is joint slot (-1 - items[k]); groupSizes[g] items belong to group g (the serial overflow group, if any, is last).
// Returns the item count. (Feeds the order-permuted oracle in the parity tests.)
S2B_API int s2b_download_solve_order(s2bWorld* world, int32_t* items, int maxItems, int32_t* groupSizes, int maxGroups,
							 int32_t* groupCount);
S2B_API void s2b_get_counters(s2bWorld* world, s2bCounters* out);
// Islands = connected components of the constraint graph of the last s2b_solve over the movable bodies (contacts with at
// least one point and joints connect; static and kinematic bodies do not — two piles on one ground are two islands). The
// reference reserves an island pool it never fills (reference src/world.h:31, src/contact.c:21-38). islandOfBody[i] = label
// of body slot i = the smallest body slot of its island, -1 for free slots; returns the number of islands (bodies without
// constraints count as islands of one). What shards a world across GPUs (island -> rank) and what the region-local solver
// schedule keeps whole inside one thread block. Synchronises.
S2B_API int s2b_download_islands(s2bWorld* world, int32_t* islandOfBody, int capacity);

// Packed per-body state {origin.x, origin.y, rot.s, rot.c, v.x, v.y, w, 0} for slots [first, first+count) written to
// a DEVICE buffer (32 B/body) — the payload of the per-step NCCL all-gather in the multi-world configuration.
S2B_API void s2b_pack_body_state(s2bWorld* world, int first, int count, void* deviceOut);

// ---- measurement ----------------------------------------------------------------------------------------------

// Run `steps` full steps back to back and return the elapsed device time in milliseconds measured with CUDA events
// on the world's stream (sync on both sides).
S2B_API float s2b_timed_steps(s2bWorld* world, int solverType, const s2bStepContext* context, int steps);
// Per-stage device time of the last s2b_step in milliseconds: {pairs, contacts, solve, finalize}.
S2B_API void s2b_last_stage_ms(s2bWorld* world, float out[4]);
// Evict L2: overwrite a scratch buffer larger than the 126 MB L2 (bench hygiene between timed iterations).
S2B_API void s2b_flush_l2(s2bWorld* world);
// Device-side work meter, accumulated by every s2b_solve: out[0] = constraint-iterations (SURVEY.md §8d: (contact
// constraints + joints) x solve passes of the variant), out[1] = solver stages run. Synchronises.
S2B_API void s2b_get_work(s2bWorld* world, uint64_t out[2], int reset);
// Device time of the last persistent solver kernel in milliseconds (CUDA events on the world's stream); 0 if the last
// solve used the multi-launch path.
S2B_API float s2b_last_solve_kernel_ms(s2bWorld* world);
// Stop-watch on the world's stream: s2b_mark_time(w, 0) ... s2b_mark_time(w, 1); s2b_elapsed_ms waits for mark 1.
S2B_API void s2b_mark_time(s2bWorld* world, int slot);
S2B_API float s2b_elapsed_ms(s2bWorld* world);
// Standalone timing of the per-colour contact impulse kernel on the current constraint set (roofline probe):
// launches the largest colour's solve kernel `reps` times, returns mean ms; *constraints receives its size.
S2B_API float s2b_time_color_kernel(s2bWorld* world, const s2bStepContext* context, int reps, int* constraints);

// Diagnostic: have the persistent solver kernel stamp %globaltimer after every grid barrier of the NEXT solves (capacity
// stamps per solve; 0 = off). s2b_get_solve_trace returns entries (code << 48 | nanoseconds), code = (pass kind << 8 | op).
S2B_API void s2b_set_solve_trace(s2bWorld* world, int capacity);
S2B_API int s2b_get_solve_trace(s2bWorld* world, uint64_t* out, int maxEntries);
S2B_API const char* s2b_version(void);
// Evaluate the device's atan2 (include/solver2d/atan2_f32.h) on the GPU for `count` host-resident (y, x) pairs: a
// probe for the parity tests, which compare it bit for bit with the host C library's atan2f.
S2B_API void s2b_eval_atan2(const float* y, const float* x, float* out, int32_t count);
// sizeof of {s2bBodyRow, s2bShapeRow, s2bJointRow, s2bContactRow, s2bStepContext, s2bCounters}: lets an FFI binding
// verify its struct mirrors at load time.
S2B_API void s2b_abi_sizes(int32_t out[6]);

#ifdef __cplusplus
}
#endif
