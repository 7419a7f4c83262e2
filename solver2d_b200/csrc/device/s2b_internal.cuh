// solver2d-b200 — device-side world: SoA columns, scratch arena, launch helpers. Internal to the CUDA library.
#pragma once

#include "s2b_device.h"
#include "solver2d/constants.h"
#include "solver2d/aabb.h"
#include "solver2d/math.h"

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <vector>

#define S2B_CHECK(call)                                                                                                \
	do                                                                                                                 \
	{                                                                                                                  \
		cudaError_t err__ = (call);                                                                                    \
		if (err__ != cudaSuccess)                                                                                      \
		{                                                                                                              \
			fprintf(stderr, "solver2d-b200: CUDA error %s at %s:%d (%s) — no CPU fallback, aborting\n",                 \
					cudaGetErrorString(err__), __FILE__, __LINE__, #call);                                             \
			abort();                                                                                                   \
		}                                                                                                              \
	} while (0)

// ---- body flags (bflags column) -------------------------------------------------------------------------------
#define S2B_BODY_VALID 0x1u
#define S2B_BODY_TYPE(f) (((f) >> 1) & 0x3u)
// a body takes part in conflict detection / write-back only if it can move in the solver
#define S2B_BODY_STATIC 0u
#define S2B_BODY_KINEMATIC 1u
#define S2B_BODY_DYNAMIC 2u

// ---- contact info word (cInfo.x) ------------------------------------------------------------------------------
// bits 0-1 pointCount, bit 2 frictionPersisted, bit 3 persisted0, bit 4 persisted1
#define S2B_CI_COUNT(x) ((x) & 0x3)
#define S2B_CI_FRICTION_PERSISTED 0x4
#define S2B_CI_PERSISTED0 0x8
#define S2B_CI_PERSISTED1 0x10

// A growable device array. grow() keeps the old contents (device-to-device copy on the world's stream).
// bumped whenever any device array is re-allocated: a captured CUDA graph bakes device pointers in, so the solver's graph
// cache keys on this epoch
inline unsigned long long& s2bAllocEpoch()
{
	static unsigned long long epoch = 0;
	return epoch;
}

// Scope guard for code whose (re)allocations no captured graph refers to (broad-phase scratch, transfer staging, the L2
// flush buffer): the epoch is put back on exit so that those allocations do not force a re-capture of the solver graph.
struct S2bEpochFreeze
{
	unsigned long long saved;
	S2bEpochFreeze() : saved(s2bAllocEpoch())
	{
	}
	~S2bEpochFreeze()
	{
		s2bAllocEpoch() = saved;
	}
};

template <typename T> struct DevArray
{
	T* p = nullptr;
	size_t cap = 0;

	void reserve(size_t n, cudaStream_t stream, bool keep = true, bool zero = true)
	{
		if (n <= cap)
		{
			return;
		}
		size_t newCap = cap ? cap : 64;
		while (newCap < n)
		{
			newCap += newCap / 2 + 64;
		}
		T* q = nullptr;
		S2B_CHECK(cudaMalloc((void**)&q, newCap * sizeof(T)));
		if (zero)
		{
			S2B_CHECK(cudaMemsetAsync(q, 0, newCap * sizeof(T), stream));
		}
		if (p != nullptr)
		{
			if (keep && cap > 0)
			{
				S2B_CHECK(cudaMemcpyAsync(q, p, cap * sizeof(T), cudaMemcpyDeviceToDevice, stream));
			}
			// stream-ordered release so in-flight kernels reading the old buffer stay valid
			S2B_CHECK(cudaFreeAsync(p, stream));
		}
		p = q;
		cap = newCap;
		s2bAllocEpoch() += 1;
	}

	void release()
	{
		if (p)
		{
			cudaFree(p);
		}
		p = nullptr;
		cap = 0;
	}
};

// per-contact persistent columns; two sets (ping-pong) so a broad-phase pass can re-sort into the other one
struct ContactColumns
{
	DevArray<unsigned long long> key; // lo shape << 32 | hi shape
	DevArray<int2> shapes;			  // (A, B) in manifold order
	DevArray<int2> bodies;			  // (A, B)
	DevArray<int4> info;			  // x: count/flags, y: id0 | id1 << 16, z: GJK cache (count | iA<<2.. ), w: cache metric bits
	DevArray<float4> nf;			  // normal.x normal.y friction 0
	DevArray<int> color;			  // colour the constraint was last solved with (-1: none)
	DevArray<float4> anchor[2];		  // localAnchorA.xy localAnchorB.xy   (body-origin relative, body frame)
	DevArray<float4> impulse[2];	  // separation normalImpulse tangentImpulse 0
	DevArray<float4> fanchor[2];	  // frictionAnchorA.xy frictionAnchorB.xy   (sticky only)
	DevArray<float4> fnormal[2];	  // frictionNormalA.xy frictionNormalB.xy   (sticky only)

	void reserve(size_t n, cudaStream_t s, bool sticky, bool keep)
	{
		key.reserve(n, s, keep);
		shapes.reserve(n, s, keep);
		bodies.reserve(n, s, keep);
		info.reserve(n, s, keep);
		nf.reserve(n, s, keep);
		color.reserve(n, s, keep);
		for (int p = 0; p < 2; ++p)
		{
			anchor[p].reserve(n, s, keep);
			impulse[p].reserve(n, s, keep);
			if (sticky)
			{
				fanchor[p].reserve(n, s, keep);
				fnormal[p].reserve(n, s, keep);
			}
		}
	}

	void release()
	{
		key.release();
		shapes.release();
		bodies.release();
		info.release();
		nf.release();
		color.release();
		for (int p = 0; p < 2; ++p)
		{
			anchor[p].release();
			impulse[p].release();
			fanchor[p].release();
			fnormal[p].release();
		}
	}
};

// raw-pointer view of the contact columns handed to kernels
struct ContactView
{
	unsigned long long* key;
	int2* shapes;
	int2* bodies;
	int4* info;
	float4* nf;
	int* color;
	float4* anchor[2];
	float4* impulse[2];
	float4* fanchor[2];
	float4* fnormal[2];
};

inline ContactView makeView(ContactColumns& c)
{
	ContactView v;
	v.key = c.key.p;
	v.shapes = c.shapes.p;
	v.bodies = c.bodies.p;
	v.info = c.info.p;
	v.nf = c.nf.p;
	v.color = c.color.p;
	for (int p = 0; p < 2; ++p)
	{
		v.anchor[p] = c.anchor[p].p;
		v.impulse[p] = c.impulse[p].p;
		v.fanchor[p] = c.fanchor[p].p;
		v.fnormal[p] = c.fnormal[p].p;
	}
	return v;
}

// per-step contact-constraint columns in solve order (group-major). Which optional columns are live depends on the
// solver variant (DESIGN.md "constraint stream").
struct ConstraintView
{
	int2* idx;		  // bodyA, bodyB | flags in the two top bits of y (see S2B_CF_*)
	float4* nf;		  // normal.x normal.y friction invI_A
	float4* anchor[2]; // COM-relative local anchors: A.xy B.xy
	float4* pm[2];	  // adjustedSeparation normalMass tangentMass invI_B(point 0) / spare(point 1)
	float2* lambda[2]; // normalImpulse tangentImpulse (read-modify-write every pass)
	float4* r0[2];	  // prepare-time world anchors rA0.xy rB0.xy (fixed-anchor variants, XPBD)
	float* sep[2];	  // prepare-time separation (PGS family, NGS)
	int* src;		  // contact slot this constraint came from
	// warm-start gather (warm_gather.cuh): what one body needs from one incident constraint, in two 16-byte rows instead of
	// six scattered columns. warmP[t] = {P0.x, P0.y, P1.x, P1.y}, P = lambda_n * n + lambda_t * t per point, rewritten by
	// whichever pass last changes the impulses before the next gather (P1.x = NaN: one-point manifold);
	// warmAnchor[t * 2 + side] = {anchor0.xy, anchor1.xy} of that side, written by prepare (COM-relative local anchors;
	// prepare-time world anchors for SoftStep). Null when the variant does not gather.
	float4* warmP;
	float4* warmAnchor;
	// per constraint: bit 0 / bit 1 = this constraint is the LAST one of the solve order that touches its body A / B. The
	// TGS_Soft bias sweep then integrates that body's position itself (s2IntegratePositions folded into the sweep, one
	// device-wide step less per sub-step; persistent.cuh). Null: positions are integrated by their own body pass.
	const int* lastTouch;
	// sticky extras
	float4* fanchor[2]; // COM-relative local friction anchors A.xy B.xy
	float2* tsep[2];	// tangentSeparation, spare
};

#define S2B_CF_TWO_POINTS 0x40000000
#define S2B_CF_STATIC_SOFT 0x80000000u
#define S2B_CF_INDEX_MASK 0x3FFFFFFF
// resident regions (persistent.cuh): body indices of a row are positions in the region's shared-memory copy; an index with
// this bit set is a body slot in global memory instead (a body no constraint can move: read only)
#define S2B_RES_GLOBAL 0x20000000

// view of the body columns
struct BodyView
{
	float4* vel;  // v.x v.y w invMass
	float4* pose; // dp.x dp.y q.s q.c
	float4* pos;  // p.x p.y invI I      (centre of mass)
	float4* org;  // origin.x origin.y localCenter.x localCenter.y
	float4* frc;  // force.x force.y torque mass
	float4* prm;  // linearDamping angularDamping gravityScale invI
	float4* aux0; // Jacobi: dv.x dv.y dw 0 ; XPBD: dp0.x dp0.y q0.s q0.c
	float4* aux1; // XPBD: v0.x v0.y w0 0
	uint8_t* flags;
	int capacity;
};

// view of the shape columns
struct ShapeView
{
	int4* head;		 // flags(valid|type<<1|moved<<4), body, proxyKey, vertex count
	int4* filter;	 // categoryBits maskBits groupIndex 0
	float4* aabb;	 // tight + speculative
	float4* fat;	 // broad-phase box
	float2* fr;		 // friction, radius
	float2* verts;	 // [shape * 8 + i]
	float2* normals; // [shape * 8 + i]
	int capacity;
};

// per-joint columns (slot order)
struct JointView
{
	int4* head;		// flags, bodyA, bodyB, 0
	float4* anchors; // localOriginAnchorA.xy localOriginAnchorB.xy
	float4* lim;	// referenceAngle lowerAngle upperAngle 0
	float4* motor;	// maxMotorTorque motorSpeed hertz dampingRatio
	float4* target; // mouse target.xy 0 0
	float4* imp;	// impulse.x impulse.y motorImpulse 0
	float4* limp;	// lowerImpulse upperImpulse 0 0
	int* color;		// colour the joint was last solved with (-1: none)
	int capacity;
};

// per-step joint-constraint columns in solve order
struct JointConstraintView
{
	int4* head;		// flags(type, limit, motor), bodyA, bodyB, source joint slot
	float4* anchor; // COM-relative local anchors A.xy B.xy
	float4* mass;	// invMassA invIA invMassB invIB
	float4* d0ax;	// centerDiff0.xy axialMass 0
	float4* lim;	// referenceAngle lowerAngle upperAngle 0
	float4* motor;	// maxMotorTorque motorSpeed 0 0
	float4* coef;	// biasCoefficient massCoefficient impulseCoefficient 0
	float4* pivot;	// pivotMass cx.x cx.y cy.x cy.y (mouse, non-fresh revolute)
	float4* imp;	// impulse.x impulse.y motorImpulse 0        (r/w)
	float4* limp;	// lowerImpulse upperImpulse 0 0              (r/w)
};

struct StageTimer
{
	cudaEvent_t ev[5];
	bool recorded = false;
};

struct s2bWorld
{
	int device = 0;
	int solverType = 0;
	cudaStream_t stream = nullptr;
	float2 gravity = {0.0f, -10.0f};
	int schedule = S2B_SCHEDULE_COLOR;
	int maxColors = 24;
	int persistent = 1;
	int useGraph = 1;		// replay the solver stage as a CUDA graph when nothing changed; s2b_set_graph / S2B_GRAPH=0 disable
	bool capturing = false;
	unsigned long long contactTableVersion = 0; // bumped whenever the contact table is replaced (pair pass commit, upload) // a stream capture of the solver stage is in progress
	// region-local schedule of the persistent kernel (persistent.cuh): 0 off, 1 when the cut set needs at most regionCutLimit
	// colours (decided on the device every time the schedule is built), 2 always; s2b_set_regions / S2B_REGIONS
	int useRegions = 1;
	int regionCutLimit = 3; // S2B_REGION_CUT_LIMIT
	int dataflow = 0;	// ticketed Gauss-Seidel passes in the persistent kernel (experimental, slower on B200: DESIGN.md §3.1);
						// s2b_set_dataflow / S2B_DATAFLOW=1 enable it
	int gatherWarm = 1; // per-body warm-start gather (warm_gather.cuh); s2b_set_warm_gather / S2B_WARM_GATHER=0 disable it
	int smCount = 148;
	int coopSupported = 0;
	int colorGrid = 0;	// cooperative grid sizes, computed once
	int solveGrid = 0;
	int solveGridSolver = -1; // variant the grid was sized for (each variant is its own kernel)
	DevArray<int> schedDirty; // [0] != 0: the set of live constraints changed since the solve schedule was built (device flag)
	DevArray<unsigned> solveBarrier; // arrival counter of the persistent kernel's grid barrier (persistent.cuh)
	unsigned long long scheduleEpoch = 0; // bumped by every host-side change the solve schedule depends on (uploads, settings)

	// bodies
	int bodyCap = 0;
	DevArray<float4> bVel, bPose, bPos, bOrg, bFrc, bPrm, bAux0, bAux1;
	DevArray<uint8_t> bFlags;

	// shapes
	int shapeCap = 0;
	DevArray<int4> sHead, sFilter;
	DevArray<float4> sAabb, sFat;
	DevArray<float2> sFr, sVerts, sNormals;

	// joints
	int jointCap = 0;
	DevArray<int4> jHead;
	DevArray<float4> jAnchors, jLim, jMotor, jTarget, jImp, jLimp;
	DevArray<int> jColor;
	DevArray<unsigned long long> jointPairKeys; // every jointed body pair: blocks new contacts
	int jointPairCount = 0;
	DevArray<unsigned long long> jointDestroyKeys; // pairs whose existing contacts are removed
	int jointDestroyCount = 0;

	// pinned read-back buffer of s2b_sync_body_state
	float* hostState = nullptr;
	// bulk paths (s2b_add_forces, s2b_download_transforms)
	void* bulkHost[2] = {nullptr, nullptr};
	size_t bulkBytes[2] = {0, 0};
	cudaEvent_t bulkEvent[2] = {nullptr, nullptr};
	int bulkNext = 0, bulkCurrent = 0;
	DevArray<char> dBulk;
	float* hostXf = nullptr;
	size_t hostXfFloats = 0;
	DevArray<float4> dXf;
	size_t hostStateFloats = 0;
	DevArray<float4> dState;

	// contacts
	ContactColumns contacts[2];
	int cur = 0;		  // which column set is live
	int contactCount = 0; // host mirror (valid after a pair pass or upload)
	bool sticky = false;

	// broad phase
	bool pairsDirty = true; // host-side structural change
	unsigned long long uploadEpoch = 0; // bumped by every row upload: a pair search started before it is stale
	int prefetchPairs = 1;	// start the pair search of the next step behind finalize (S2B_PREFETCH_PAIRS=0: off)
	int kempe = 1;		// empty a sparse top colour by Kempe chains after colouring (S2B_KEMPE=0 disables)
	int wholeIslandBodies = 1200; // regions: islands up to this size are never cut (S2B_WHOLE_ISLAND)
	int residentRegions = 1; // TGS_Soft: regions with nothing device-wide to solve keep their bodies in shared memory (S2B_RESIDENT=0 disables)
	int hubDegree = 48; // constraints of a body with more incident constraints go to the serial overflow group uncoloured (S2B_HUB_DEGREE, 0 = colour them)
	int fusePositions = 1; // TGS_Soft: s2IntegratePositions folded into the bias sweep (S2B_FUSE_POSITIONS=0 disables)
	int kempeGrid = 0;
	DevArray<int> dMovedFlag; // [0] = number of proxies moved in last finalize (device counter)
	int pairPassCount = 0;
	int treeHeight = 0;
	int largeLeafCount = 0;
	int pairRebuildCount = 0;

	// solve-order hint (validation)
	std::vector<unsigned long long> orderHint;

	// scratch + bookkeeping for the solver stage live in solver_state.cuh (opaque here)
	struct SolverScratch* scratch = nullptr;
	struct BroadScratch* broad = nullptr;

	// pinned host mailbox for small device->host counters
	int* hostMail = nullptr; // pinned, 64 ints
	int* devMail = nullptr;	 // device, 64 ints

	int kernelLaunches = 0;
	// device-side work meter: [0] constraint-iterations, [1] solver stages run (bench metric, SURVEY §8d)
	DevArray<unsigned long long> dWork;
	// device time of the last persistent solver kernel (roofline probe)
	cudaEvent_t solveKernelStart = nullptr, solveKernelEnd = nullptr;
	bool solveKernelTimed = false;
	cudaEvent_t markEvents[2] = {nullptr, nullptr};
	cudaEvent_t movedEvent = nullptr; // recorded behind the D2H copy of the moved-proxy counter at the end of every step
	// transforms are read back on a stream of their own when finalize was the last thing to write them: the read-back then
	// runs beside whatever the world's stream has queued behind finalize (the pair search of the next step) instead of after it
	cudaStream_t copyStream = nullptr;
	unsigned long long xfSeq = 0, finalizeSeq = ~0ull; // bumped by everything that writes body transforms / at the last finalize
	int sideCopies = 1;								   // S2B_SIDE_COPIES=0: read back on the world's stream
	StageTimer timer;
	float stageMs[4] = {0, 0, 0, 0};

	DevArray<char> l2Flush;
};

inline BodyView bodyView(s2bWorld* w)
{
	BodyView v;
	v.vel = w->bVel.p;
	v.pose = w->bPose.p;
	v.pos = w->bPos.p;
	v.org = w->bOrg.p;
	v.frc = w->bFrc.p;
	v.prm = w->bPrm.p;
	v.aux0 = w->bAux0.p;
	v.aux1 = w->bAux1.p;
	v.flags = w->bFlags.p;
	v.capacity = w->bodyCap;
	return v;
}

inline ShapeView shapeView(s2bWorld* w)
{
	ShapeView v;
	v.head = w->sHead.p;
	v.filter = w->sFilter.p;
	v.aabb = w->sAabb.p;
	v.fat = w->sFat.p;
	v.fr = w->sFr.p;
	v.verts = w->sVerts.p;
	v.normals = w->sNormals.p;
	v.capacity = w->shapeCap;
	return v;
}

inline JointView jointView(s2bWorld* w)
{
	JointView v;
	v.head = w->jHead.p;
	v.anchors = w->jAnchors.p;
	v.lim = w->jLim.p;
	v.motor = w->jMotor.p;
	v.target = w->jTarget.p;
	v.imp = w->jImp.p;
	v.limp = w->jLimp.p;
	v.color = w->jColor.p;
	v.capacity = w->jointCap;
	return v;
}

// mailbox slots
enum
{
	MAIL_MOVED = 0,
	MAIL_CONSTRAINTS = 1,
	MAIL_GROUPS = 2,
	MAIL_OVERFLOW = 3,
	MAIL_NEW_PAIRS = 4,
	MAIL_KEPT = 5,
	MAIL_JOINTS = 6,
	MAIL_UNCOLORED = 7,
	MAIL_PAIR_OVERFLOW = 8,
	MAIL_REGIONS_ON = 9, // CNT_REGIONS_ON of the last schedule built outside a graph with regions on trial (a hint, read a step later)
	MAIL_COUNT = 64
};

inline int gridFor(int n, int block)
{
	return (n + block - 1) / block;
}

#define S2B_LAUNCH(world, kernel, grid, block, smem, ...)                                                              \
	do                                                                                                                 \
	{                                                                                                                  \
		kernel<<<(grid), (block), (smem), (world)->stream>>>(__VA_ARGS__);                                             \
		(world)->kernelLaunches += 1;                                                                                  \
	} while (0)

// stage entry points implemented in the other translation units
void s2bBroadphaseUpdatePairs(s2bWorld* w);
void s2bPrefetchPairSearch(s2bWorld* w);
float s2bLastPairSearchMs(s2bWorld* w);
void s2bNarrowphaseUpdate(s2bWorld* w);
void s2bSolve(s2bWorld* w, int solverType, const s2bStepContext* ctx);
void s2bFinalize(s2bWorld* w);
void s2bFreeSolverScratch(s2bWorld* w);
void s2bFreeBroadScratch(s2bWorld* w);
