// solver2d-b200 — the solver stage of s2World_Step on the device.
//
// Replaces the per-variant entry points s2Solve_* (reference src/solvers.h:70-79, dispatched at world.c:206-256).
// Pipeline per step, all on the world's stream, no host synchronisation on the production path:
//
//   gather      live joints and manifolds with >= 1 point, compacted in slot order      (reference gather loop,
//               e.g. src/solve_tgs_soft.c:162-179: this *is* the sequential Gauss-Seidel order of the reference)
//   schedule    partition joints + contact constraints into groups with no shared movable body:
//                 COLOR      Jones-Plassmann colouring of the constraint graph on the device (<= 64 colours, the
//                            rest spills to a serial overflow group), solve order = colour-major;
//                 WAVEFRONT  order-preserving levels (validation path, bit-exact vs the sequential reference)
//   prepare     build the SoA constraint streams in solve order (coalesced 128-bit rows)
//   iterate     the variant's schedule of body passes and per-group constraint passes, either as ONE persistent
//               cooperative kernel (grid barrier between groups) or as one launch per group (profiling / cross-check)
//   store       accumulated impulses back to the persistent manifolds / joints
#include "persistent.cuh"

#include <cooperative_groups.h>
#include <cuda/barrier>
#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <algorithm>

namespace cg = cooperative_groups;

// ---------------------------------------------------------------------------------------------------------------
// scratch management
// ---------------------------------------------------------------------------------------------------------------

SolverScratch* s2bGetSolverScratch(s2bWorld* w)
{
	if (w->scratch == nullptr)
	{
		w->scratch = new SolverScratch();
	}
	return w->scratch;
}

void s2bFreeSolverScratch(s2bWorld* w)
{
	SolverScratch* s = w->scratch;
	if (s == nullptr)
	{
		return;
	}
	if (s->graphExec != nullptr)
	{
		cudaGraphExecDestroy(s->graphExec);
		s->graphExec = nullptr;
	}
	s->counts.release();
	s->activeFlag.release();
	s->activeSlots.release();
	s->jointFlag.release();
	s->jointSlots.release();
	s->itemBodies.release();
	s->degree.release();
	s->adjStart.release();
	s->adjCursor.release();
	s->adj.release();
	s->colorA.release();
	s->colorB.release();
	s->colorC.release();
	s->kempeState.release();
	s->kempeClaim.release();
	s->kempePath.release();
	s->itemRegion.release();
	s->sortKeyIn.release();
	s->sortKeyOut.release();
	s->bodyKeyIn.release();
	s->bodyKeyOut.release();
	s->bodyValIn.release();
	s->bodySorted.release();
	s->island.release();
	s->islandParent.release();
	s->islandSize.release();
	s->islandStart.release();
	s->regCount.release();
	s->regBodies.release();
	s->bodyRegion.release();
	s->bodyLocal.release();
	s->regBodyStart.release();
	s->cRegOff.release();
	s->jRegOff.release();
	s->sortValIn.release();
	s->sortValOut.release();
	s->cGroupOff.release();
	s->jGroupOff.release();
	s->cPerm.release();
	s->jPerm.release();
	s->cubTemp.release();
	s->itemVal.release();
	s->incWork.release();
	s->incList.release();
	s->lastTouch.release();
	s->heavyBodies.release();
	s->ovBodies.release();
	s->longBodies.release();
	s->ovBodySlot.release();
	s->flow.release();
	s->bodyTicket.release();
	s->trace.release();
	s->idx.release();
	s->nf.release();
	for (int p = 0; p < 2; ++p)
	{
		s->anchor[p].release();
		s->pm[p].release();
		s->r0[p].release();
		s->fanchor[p].release();
		s->lambda[p].release();
		s->tsep[p].release();
		s->sep[p].release();
	}
	s->src.release();
	s->warmP.release();
	s->warmAnchor.release();
	s->jhead.release();
	s->janchor.release();
	s->jmass.release();
	s->jd0ax.release();
	s->jlim.release();
	s->jmotor.release();
	s->jcoef.release();
	s->jpivot.release();
	s->jimp.release();
	s->jlimp.release();
	delete s;
	w->scratch = nullptr;
}

// which optional constraint columns a variant needs
struct VariantColumns
{
	bool r0;   // prepare-time world anchors
	bool sep;  // prepare-time separation
	bool sticky;
};

static VariantColumns columnsFor(int solverType)
{
	VariantColumns c = {false, false, false};
	switch (solverType)
	{
		case 0: // Jacobi
		case 1: // PGS
		case 2: // PGS_NGS
		case 4: // PGS_Soft
			c.r0 = true;
			c.sep = true;
			break;
		case 3: // PGS_NGS_Block: fixed anchors + the block columns (K, K^-1, velocity bias) in the sticky scratch columns
			c.r0 = true;
			c.sticky = true;
			break;
		case 5: // SoftStep
			c.r0 = true;
			break;
		case 6: // TGS_Sticky
			c.sticky = true;
			break;
		case 7: // TGS_Soft
			break;
		case 8: // TGS_NGS
			c.sep = true;
			break;
		case 9: // XPBD
			c.r0 = true;
			c.sep = true;
			break;
	}
	return c;
}

// ---------------------------------------------------------------------------------------------------------------
// gather
// ---------------------------------------------------------------------------------------------------------------

__global__ void s2bFlagActive(ContactView contacts, int contactCount, JointView joints, int jointCap, int* activeFlag,
							  int* jointFlag)
{
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < contactCount)
	{
		activeFlag[i] = S2B_CI_COUNT(contacts.info[i].x) > 0 ? 1 : 0;
	}
	if (i < jointCap)
	{
		jointFlag[i] = (joints.head[i].x & S2B_ROW_VALID) ? 1 : 0;
	}
}

// Conflict endpoints of every item (joints first, then contacts, both in natural order): a body index if the
// constraint can change that body's velocity/position, else -1 (SURVEY §7 H3: static and kinematic bodies are
// excluded from conflict detection and from write-back).
__global__ void s2bItemEndpoints(const int* counts, const int* jointSlots, const int* activeSlots, JointView joints,
								 ContactView contacts, BodyView bodies, int2* itemBodies, int* degree)
{
	int nJ = counts[CNT_JOINTS], nC = counts[CNT_CONTACTS];
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= nJ + nC)
	{
		return;
	}
	int a, b;
	if (i < nJ)
	{
		int4 head = joints.head[jointSlots[i]];
		a = head.y;
		b = head.z;
		if (((head.x >> 1) & 0x7) == S2B_JOINT_MOUSE)
		{
			a = -1; // the mouse joint only acts on body B
		}
	}
	else
	{
		int2 bo = contacts.bodies[activeSlots[i - nJ]];
		a = bo.x;
		b = bo.y;
	}
	// -1: cannot be moved by a constraint and does not move by itself either; -2: cannot be moved by a constraint but its
	// pose changes every sub-step (a kinematic body) — no conflict, but whoever reads it has to stay in step with the pass
	// that integrates it (s2bClassifyItemsKernel keeps such constraints out of the region-local phases)
	if (a >= 0)
	{
		bool movable = bodies.vel[a].w != 0.0f || bodies.prm[a].w != 0.0f;
		a = movable ? a : (S2B_BODY_TYPE(bodies.flags[a]) == S2B_BODY_STATIC ? -1 : -2);
	}
	if (b >= 0)
	{
		bool movable = bodies.vel[b].w != 0.0f || bodies.prm[b].w != 0.0f;
		b = movable ? b : (S2B_BODY_TYPE(bodies.flags[b]) == S2B_BODY_STATIC ? -1 : -2);
	}
	if (a == b && a >= 0)
	{
		b = -1;
	}
	itemBodies[i] = make_int2(a, b);
	if (degree != nullptr)
	{
		if (a >= 0)
		{
			atomicAdd(degree + a, 1);
		}
		if (b >= 0)
		{
			atomicAdd(degree + b, 1);
		}
	}
}

__global__ void s2bFillAdjacency(const int* counts, const int2* itemBodies, const int* adjStart, int* adjCursor, int* adj)
{
	int n = counts[CNT_JOINTS] + counts[CNT_CONTACTS];
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n)
	{
		return;
	}
	int2 e = itemBodies[i];
	if (e.x >= 0)
	{
		adj[adjStart[e.x] + atomicAdd(adjCursor + e.x, 1)] = i;
	}
	if (e.y >= 0)
	{
		adj[adjStart[e.y] + atomicAdd(adjCursor + e.y, 1)] = i;
	}
}

// ---------------------------------------------------------------------------------------------------------------
// Colouring of the constraint graph (items = nodes; two items conflict when they share a movable body).
//
// Colours are PERSISTENT: every contact slot and joint slot remembers the colour it was solved with, so on a settled
// scene nothing has to be coloured at all and only constraints that appeared this step (new pair, manifold that gained
// its first point, re-uploaded joint) are uncoloured when the kernel starts.
// Uncoloured items are coloured by speculative rounds (Gebremedhin-Manne): every uncoloured item tentatively takes the
// smallest colour no *committed* neighbour holds; among neighbours that took the same tentative colour in the same
// round only the one with the highest (hashed) priority commits, the others retry. Each round is two grid-wide phases;
// a handful of rounds colours a whole scene from scratch. The outcome depends only on the item set and the persisted
// colours, never on thread scheduling.
// Colour codes: -1 uncoloured, 0..maxColors-1, S2B_OVERFLOW_KEY = no colour below maxColors was free (serial group).
// ---------------------------------------------------------------------------------------------------------------

__device__ __forceinline__ unsigned s2bPriority(unsigned i)
{
	// integer hash (murmur3 finaliser); ties are broken by the index itself
	unsigned h = i * 0x9E3779B1u + 0x7F4A7C15u;
	h ^= h >> 16;
	h *= 0x85EBCA6Bu;
	h ^= h >> 13;
	h *= 0xC2B2AE35u;
	h ^= h >> 16;
	return h;
}

// Who wins when two neighbouring items pick the same tentative colour. During the first S2B_INDEX_PRIORITY_ROUNDS rounds
// the item with the SMALLER natural index wins: items are in shape-pair key order, which follows the geometry of scenes
// that were built in order (stacks, pyramids, grids), and greedy colouring in that order is near-optimal there — the
// 100 k-box pyramid gets 7 colours instead of the 10 a random order gives (6 is the lower bound: every box touches 6
// others). The price is more rounds (a row of the pyramid is a chain in index order: ~1.5 rounds per box of a row), paid
// once because colours persist. Chains longer than the limit (a 100 k-link rope) fall back to hashed priorities, whose
// round count is logarithmic.
#define S2B_INDEX_PRIORITY_ROUNDS 4096

__device__ __forceinline__ bool s2bHigherPriority(unsigned j, unsigned i, bool byIndex)
{
	if (byIndex)
	{
		return j < i;
	}
	unsigned pj = s2bPriority(j), pi = s2bPriority(i);
	return pj > pi || (pj == pi && j > i);
}

// seed the working colours from the persistent columns (joints first, then contact constraints)
__global__ void s2bSeedColors(const int* counts, const int* jointSlots, const int* activeSlots, const int* jointColor,
							  const int* contactColor, int* color, int maxColors)
{
	int nJ = counts[CNT_JOINTS], nC = counts[CNT_CONTACTS];
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= nJ + nC)
	{
		return;
	}
	int c = i < nJ ? jointColor[jointSlots[i]] : contactColor[activeSlots[i - nJ]];
	// overflow is re-evaluated every step; a colour beyond the current limit is dropped
	color[i] = (c >= 0 && c < maxColors) ? c : -1;
}

__global__ void s2bStoreColors(const int* counts, const int* jointSlots, const int* activeSlots, int* jointColor,
							   int* contactColor, const int* color)
{
	int nJ = counts[CNT_JOINTS], nC = counts[CNT_CONTACTS];
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= nJ + nC)
	{
		return;
	}
	if (i < nJ)
	{
		jointColor[jointSlots[i]] = color[i];
	}
	else
	{
		contactColor[activeSlots[i - nJ]] = color[i];
	}
}

// Cooperative kernel: speculative rounds until nothing is left uncoloured.
// `tent` holds (round << 8 | colour) so a value written in an earlier round can never be mistaken for this round's.
// validate != 0: persisted colours are first CHECKED against the current conflict graph — a body that became movable since
// its constraints were coloured (a shape with density added to a massless body) makes constraints that share it conflict;
// of two neighbours with the same colour the one with the larger index is uncoloured and picks again. Decided on the
// colours as they were (two phases), so the outcome does not depend on thread timing.
// abortAbove >= 0: give up as soon as any item would need a colour beyond it (the cut colouring: regions are only used when
// the cut set needs few colours, so a long run of rounds for a hub's hundreds of mutually conflicting constraints would be
// wasted) and leave CNT_CUT_ABORT set.
// hubDegree > 0: a constraint that touches a body with more incident constraints than that goes straight to the serial
// overflow group. All constraints of such a body conflict with one another, so each would need a colour of its own — a
// device-wide step (~2.8 us) for what the serial walk does in ~0.5 us — and the rest of the scene would be dragged through
// those steps as well (10 k-box tumbler: 24 colours with the drum's constraints coloured, 9 without).
__global__ void __launch_bounds__(256) s2bColorKernel(int* counts, const int2* itemBodies, const int* adjStart, const int* adj, int* color,
													  int* tent, int maxColors, int indexRounds, int validate, int abortAbove, const int* hubs,
													  int hubDegree)
{
	cg::grid_group grid = cg::this_grid();
	int n = counts[CNT_JOINTS] + counts[CNT_CONTACTS];
	int tid = blockIdx.x * blockDim.x + threadIdx.x;
	int stride = gridDim.x * blockDim.x;

	if (abortAbove >= 0 && hubs != nullptr && hubs[0] > 0)
	{
		// a hub body belongs to no region: its hundreds of constraints are all in the cut set and conflict with one another,
		// so the cut set needs at least that many colours — regions are off, and every thread of every one of those
		// constraints walking the hub's whole adjacency list round after round would cost milliseconds for nothing
		if (tid == 0)
		{
			counts[CNT_CUT_ABORT] = 1;
		}
		return;
	}

	if (validate)
	{
		for (int i = tid; i < n; i += stride)
		{
			int ci = color[i];
			int keep = 1;
			if (ci >= 0 && ci < S2B_MAX_COLORS)
			{
				int2 e = itemBodies[i];
#pragma unroll
				for (int side = 0; side < 2; ++side)
				{
					int body = side == 0 ? e.x : e.y;
					if (body < 0)
					{
						continue;
					}
					int begin = adjStart[body], end = adjStart[body + 1];
					if (hubDegree > 0 && end - begin > hubDegree)
					{
						keep = 0; // the body has become a hub since this constraint was coloured
						continue;
					}
					for (int k = begin; k < end; ++k)
					{
						int j = adj[k];
						if (j < i && color[j] == ci)
						{
							keep = 0;
						}
					}
				}
			}
			tent[i] = keep;
		}
		grid.sync();
		for (int i = tid; i < n; i += stride)
		{
			if (tent[i] == 0)
			{
				color[i] = -1;
			}
		}
		__threadfence();
		grid.sync();
	}

	// nothing to colour (the common case on a settled scene): leave without a single grid barrier.
	// Every thread evaluates the same predicate on data written by earlier kernels, so the exit is uniform.
	{
		__shared__ int blockUncoloured;
		if (threadIdx.x == 0)
		{
			blockUncoloured = 0;
		}
		__syncthreads();
		int mine = 0;
		for (int i = tid; i < n; i += stride)
		{
			mine |= (color[i] == -1) ? 1 : 0;
			tent[i] = 0; // stamps of earlier steps must not look like this step's
		}
		if (mine)
		{
			atomicOr(&blockUncoloured, 1);
		}
		__syncthreads();
		if (blockUncoloured)
		{
			atomicAdd(counts + CNT_UNCOLOURED, 1);
		}
	}
	grid.sync();
	if (*((volatile int*)(counts + CNT_UNCOLOURED)) == 0)
	{
		return;
	}

	for (int round = 1; round < 100000; ++round)
	{
		// phase A: tentative colours
		for (int i = tid; i < n; i += stride)
		{
			if (color[i] != -1)
			{
				continue;
			}
			int2 e = itemBodies[i];
			unsigned long long forbidden = 0ull;
#pragma unroll
			for (int side = 0; side < 2; ++side)
			{
				int body = side == 0 ? e.x : e.y;
				if (body < 0)
				{
					continue;
				}
				int begin = adjStart[body], end = adjStart[body + 1];
				if (hubDegree > 0 && end - begin > hubDegree)
				{
					forbidden = ~0ull; // serial overflow group
					continue;
				}
				for (int k = begin; k < end; ++k)
				{
					int cj = color[adj[k]];
					if (cj >= 0 && cj < S2B_MAX_COLORS)
					{
						forbidden |= 1ull << cj;
					}
				}
			}
			unsigned long long freeMask = ~forbidden;
			int pick = freeMask == 0ull ? S2B_MAX_COLORS : (__ffsll((long long)freeMask) - 1);
			if (pick >= maxColors)
			{
				pick = S2B_OVERFLOW_KEY;
			}
			if (abortAbove >= 0 && pick > abortAbove)
			{
				counts[CNT_CUT_ABORT] = 1;
			}
			tent[i] = (round << 8) | pick;
		}
		grid.sync();
		if (abortAbove >= 0 && *((volatile int*)(counts + CNT_CUT_ABORT)) != 0)
		{
			return; // uniform: read after the barrier by every thread
		}

		// phase B: commit unless a higher-priority neighbour took the same colour in this round
		int* counter = counts + CNT_REMAINING + (round % 3);
		int localRemaining = 0;
		for (int i = tid; i < n; i += stride)
		{
			if (color[i] != -1)
			{
				continue;
			}
			int mine = tent[i];
			int pick = mine & 0xFF;
			bool commit = true;
			if (pick != S2B_OVERFLOW_KEY)
			{
				int2 e = itemBodies[i];
#pragma unroll
				for (int side = 0; side < 2; ++side)
				{
					int body = side == 0 ? e.x : e.y;
					if (body < 0)
					{
						continue;
					}
					int begin = adjStart[body], end = adjStart[body + 1];
					for (int k = begin; k < end; ++k)
					{
						int j = adj[k];
						if (j != i && tent[j] == mine && s2bHigherPriority((unsigned)j, (unsigned)i, round <= indexRounds))
						{
							commit = false;
						}
					}
				}
			}
			if (commit)
			{
				color[i] = pick;
			}
			else
			{
				localRemaining += 1;
			}
		}
		if (localRemaining > 0)
		{
			atomicAdd(counter, localRemaining);
		}
		grid.sync();
		int remaining = *((volatile int*)counter);
		if (tid == 0)
		{
			counts[CNT_REMAINING + ((round + 2) % 3)] = 0;
			counts[CNT_ROUNDS] = round;
		}
		if (remaining == 0)
		{
			break;
		}
	}
}


// ---------------------------------------------------------------------------------------------------------------
// Emptying a sparse top colour (Kempe chains).
//
// Greedy colouring of a regular contact lattice ends with a handful of stragglers in one colour too many (36 of the 299 490
// constraints of the 100 k-box pyramid sit alone in a 7th colour; every box touches 6 others, so 6 is the optimum) — and
// every colour costs the solver one device-wide step per sweep, however few constraints it holds. A straggler e = (u, v)
// of the top colour has a colour `alpha` free at u and a colour `beta` free at v (its bodies have fewer neighbours than
// there are colours below), just never the same one. The constraints coloured alpha or beta form paths that alternate
// between the two; swapping the two colours along the path that starts at v frees alpha at v as well — unless that path
// ends at u — and e takes alpha (Vizing's argument for edge colourings; ours is one: constraints are the edges of the body
// graph). Static bodies end a path: they constrain nothing.
//
// One block per straggler walks its path (read-only, recorded); then every walker claims the bodies of its path
// (atomicMin of its rank, rank = order of the item indices, so the winners do not depend on timing); the walkers that own
// all their bodies swap. Paths of different winners share no body, hence no constraint, and what a walk read is still true
// when it is applied. Losers walk again next round. The walks are long dependent chains (up to S2B_KEMPE_MAX_HOPS hops of
// a few L2 round trips each — milliseconds), paid once: colours persist, and a top colour that could not be emptied is
// left alone for the next S2B_KEMPE_BACKOFF rebuilds.
// ---------------------------------------------------------------------------------------------------------------
#define S2B_KEMPE_MAX_ITEMS 512
#define S2B_KEMPE_MAX_HOPS 4096
#define S2B_KEMPE_ROUNDS 6
#define S2B_KEMPE_MAX_DEGREE 32
#define S2B_KEMPE_BACKOFF 32
#define S2B_KEMPE_QUIET_STEPS 8
#define S2B_REGION_RETRY 32

enum
{
	KS_BACKOFF = 0, // rebuilds to sit out (persists from launch to launch)
	KS_RUNS = 1,	// statistics: launches that walked, stragglers recoloured
	KS_FIXED = 2,
	KS_EVER = 3,	// a schedule has been built before
	KS_HIST = 8,	  // 64: items per colour
	KS_CURSOR = 72,	  // fill cursor of the straggler list
	KS_PROGRESS = 80, // 8: stragglers recoloured in round r
	KS_REMAINING = 88, // 8: stragglers still in the top colour after round r
	KS_LIST = 96,								// the stragglers (item indices)
	KS_LENGTH = KS_LIST + S2B_KEMPE_MAX_ITEMS,	// recorded path length, -1 no usable path, -2 no longer a straggler
	KS_ALPHA = KS_LENGTH + S2B_KEMPE_MAX_ITEMS,
	KS_BETA = KS_ALPHA + S2B_KEMPE_MAX_ITEMS,
	KS_SIZE = KS_BETA + S2B_KEMPE_MAX_ITEMS
};

// colours held by the items around `body` (every item but `skip`); *hub is raised when the body has too many to bother
__device__ __forceinline__ unsigned long long s2bColoursAround(const int* adjStart, const int* adj, const int* color, int body, int skip, bool* hub)
{
	int begin = adjStart[body], end = adjStart[body + 1];
	if (end - begin > S2B_KEMPE_MAX_DEGREE)
	{
		*hub = true;
		return ~0ull;
	}
	unsigned long long used = 0ull;
	for (int k = begin; k < end; ++k)
	{
		int j = adj[k];
		int c = color[j];
		if (j != skip && c >= 0 && c < S2B_MAX_COLORS)
		{
			used |= 1ull << c;
		}
	}
	return used;
}

// the alpha/beta path from v for straggler `item` = (u, v); records its constraints; returns the length or -1
__device__ __forceinline__ int s2bKempeWalk(const int2* itemBodies, const int* adjStart, const int* adj, const int* color, int item, int u, int v,
											 int alpha, int beta, int* path)
{
	int body = v, want = alpha, length = 0;
	for (;;)
	{
		int begin = adjStart[body], end = adjStart[body + 1];
		if (end - begin > S2B_KEMPE_MAX_DEGREE)
		{
			return -1;
		}
		int next = -1;
		for (int k = begin; k < end; ++k)
		{
			int j = adj[k];
			if (j != item && color[j] == want)
			{
				next = j;
			}
		}
		if (next < 0)
		{
			return length; // dead end: `want` is free here
		}
		if (length == S2B_KEMPE_MAX_HOPS)
		{
			return -1;
		}
		path[length++] = next;
		int2 e = itemBodies[next];
		int other = e.x == body ? e.y : e.x;
		if (other < 0)
		{
			return length; // a body that cannot move ends the path
		}
		if (other == u)
		{
			return -1; // the swap would take alpha away from u
		}
		body = other;
		want = want == alpha ? beta : alpha;
	}
}

// sched = the words of s2bScheduleGate. The pass runs on the first schedule ever built and on rebuilds that follow
// S2B_KEMPE_QUIET_STEPS steps without one: a scene whose constraints change every step (a pile still falling) would pay
// the walks again and again for colours that do not last.
__global__ void __launch_bounds__(256) s2bKempeKernel(const int* counts, const int2* itemBodies, const int* adjStart, const int* adj, int* color,
													  int* state, int* claim, int* paths, int bodyCapacity, int* sched)
{
	cg::grid_group grid = cg::this_grid();
	// only when the colouring kernel had something to colour, or a skipped pass is owed (a settled scene costs this launch
	// and nothing else)
	int owed = *((volatile int*)(sched + 2));
	if (counts[CNT_UNCOLOURED] == 0 && owed == 0)
	{
		return;
	}
	int tid = blockIdx.x * blockDim.x + threadIdx.x;
	int stride = gridDim.x * blockDim.x;
	int n = counts[CNT_JOINTS] + counts[CNT_CONTACTS];
	int backoff = *((volatile int*)(state + KS_BACKOFF));
	int ever = *((volatile int*)(state + KS_EVER));
	int quiet = *((volatile int*)(sched + 3));
	bool churning = ever != 0 && quiet < S2B_KEMPE_QUIET_STEPS;
	grid.sync(); // (everybody has read the words before thread 0 changes them)
	if (tid == 0)
	{
		state[KS_EVER] = 1;
		sched[2] = churning ? 1 : 0;
		sched[3] = 0;
	}
	if (churning)
	{
		return;
	}
	if (backoff > 0)
	{
		if (tid == 0)
		{
			state[KS_BACKOFF] = backoff - 1;
		}
		return;
	}

	__shared__ int hist[S2B_MAX_COLORS];
	for (int attempt = 0; attempt < 2; ++attempt)
	{
		for (int k = tid; k < KS_SIZE - KS_HIST; k += stride)
		{
			state[KS_HIST + k] = 0;
		}
		if (threadIdx.x < S2B_MAX_COLORS)
		{
			hist[threadIdx.x] = 0;
		}
		__syncthreads();
		grid.sync();
		for (int i = tid; i < n; i += stride)
		{
			int c = color[i];
			if (c >= 0 && c < S2B_MAX_COLORS)
			{
				atomicAdd(&hist[c], 1);
			}
		}
		__syncthreads();
		if (threadIdx.x < S2B_MAX_COLORS && hist[threadIdx.x] > 0)
		{
			atomicAdd(state + KS_HIST + threadIdx.x, hist[threadIdx.x]);
		}
		grid.sync();
		int top = -1;
		for (int c = S2B_MAX_COLORS - 1; c >= 0; --c)
		{
			if (*((volatile int*)(state + KS_HIST + c)) > 0)
			{
				top = c;
				break;
			}
		}
		int nTop = top >= 0 ? *((volatile int*)(state + KS_HIST + top)) : 0;
		// sparse = a small fraction of an average colour (and few enough to walk)
		if (top < 2 || nTop > S2B_KEMPE_MAX_ITEMS || (long long)nTop * 16 * (top + 1) > (long long)n)
		{
			return; // uniform. Nothing sparse on top: the colouring stands
		}
		for (int i = tid; i < n; i += stride)
		{
			if (color[i] == top)
			{
				state[KS_LIST + atomicAdd(state + KS_CURSOR, 1)] = i;
			}
		}
		if (tid == 0)
		{
			state[KS_RUNS] += 1;
		}
		__threadfence();
		grid.sync();

		bool emptied = false;
		for (int round = 0; round < S2B_KEMPE_ROUNDS; ++round)
		{
			for (int b = tid; b <= bodyCapacity; b += stride)
			{
				claim[b] = 0x7FFFFFFF;
			}
			// ---- walk (one thread of a block per straggler) ----
			if (threadIdx.x == 0)
			{
				for (int q = blockIdx.x; q < nTop; q += gridDim.x)
				{
					int item = state[KS_LIST + q];
					int* path = paths + (size_t)q * S2B_KEMPE_MAX_HOPS;
					int length = -1, alphaOut = -1, betaOut = -1;
					if (color[item] != top)
					{
						length = -2;
					}
					else
					{
						int2 e = itemBodies[item];
						bool hub = false;
						if (e.x >= 0 && e.y >= 0)
						{
							unsigned long long below = (1ull << top) - 1ull;
							unsigned long long freeU = ~s2bColoursAround(adjStart, adj, color, e.x, item, &hub) & below;
							unsigned long long freeV = ~s2bColoursAround(adjStart, adj, color, e.y, item, &hub) & below;
							if (hub == false && (freeU & freeV) != 0ull)
							{
								// (earlier swaps around it left a common colour)
								alphaOut = __ffsll((long long)(freeU & freeV)) - 1;
								betaOut = alphaOut;
								length = 0;
							}
							else if (hub == false)
							{
								for (unsigned long long fu = freeU; fu != 0ull && length < 0; fu &= fu - 1ull)
								{
									int alpha = __ffsll((long long)fu) - 1;
									for (unsigned long long fv = freeV; fv != 0ull && length < 0; fv &= fv - 1ull)
									{
										int beta = __ffsll((long long)fv) - 1;
										length = s2bKempeWalk(itemBodies, adjStart, adj, color, item, e.x, e.y, alpha, beta, path);
										alphaOut = alpha;
										betaOut = beta;
									}
								}
								// the same from the other end: a colour free at v, the path that starts at u
								for (unsigned long long fv = freeV; fv != 0ull && length < 0; fv &= fv - 1ull)
								{
									int alpha = __ffsll((long long)fv) - 1;
									for (unsigned long long fu = freeU; fu != 0ull && length < 0; fu &= fu - 1ull)
									{
										int beta = __ffsll((long long)fu) - 1;
										length = s2bKempeWalk(itemBodies, adjStart, adj, color, item, e.y, e.x, alpha, beta, path);
										alphaOut = alpha;
										betaOut = beta;
									}
								}
							}
						}
					}
					state[KS_LENGTH + q] = length;
					state[KS_ALPHA + q] = alphaOut;
					state[KS_BETA + q] = betaOut;
				}
			}
			__threadfence();
			grid.sync();
			// ---- claim ----
			if (threadIdx.x == 0)
			{
				for (int q = blockIdx.x; q < nTop; q += gridDim.x)
				{
					int length = state[KS_LENGTH + q];
					if (length < 0)
					{
						continue;
					}
					int item = state[KS_LIST + q];
					int rank = 0;
					for (int k = 0; k < nTop; ++k)
					{
						rank += state[KS_LIST + k] < item ? 1 : 0;
					}
					const int* path = paths + (size_t)q * S2B_KEMPE_MAX_HOPS;
					int2 e = itemBodies[item];
					atomicMin(claim + e.x, rank);
					atomicMin(claim + e.y, rank);
					for (int k = 0; k < length; ++k)
					{
						int2 pe = itemBodies[path[k]];
						if (pe.x >= 0)
						{
							atomicMin(claim + pe.x, rank);
						}
						if (pe.y >= 0)
						{
							atomicMin(claim + pe.y, rank);
						}
					}
				}
			}
			__threadfence();
			grid.sync();
			// ---- swap where every body of the path is ours ----
			if (threadIdx.x == 0)
			{
				for (int q = blockIdx.x; q < nTop; q += gridDim.x)
				{
					int length = state[KS_LENGTH + q];
					if (length == -2)
					{
						continue;
					}
					bool mine = length >= 0;
					int item = state[KS_LIST + q];
					const int* path = paths + (size_t)q * S2B_KEMPE_MAX_HOPS;
					if (mine)
					{
						int rank = 0;
						for (int k = 0; k < nTop; ++k)
						{
							rank += state[KS_LIST + k] < item ? 1 : 0;
						}
						int2 e = itemBodies[item];
						mine = claim[e.x] == rank && claim[e.y] == rank;
						for (int k = 0; k < length && mine; ++k)
						{
							int2 pe = itemBodies[path[k]];
							mine = (pe.x < 0 || claim[pe.x] == rank) && (pe.y < 0 || claim[pe.y] == rank);
						}
					}
					if (mine)
					{
						int alpha = state[KS_ALPHA + q], beta = state[KS_BETA + q];
						for (int k = 0; k < length; ++k)
						{
							int j = path[k];
							color[j] = color[j] == alpha ? beta : alpha;
						}
						color[item] = alpha;
						atomicAdd(state + KS_PROGRESS + round, 1);
						atomicAdd(state + KS_FIXED, 1);
					}
					else
					{
						atomicAdd(state + KS_REMAINING + round, 1);
					}
				}
			}
			__threadfence();
			grid.sync();
			int progress = *((volatile int*)(state + KS_PROGRESS + round));
			int remaining = *((volatile int*)(state + KS_REMAINING + round));
			if (remaining == 0)
			{
				emptied = true;
				break;
			}
			if (progress == 0)
			{
				break;
			}
		}
		if (emptied == false)
		{
			if (tid == 0)
			{
				state[KS_BACKOFF] = S2B_KEMPE_BACKOFF;
			}
			return;
		}
		grid.sync(); // (the state words are reset at the top of the next attempt)
	}
}

// ---------------------------------------------------------------------------------------------------------------
// Regions (persistent.cuh): the bodies are cut into `regions` spatially compact sets of equal size — consecutive runs
// of the Hilbert order of their centres of mass — one per block of the persistent kernel. Hub bodies (more incident
// constraints than S2B_HEAVY_DEGREE: a container wall, the ground under a whole pile is static and does not count)
// stay outside: every constraint that touches one is in the cut set and their body passes run grid-wide.
// ---------------------------------------------------------------------------------------------------------------

// order-preserving map float -> unsigned (larger float = larger key); NaN sorts high, harmless here
__device__ __forceinline__ unsigned s2bOrderedKey(float f)
{
	unsigned u = __float_as_uint(f);
	return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ float s2bFromOrderedKey(unsigned k)
{
	unsigned u = (k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k;
	return __uint_as_float(u);
}

// bounding box of the centres of all valid bodies (4 x atomicMax on keys: max x, max -x, max y, max -y)
__global__ void s2bBodyBoundsKernel(BodyView bodies, int* counts)
{
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	unsigned kx = 0, knx = 0, ky = 0, kny = 0;
	if (i < bodies.capacity && (bodies.flags[i] & S2B_BODY_VALID))
	{
		float4 pos = bodies.pos[i];
		kx = s2bOrderedKey(pos.x);
		knx = s2bOrderedKey(-pos.x);
		ky = s2bOrderedKey(pos.y);
		kny = s2bOrderedKey(-pos.y);
	}
	// warp-level maxima first: one atomic per warp and bound
	for (int d = 16; d > 0; d >>= 1)
	{
		kx = max(kx, __shfl_xor_sync(0xFFFFFFFFu, kx, d));
		knx = max(knx, __shfl_xor_sync(0xFFFFFFFFu, knx, d));
		ky = max(ky, __shfl_xor_sync(0xFFFFFFFFu, ky, d));
		kny = max(kny, __shfl_xor_sync(0xFFFFFFFFu, kny, d));
	}
	if ((threadIdx.x & 31) == 0 && (kx | knx | ky | kny) != 0)
	{
		unsigned* b = (unsigned*)(counts + CNT_BOUNDS);
		atomicMax(b + 0, kx);
		atomicMax(b + 1, knx);
		atomicMax(b + 2, ky);
		atomicMax(b + 3, kny);
	}
}

// position along the Hilbert curve of order 16 through the cell (x, y), x, y < 65536
__device__ __forceinline__ unsigned s2bHilbert16(unsigned x, unsigned y)
{
	unsigned d = 0;
	for (unsigned s = 32768u; s > 0; s >>= 1)
	{
		unsigned rx = (x & s) ? 1u : 0u, ry = (y & s) ? 1u : 0u;
		d += s * s * ((3u * rx) ^ ry);
		if (ry == 0)
		{
			if (rx == 1)
			{
				x = 65535u - x;
				y = 65535u - y;
			}
			unsigned t = x;
			x = y;
			y = t;
		}
	}
	return d;
}

// ---- islands: connected components of the constraint graph over the movable bodies (union-find) -------------------
// The reference reserves an island pool it never fills (reference src/world.h:31, design note src/contact.c:21-38); here
// the islands are what keeps the region schedule cheap: an island that fits a block stays whole in ONE region, so a world
// made of many small islands (batched worlds, bridges, rag dolls, debris) has no cut set at all and its Gauss-Seidel sweeps
// need no grid barrier. Lock-free union by index (hook the larger root under the smaller with atomicCAS, path halving on
// the way — the ECL-CC scheme): one pass over the items, one flatten pass; the label of an island is its smallest body slot,
// so the result does not depend on thread timing.

__device__ __forceinline__ int s2bIslandFind(int* parent, int x)
{
	volatile int* vp = parent;
	int p = vp[x];
	while (p != x)
	{
		int gp = vp[p];
		if (gp != p)
		{
			vp[x] = gp; // path halving: gp is an ancestor of x whatever other threads do meanwhile (parents only decrease)
		}
		x = p;
		p = gp;
	}
	return x;
}

__global__ void s2bIslandInitKernel(int bodyCapacity, int* parent)
{
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < bodyCapacity)
	{
		parent[i] = i;
	}
}

__global__ void s2bIslandHookKernel(const int* counts, const int2* itemBodies, int* parent)
{
	int n = counts[CNT_JOINTS] + counts[CNT_CONTACTS];
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n)
	{
		return;
	}
	int2 e = itemBodies[i]; // movable endpoints only: a static body (the ground) does not connect what rests on it
	if (e.x < 0 || e.y < 0)
	{
		return;
	}
	int a = e.x, b = e.y;
	for (;;)
	{
		a = s2bIslandFind(parent, a);
		b = s2bIslandFind(parent, b);
		if (a == b)
		{
			break;
		}
		int hi = max(a, b), lo = min(a, b);
		int old = atomicCAS(parent + hi, hi, lo);
		if (old == hi)
		{
			break;
		}
		a = old; // someone hooked `hi` meanwhile: continue from where it points now
		b = lo;
	}
}

// label of every body slot = smallest body slot of its island; island sizes counted at the label. The forest is final
// when this runs and is only READ here (a find that compresses paths would race with the label writes of other threads).
__global__ void s2bIslandFlattenKernel(BodyView bodies, const int* parent, int* label, int* islandSize)
{
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= bodies.capacity)
	{
		return;
	}
	int root = i;
	for (int p = parent[root]; p != root; p = parent[root])
	{
		root = p;
	}
	label[i] = root;
	if (bodies.flags[i] & S2B_BODY_VALID)
	{
		atomicAdd(islandSize + root, 1);
	}
}

__device__ __forceinline__ unsigned s2bHilbertOfBody(const BodyView& bodies, const int* counts, int i)
{
	const unsigned* b = (const unsigned*)(counts + CNT_BOUNDS);
	float maxX = s2bFromOrderedKey(b[0]), minX = -s2bFromOrderedKey(b[1]);
	float maxY = s2bFromOrderedKey(b[2]), minY = -s2bFromOrderedKey(b[3]);
	float extent = fmaxf(maxX - minX, maxY - minY);
	float scale = extent > 0.0f ? 65535.0f / extent : 0.0f;
	float4 pos = bodies.pos[i];
	float fx = (pos.x - minX) * scale, fy = (pos.y - minY) * scale;
	unsigned qx = fx >= 0.0f ? (fx < 65535.0f ? (unsigned)fx : 65535u) : 0u;
	unsigned qy = fy >= 0.0f ? (fy < 65535.0f ? (unsigned)fy : 65535u) : 0u;
	return s2bHilbert16(qx, qy);
}

// Sort key of every body slot: (Hilbert position of its ISLAND's label body) << 32 | its own Hilbert position — islands are
// contiguous in the sorted order and laid out along the curve inside — or all ones for slots that belong to no region
// (free slots, hub bodies). Hub bodies are appended to the hub list (order irrelevant: each is processed on its own).
__global__ void s2bBodyKeysKernel(BodyView bodies, int* counts, const int* degree, const int* island, unsigned long long* keys, int* vals,
								  int* hubs)
{
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= bodies.capacity)
	{
		return;
	}
	vals[i] = i;
	unsigned long long key = ~0ull;
	if (bodies.flags[i] & S2B_BODY_VALID)
	{
		if (degree[i] > S2B_HEAVY_DEGREE)
		{
			hubs[1 + atomicAdd(hubs, 1)] = i;
		}
		else
		{
			unsigned own = s2bHilbertOfBody(bodies, counts, i);
			unsigned isl = s2bHilbertOfBody(bodies, counts, island[i]);
			key = ((unsigned long long)isl << 32) | own;
			if (key == ~0ull)
			{
				key -= 1;
			}
			atomicAdd(counts + CNT_OWNED, 1);
		}
	}
	keys[i] = key;
}

// first rank of every island in the sorted order (at the island's label). Islands are runs of the sorted order (the island
// is the major sort key), so only the first rank of a run has to post its position: a handful of atomics per island instead
// of one per body — on a single 100 k-body island that was 100 k atomicMin on one address.
__global__ void s2bIslandStartKernel(const int* counts, const int* sortedBodies, const int* island, int* islandStart)
{
	int k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k < counts[CNT_OWNED])
	{
		int label = island[sortedBodies[k]];
		if (k == 0 || island[sortedBodies[k - 1]] != label)
		{
			atomicMin(islandStart + label, k);
		}
	}
}

// lanes of the warp that hold the same key as this one, and this lane's rank among them (warp-aggregated atomics)
__device__ __forceinline__ unsigned s2bPeers(int key, bool active, int* rank)
{
	unsigned peers = __match_any_sync(0xFFFFFFFFu, active ? key : -1 - (int)(threadIdx.x & 31));
	*rank = __popc(peers & ((1u << (threadIdx.x & 31)) - 1u));
	return peers;
}

// Region of every body. The owned bodies are cut into `regions` chunks of equal size along the sorted order; an island of
// at most two chunks goes WHOLE to the region its first body falls in (a block walks up to ~600 bodies per colour step at no
// extra cost and twice that in two waves, cheaper than any cut set); larger islands are split along the curve.
// wholeIsland: an island of at most that many bodies also stays whole when it is larger than two chunks — few small worlds
// on many blocks (32 piles of 1 035 boxes for 148 blocks): a block that owns one such island solves each of its colours in
// about one round of its threads, with no device-wide step at all, while cutting it would put a cut set back in.
__global__ void s2bAssignRegionsKernel(const int* counts, int bodyCapacity, int regions, const int* sortedBodies, const int* island,
									   const int* islandStart, const int* islandSize, int* bodyRegion, int* regCount, int wholeIsland)
{
	int k = blockIdx.x * blockDim.x + threadIdx.x;
	int owned = counts[CNT_OWNED];
	int chunk = max((owned + regions - 1) / regions, 1);
	int region = -1;
	bool inRange = k < bodyCapacity;
	int body = inRange ? sortedBodies[k] : 0;
	if (inRange && k < owned)
	{
		int label = island[body];
		int rank = islandSize[label] <= max(2 * chunk, wholeIsland) ? islandStart[label] : k;
		region = min(rank / chunk, regions - 1);
	}
	// neighbours in the sorted order mostly share a region: one atomic per (warp, region)
	int lane;
	unsigned peers = s2bPeers(region, region >= 0, &lane);
	if (region >= 0 && lane == 0)
	{
		atomicAdd(regCount + region, __popc(peers));
	}
	if (inRange)
	{
		bodyRegion[body] = region;
	}
}

// regBodyStart = exclusive scan of the region sizes (one block; regions <= 511); the cursors start at the same offsets
__global__ void __launch_bounds__(512) s2bRegionOffsetsKernel(int regions, const int* regCount, int* regBodyStart, int* regCursor, int* counts)
{
	__shared__ int s[512];
	int t = threadIdx.x;
	s[t] = t < regions ? regCount[t] : 0;
	__syncthreads();
	for (int d = 1; d < 512; d <<= 1)
	{
		int v = t >= d ? s[t - d] : 0;
		__syncthreads();
		s[t] += v;
		__syncthreads();
	}
	if (t < regions)
	{
		int begin = s[t] - regCount[t];
		regBodyStart[t] = begin;
		regCursor[t] = begin;
		atomicMax(counts + CNT_MAX_REGION, regCount[t]);
		if (t == regions - 1)
		{
			regBodyStart[regions] = s[t];
		}
	}
}

// body lists of the regions (order inside a region is irrelevant: body passes treat every body on its own)
__global__ void s2bFillRegionBodiesKernel(const int* counts, const int* sortedBodies, const int* bodyRegion, int* regCursor, int* regBodies,
										  const int* regBodyStart, int* bodyLocal)
{
	int k = blockIdx.x * blockDim.x + threadIdx.x;
	bool active = k < counts[CNT_OWNED];
	int body = active ? sortedBodies[k] : 0;
	int region = active ? bodyRegion[body] : -1;
	int lane;
	unsigned peers = s2bPeers(region, active, &lane);
	int base = 0;
	if (active && lane == 0)
	{
		base = atomicAdd(regCursor + region, __popc(peers));
	}
	base = __shfl_sync(0xFFFFFFFFu, base, __ffs(peers) - 1);
	if (active)
	{
		regBodies[base + lane] = body;
		bodyLocal[body] = base + lane - regBodyStart[region];
	}
}

// interior / cut classification of every item and the seed of the cut colouring.
// useRegions == 0: every item is in the "cut" set and keeps its primary colour there (one device-wide group per colour).
__global__ void s2bClassifyItemsKernel(int* counts, const int2* itemBodies, const int* bodyRegion, const int* color, int useRegions,
									   int* itemRegion, int* cutColor)
{
	int n = counts[CNT_JOINTS] + counts[CNT_CONTACTS];
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	int colorsHere = 0, primaryHere = 0, cutHere = 0;
	if (i < n)
	{
		int c = color[i];
		int region = -1;
		if (useRegions)
		{
			int2 e = itemBodies[i];
			if (e.x == -1 && e.y == -1)
			{
				region = 0; // touches no movable body: conflicts with nothing
			}
			else if (e.x < 0 && e.y < 0)
			{
				region = -1; // (a kinematic body among them: see below)
			}
			else
			{
				int ra = e.x >= 0 ? bodyRegion[e.x] : -2, rb = e.y >= 0 ? bodyRegion[e.y] : -2;
				if (e.x == -2 || e.y == -2)
				{
					// the other body is kinematic: its pose is integrated by the block that owns it, so this constraint runs
					// in the device-wide steps, which are ordered against every block's body passes
					region = -1;
				}
				else if (ra == -2)
				{
					region = rb;
				}
				else if (rb == -2 || rb == ra)
				{
					region = ra;
				}
			}
		}
		bool overflow = c < 0 || c >= S2B_MAX_COLORS;
		if (overflow)
		{
			region = -1;
		}
		itemRegion[i] = region;
		// 254 = takes no part in the cut colouring (interior, or already in the serial overflow group)
		cutColor[i] = region >= 0 ? 254 : (overflow ? S2B_OVERFLOW_KEY : (useRegions ? -1 : c));
		if (overflow == false)
		{
			colorsHere = c + 1;
			primaryHere = region >= 0 ? c + 1 : 0;
			cutHere = region < 0 ? 1 : 0;
		}
	}
	for (int d = 16; d > 0; d >>= 1)
	{
		colorsHere = max(colorsHere, __shfl_xor_sync(0xFFFFFFFFu, colorsHere, d));
		primaryHere = max(primaryHere, __shfl_xor_sync(0xFFFFFFFFu, primaryHere, d));
		cutHere += __shfl_xor_sync(0xFFFFFFFFu, cutHere, d);
	}
	if ((threadIdx.x & 31) == 0)
	{
		if (colorsHere > 0)
		{
			atomicMax(counts + CNT_COLORS, colorsHere);
		}
		if (primaryHere > 0)
		{
			atomicMax(counts + CNT_PRIMARY, primaryHere);
		}
		if (cutHere > 0)
		{
			atomicAdd(counts + CNT_CUT, cutHere);
		}
	}
}

// Solve-order keys, 16 bits, joints and contacts in separate arrays (values = natural index):
//   region * 64 + colour      interior constraints, region-major (region < 511)
//   0x8000 + cut colour       the cut set (or, without regions, every constraint by its colour)
//   0xFFFE                    serial overflow group
//   0xFFFF                    unused tail of the arrays (memset), sorts behind everything
#define S2B_KEY_CUT 0x8000
#define S2B_KEY_OVERFLOW 0xFFFE
#define S2B_KEY_DEAD 0xFFFF

// colours used by the cut set (largest cut colour + 1)
__global__ void s2bCutColorCountKernel(int* counts, const int* cutColor)
{
	int n = counts[CNT_JOINTS] + counts[CNT_CONTACTS];
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	int c = 0;
	if (i < n)
	{
		int cc = cutColor[i];
		c = (cc >= 0 && cc < S2B_MAX_COLORS) ? cc + 1 : 0;
	}
	for (int d = 16; d > 0; d >>= 1)
	{
		c = max(c, __shfl_xor_sync(0xFFFFFFFFu, c, d));
	}
	if ((threadIdx.x & 31) == 0 && c > 0)
	{
		atomicMax(counts + CNT_CUT_COLORS, c);
	}
}

// Regions pay when the cut set needs few colours: a sweep then costs (cut colours) device-wide steps + 7 block-local ones
// instead of one device-wide step per colour. Islands, batched worlds, bridges, anything that fits one block: 0-3 cut
// colours. A single dense pile cut along the jagged border of Hilbert chunks has boundary bodies with 3-6 cut constraints
// and needs 6 — as many as the pile has colours — so there the plain colour-major order is kept (measured, DESIGN.md §3.1).
// The decision is taken here, on the device, from the cut colouring; every later kernel reads CNT_REGIONS_ON.
__global__ void s2bMakeSortKeys(int* counts, const int* color, const int* itemRegion, const int* cutColor, int regionCutLimit,
								unsigned short* jKeys, int* jVals, unsigned short* cKeys, int* cVals)
{
	int nJ = counts[CNT_JOINTS], nC = counts[CNT_CONTACTS];
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	bool regionsOn = regionCutLimit >= 0 && counts[CNT_CUT_ABORT] == 0 && counts[CNT_CUT_COLORS] <= regionCutLimit;
	if (i == 0)
	{
		counts[CNT_REGIONS_ON] = regionsOn ? 1 : 0;
		if (regionsOn == false)
		{
			counts[CNT_PRIMARY] = 0;
		}
		if (counts[CNT_CUT_ABORT] != 0)
		{
			counts[CNT_CUT_COLORS] = S2B_MAX_COLORS; // "more than regions are worth" (the colouring was not finished)
		}
	}
	if (i >= nJ + nC)
	{
		return;
	}
	int region = regionsOn ? itemRegion[i] : -1;
	int key;
	if (regionsOn == false)
	{
		int c = color[i];
		key = (c >= 0 && c < S2B_MAX_COLORS) ? S2B_KEY_CUT + c : S2B_KEY_OVERFLOW;
	}
	else if (region >= 0)
	{
		key = region * S2B_MAX_COLORS + color[i];
	}
	else
	{
		int cc = cutColor[i];
		key = (cc >= 0 && cc < S2B_MAX_COLORS) ? S2B_KEY_CUT + cc : S2B_KEY_OVERFLOW;
	}
	if (i < nJ)
	{
		jKeys[i] = (unsigned short)key;
		jVals[i] = i;
	}
	else
	{
		cKeys[i - nJ] = (unsigned short)key;
		cVals[i - nJ] = i - nJ;
	}
}

__device__ __forceinline__ int s2bLowerBoundKey(const unsigned short* keys, int n, int key)
{
	int lo = 0, hi = n;
	while (lo < hi)
	{
		int mid = (lo + hi) >> 1;
		if ((int)keys[mid] < key)
		{
			lo = mid + 1;
		}
		else
		{
			hi = mid;
		}
	}
	return lo;
}

// Offset tables from the sorted keys (binary searches; entries beyond the live count hold S2B_KEY_DEAD):
//   regOff[r * 65 + c]  = first row of (region r, colour c), c = 64: end of region r
//   groupOff[g]         = first row of device-wide group g < 64; [64] = overflow group; [65] = live count
__global__ void s2bBuildTablesKernel(int regions, const unsigned short* jSorted, int jN, const unsigned short* cSorted, int cN, int* jRegOff,
									 int* cRegOff, int* jGroupOff, int* cGroupOff)
{
	int e = blockIdx.x * blockDim.x + threadIdx.x;
	int regEntries = regions * S2B_REG_STRIDE;
	if (e < regEntries)
	{
		int r = e / S2B_REG_STRIDE, c = e % S2B_REG_STRIDE;
		int key = r * S2B_MAX_COLORS + c; // c == 64: first key of the next region
		jRegOff[e] = s2bLowerBoundKey(jSorted, jN, key);
		cRegOff[e] = s2bLowerBoundKey(cSorted, cN, key);
		return;
	}
	int g = e - regEntries;
	if (g <= S2B_MAX_COLORS + 1)
	{
		int key = g < S2B_MAX_COLORS ? S2B_KEY_CUT + g : (g == S2B_MAX_COLORS ? S2B_KEY_OVERFLOW : S2B_KEY_DEAD);
		jGroupOff[g] = s2bLowerBoundKey(jSorted, jN, key);
		cGroupOff[g] = s2bLowerBoundKey(cSorted, cN, key);
	}
}

// + whether the regions can run out of shared memory (persistent.cuh, resident regions): regions on, nothing device-wide to
// solve (no cut set, no overflow group, no hub), no joints, every region small enough
__global__ void s2bFinishGroups(int* counts, const int* cOff, const int* jOff, const int* heavyBodies, int residentCapacity)
{
	// number of device-wide groups actually used (largest non-empty one + 1)
	int groups = 0;
	for (int c = 0; c < S2B_MAX_COLORS; ++c)
	{
		if (cOff[c + 1] > cOff[c] || jOff[c + 1] > jOff[c])
		{
			groups = c + 1;
		}
	}
	counts[CNT_GROUPS] = groups;
	counts[CNT_OVERFLOW_C] = cOff[S2B_MAX_COLORS + 1] - cOff[S2B_MAX_COLORS];
	counts[CNT_OVERFLOW_J] = jOff[S2B_MAX_COLORS + 1] - jOff[S2B_MAX_COLORS];
	bool resident = residentCapacity > 0 && counts[CNT_REGIONS_ON] != 0 && groups == 0 && counts[CNT_OVERFLOW_C] + counts[CNT_OVERFLOW_J] == 0 &&
					counts[CNT_JOINTS] == 0 && counts[CNT_CONTACTS] > 0 && counts[CNT_MAX_REGION] <= residentCapacity &&
					(heavyBodies == nullptr || heavyBodies[0] == 0);
	counts[CNT_RESIDENT] = resident ? 1 : 0;
}

// The distinct bodies the serial overflow group touches (movable or not), numbered in arrival order (the numbering is
// only a cache layout: persistent.cuh stages these bodies in shared memory for the serial walk).
__global__ void s2bOverflowBodiesKernel(const int* counts, const int* jGroupOff, const int* cGroupOff, const int* jPerm, const int* cPerm,
										const int* jointSlots, const int* activeSlots, JointView joints, ContactView contacts, int* ovBodySlot,
										int* ovBodies)
{
	int ovJ = counts[CNT_OVERFLOW_J], ovC = counts[CNT_OVERFLOW_C];
	int k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= ovJ + ovC)
	{
		return;
	}
	int a, b;
	if (k < ovJ)
	{
		int4 head = joints.head[jointSlots[jPerm[jGroupOff[S2B_MAX_COLORS] + k]]];
		a = head.y;
		b = head.z;
	}
	else
	{
		int2 bo = contacts.bodies[activeSlots[cPerm[cGroupOff[S2B_MAX_COLORS] + (k - ovJ)]]];
		a = bo.x;
		b = bo.y;
	}
#pragma unroll
	for (int side = 0; side < 2; ++side)
	{
		int body = side == 0 ? a : b;
		if (body >= 0 && atomicCAS(ovBodySlot + body, -1, -2) == -1)
		{
			int slot = atomicAdd(ovBodies, 1);
			ovBodies[1 + slot] = body;
			ovBodySlot[body] = slot;
		}
	}
}

// src[t] = contact slot of the constraint at solve position t
__global__ void s2bBuildSources(const int* counts, const int* cPerm, const int* activeSlots, int* src)
{
	int n = counts[CNT_CONTACTS];
	int t = blockIdx.x * blockDim.x + threadIdx.x;
	if (t < n)
	{
		src[t] = activeSlots[cPerm[t]];
	}
}

// ---- building the sorted incidence lists (once per step, after the solve order is known) --------------------------

// value of an item in the per-body sort: high word = (group << 1 | isContact), low word = the incidence entry without its
// side bit, whose top bits are the stream position t. Sorting the 64-bit values orders by (group, joints first, t).
__global__ void s2bItemOrderKernel(const int* counts, const int* cPerm, const int* jPerm, const int* cGroupOff, const int* jGroupOff,
								   int tableEntries, unsigned long long* itemVal)
{
	int nJ = counts[CNT_JOINTS], nC = counts[CNT_CONTACTS];
	int p = blockIdx.x * blockDim.x + threadIdx.x;
	if (p >= nJ + nC)
	{
		return;
	}
	bool isContact = p >= nJ;
	int t = isContact ? p - nJ : p;
	const int* off = isContact ? cGroupOff : jGroupOff;
	// largest g in [0, tableEntries) with off[g] <= t
	int lo = 0, hi = tableEntries - 1;
	while (lo < hi)
	{
		int mid = (lo + hi + 1) >> 1;
		if (off[mid] <= t)
		{
			lo = mid;
		}
		else
		{
			hi = mid - 1;
		}
	}
	int natural = isContact ? cPerm[t] : jPerm[t];
	int item = isContact ? nJ + natural : natural;
	unsigned long long key = ((unsigned long long)(unsigned)((lo << 1) | (isContact ? 1 : 0))) << 32;
	unsigned entry = ((unsigned)t << 2) | (isContact ? S2B_INC_CONTACT : 0);
	itemVal[item] = key | entry;
}

// The same from the 16-bit solve-order keys of the colour schedule (solver.cu, s2bMakeSortKeys): the key of an item IS its
// group in serial order (region x colour, then cut colours, then the overflow group).
__global__ void s2bItemOrderFromKeysKernel(const int* counts, const int* cPerm, const int* jPerm, const unsigned short* jKeys,
										   const unsigned short* cKeys, unsigned long long* itemVal)
{
	int nJ = counts[CNT_JOINTS], nC = counts[CNT_CONTACTS];
	int p = blockIdx.x * blockDim.x + threadIdx.x;
	if (p >= nJ + nC)
	{
		return;
	}
	bool isContact = p >= nJ;
	int t = isContact ? p - nJ : p;
	int natural = isContact ? cPerm[t] : jPerm[t];
	int item = isContact ? nJ + natural : natural;
	unsigned groupKey = isContact ? cKeys[natural] : jKeys[natural];
	unsigned long long key = ((unsigned long long)((groupKey << 1) | (isContact ? 1u : 0u))) << 32;
	unsigned entry = ((unsigned)t << 2) | (isContact ? S2B_INC_CONTACT : 0);
	itemVal[item] = key | entry;
}

// Besides the sorted list this also hands every constraint its ORDINAL in the lists of its two bodies (k-th of d incident
// items): what the ticketed Gauss-Seidel passes (solver.cu, "dataflow") wait on instead of a grid barrier.
// lists longer than this are sorted by a whole block (s2bSortLongIncidenceKernel) instead of one thread
#define S2B_LONG_LIST 24
#define S2B_LONG_LIST_SHARED 2048

__global__ void s2bSortIncidenceKernel(int bodyCapacity, const int* adjStart, const int* adj, const int2* itemBodies,
									   const unsigned long long* itemVal, unsigned long long* work, int* incList, int2* cFlowA,
									   int2* cFlowB, int2* jFlowA, int2* jFlowB, int* heavyBodies, int* longBodies)
{
	int b = blockIdx.x * blockDim.x + threadIdx.x;
	if (b >= bodyCapacity)
	{
		return;
	}
	int begin = adjStart[b], end = adjStart[b + 1];
	int n = end - begin;
	if (n == 0)
	{
		return;
	}
	if (heavyBodies != nullptr && n > S2B_HEAVY_DEGREE)
	{
		heavyBodies[1 + atomicAdd(heavyBodies, 1)] = b; // the list holds bodyCapacity entries
	}
	if (n > S2B_LONG_LIST)
	{
		// a hub body (container wall: hundreds of entries): one thread sorting it in global memory takes milliseconds
		longBodies[1 + atomicAdd(longBodies, 1)] = b;
		return;
	}
	if (n <= 8)
	{
		// the common case (a box touches ~6 others): sort in registers, touch global memory once per entry
		unsigned long long r[8];
#pragma unroll
		for (int k = 0; k < 8; ++k)
		{
			r[k] = ~0ull;
			if (k < n)
			{
				int item = adj[begin + k];
				unsigned long long val = itemVal[item];
				if (itemBodies[item].x != b)
				{
					val |= S2B_INC_SIDE_B;
				}
				r[k] = val;
			}
		}
		// odd-even transposition network on 8 keys (padding keys are the largest value and stay at the end)
#pragma unroll
		for (int pass = 0; pass < 8; ++pass)
		{
#pragma unroll
			for (int k = pass & 1; k + 1 < 8; k += 2)
			{
				unsigned long long lo = r[k] < r[k + 1] ? r[k] : r[k + 1];
				unsigned long long hi = r[k] < r[k + 1] ? r[k + 1] : r[k];
				r[k] = lo;
				r[k + 1] = hi;
			}
		}
#pragma unroll
		for (int k = 0; k < 8; ++k)
		{
			if (k < n)
			{
				int e = (int)(unsigned)(r[k] & 0xFFFFFFFFull);
				incList[begin + k] = e;
				if (cFlowA != nullptr)
				{
					int t = e >> 2;
					int2 ticket = make_int2(k, n);
					if (e & S2B_INC_CONTACT)
					{
						((e & S2B_INC_SIDE_B) ? cFlowB : cFlowA)[t] = ticket;
					}
					else
					{
						((e & S2B_INC_SIDE_B) ? jFlowB : jFlowA)[t] = ticket;
					}
				}
			}
		}
		return;
	}
	unsigned long long* v = work + begin;
	for (int k = 0; k < n; ++k)
	{
		int item = adj[begin + k];
		unsigned long long val = itemVal[item];
		if (itemBodies[item].x != b)
		{
			val |= S2B_INC_SIDE_B;
		}
		v[k] = val;
	}
	if (n <= 24)
	{
		for (int k = 1; k < n; ++k)
		{
			unsigned long long x = v[k];
			int m = k - 1;
			while (m >= 0 && v[m] > x)
			{
				v[m + 1] = v[m];
				m -= 1;
			}
			v[m + 1] = x;
		}
	}
	else
	{
		// heap sort: bodies touching hundreds of constraints (a container wall) stay O(n log n)
		for (int start = n / 2 - 1; start >= 0; --start)
		{
			int root = start;
			for (;;)
			{
				int child = 2 * root + 1;
				if (child >= n)
				{
					break;
				}
				if (child + 1 < n && v[child] < v[child + 1])
				{
					child += 1;
				}
				if (v[root] >= v[child])
				{
					break;
				}
				unsigned long long tmp = v[root];
				v[root] = v[child];
				v[child] = tmp;
				root = child;
			}
		}
		for (int last = n - 1; last > 0; --last)
		{
			unsigned long long tmp = v[0];
			v[0] = v[last];
			v[last] = tmp;
			int root = 0;
			for (;;)
			{
				int child = 2 * root + 1;
				if (child >= last)
				{
					break;
				}
				if (child + 1 < last && v[child] < v[child + 1])
				{
					child += 1;
				}
				if (v[root] >= v[child])
				{
					break;
				}
				unsigned long long t2 = v[root];
				v[root] = v[child];
				v[child] = t2;
				root = child;
			}
		}
	}
	for (int k = 0; k < n; ++k)
	{
		int e = (int)(unsigned)(v[k] & 0xFFFFFFFFull);
		incList[begin + k] = e;
		if (cFlowA != nullptr)
		{
			int t = e >> 2;
			int2 ticket = make_int2(k, n);
			if (e & S2B_INC_CONTACT)
			{
				((e & S2B_INC_SIDE_B) ? cFlowB : cFlowA)[t] = ticket;
			}
			else
			{
				((e & S2B_INC_SIDE_B) ? jFlowB : jFlowA)[t] = ticket;
			}
		}
	}
}

// Long incidence lists, one block per body: bitonic sort of the 64-bit values in shared memory (up to 2048 entries; longer
// lists fall back to a heap sort by one thread), then the same outputs as s2bSortIncidenceKernel.
__global__ void __launch_bounds__(256) s2bSortLongIncidenceKernel(const int* longBodies, const int* adjStart, const int* adj, const int2* itemBodies,
																  const unsigned long long* itemVal, unsigned long long* work, int* incList, int2* cFlowA,
																  int2* cFlowB, int2* jFlowA, int2* jFlowB)
{
	__shared__ unsigned long long sKeys[S2B_LONG_LIST_SHARED];
	int count = longBodies[0];
	for (int which = blockIdx.x; which < count; which += gridDim.x)
	{
		int b = longBodies[1 + which];
		int begin = adjStart[b], end = adjStart[b + 1];
		int n = end - begin;
		unsigned long long* v = work + begin;
		for (int k = threadIdx.x; k < n; k += blockDim.x)
		{
			int item = adj[begin + k];
			unsigned long long val = itemVal[item];
			if (itemBodies[item].x != b)
			{
				val |= S2B_INC_SIDE_B;
			}
			v[k] = val;
		}
		__syncthreads();
		if (n <= S2B_LONG_LIST_SHARED)
		{
			int padded = 1;
			while (padded < n)
			{
				padded <<= 1;
			}
			for (int k = threadIdx.x; k < padded; k += blockDim.x)
			{
				sKeys[k] = k < n ? v[k] : ~0ull;
			}
			__syncthreads();
			for (int size = 2; size <= padded; size <<= 1)
			{
				for (int stride = size >> 1; stride > 0; stride >>= 1)
				{
					for (int k = threadIdx.x; k < padded; k += blockDim.x)
					{
						int partner = k ^ stride;
						if (partner > k)
						{
							bool ascending = (k & size) == 0;
							unsigned long long x = sKeys[k], y = sKeys[partner];
							if ((x > y) == ascending)
							{
								sKeys[k] = y;
								sKeys[partner] = x;
							}
						}
					}
					__syncthreads();
				}
			}
			for (int k = threadIdx.x; k < n; k += blockDim.x)
			{
				v[k] = sKeys[k];
			}
			__syncthreads();
		}
		else if (threadIdx.x == 0)
		{
			// heap sort in global memory (lists beyond the shared-memory buffer: not seen in practice)
			for (int start = n / 2 - 1; start >= 0; --start)
			{
				int root = start;
				for (;;)
				{
					int child = 2 * root + 1;
					if (child >= n)
					{
						break;
					}
					if (child + 1 < n && v[child] < v[child + 1])
					{
						child += 1;
					}
					if (v[root] >= v[child])
					{
						break;
					}
					unsigned long long tmp = v[root];
					v[root] = v[child];
					v[child] = tmp;
					root = child;
				}
			}
			for (int last = n - 1; last > 0; --last)
			{
				unsigned long long tmp = v[0];
				v[0] = v[last];
				v[last] = tmp;
				int root = 0;
				for (;;)
				{
					int child = 2 * root + 1;
					if (child >= last)
					{
						break;
					}
					if (child + 1 < last && v[child] < v[child + 1])
					{
						child += 1;
					}
					if (v[root] >= v[child])
					{
						break;
					}
					unsigned long long t2 = v[root];
					v[root] = v[child];
					v[child] = t2;
					root = child;
				}
			}
		}
		__syncthreads();
		for (int k = threadIdx.x; k < n; k += blockDim.x)
		{
			int e = (int)(unsigned)(v[k] & 0xFFFFFFFFull);
			incList[begin + k] = e;
			if (cFlowA != nullptr)
			{
				int t = e >> 2;
				int2 ticket = make_int2(k, n);
				if (e & S2B_INC_CONTACT)
				{
					((e & S2B_INC_SIDE_B) ? cFlowB : cFlowA)[t] = ticket;
				}
				else
				{
					((e & S2B_INC_SIDE_B) ? jFlowB : jFlowA)[t] = ticket;
				}
			}
		}
		__syncthreads();
	}
}

// ConstraintView::lastTouch from the sorted incidence lists: the last entry of a body's list is the last constraint of the
// solve order that touches it. Bit 2 marks a constraint row as such for side A (bit 0) / B (bit 1); a body whose last
// toucher is a joint gets no mark at all (the persistent kernel only folds when there are no joints).
__global__ void s2bLastTouchKernel(int bodyCapacity, const int* incStart, const int* incList, int* lastTouch)
{
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= bodyCapacity)
	{
		return;
	}
	int begin = incStart[i], end = incStart[i + 1];
	if (end > begin)
	{
		int e = incList[end - 1];
		if (e & S2B_INC_CONTACT)
		{
			atomicOr(lastTouch + (e >> 2), (e & S2B_INC_SIDE_B) ? 2 : 1);
		}
	}
}

// ---- launch-by-launch kernels (profiling / cross-check path) ----------------------------------------------------

__global__ void __launch_bounds__(S2B_BLOCK) s2bBodyPassKernel(SolveArgs a, int bodyOp)
{
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < a.bodies.capacity)
	{
		s2bRunBodyOp(bodyOp, a, i);
	}
}

// THE per-colour impulse kernel on its own (TGS_Soft solve / relax over one colour): what the persistent kernel executes
// between two grid barriers, as a plain kernel with only this op in it (lean registers, full occupancy). Used by the
// roofline probe s2b_time_color_kernel.
__global__ void __launch_bounds__(S2B_BLOCK) s2bTgsSoftColorKernel(SolveArgs a, int cBegin, int cEnd, int useBias)
{
	int t = cBegin + blockIdx.x * blockDim.x + threadIdx.x;
	if (t < cEnd)
	{
		s2bSolveContactTgsSoft(a, t, a.ctx.inv_h, useBias != 0);
	}
}

// The same kernel with the constraint stream staged through shared memory by the TMA engine: the block's slice of every
// stream column is one contiguous run, so one thread issues eight 1-D bulk copies (cp.async.bulk, completion counted on an
// mbarrier) and the 256 threads then read their row from shared memory; only the gather of the two bodies and the final
// stores go through the load/store units. Same arithmetic, same bits.
#define S2B_BULK_BLOCK 256
#define S2B_BULK_ROWS (S2B_BULK_BLOCK + 2) // the slice may start one row early to keep 8-byte columns 16-byte aligned

__global__ void __launch_bounds__(S2B_BULK_BLOCK) s2bTgsSoftColorKernelBulk(SolveArgs a, int cBegin, int cEnd, int useBias)
{
	using BlockBarrier = cuda::barrier<cuda::thread_scope_block>;
	__shared__ alignas(16) int2 sIdx[S2B_BULK_ROWS];
	__shared__ alignas(16) float4 sNf[S2B_BULK_ROWS];
	__shared__ alignas(16) float4 sAnchor[2][S2B_BULK_ROWS];
	__shared__ alignas(16) float4 sPm[2][S2B_BULK_ROWS];
	__shared__ alignas(16) float2 sLambda[2][S2B_BULK_ROWS];
#pragma nv_diag_suppress static_var_with_dynamic_init
	__shared__ BlockBarrier bar;

	int t0 = cBegin + blockIdx.x * blockDim.x;
	int ta = t0 & ~1;									 // even row: 16-byte aligned in the 8-byte columns
	int tEnd = min(t0 + (int)blockDim.x, cEnd);
	int rows = ((tEnd - ta) + 1) & ~1;					 // even count: byte sizes are multiples of 16
	if (threadIdx.x == 0)
	{
		init(&bar, blockDim.x);
		cuda::device::experimental::fence_proxy_async_shared_cta();
	}
	__syncthreads();
	BlockBarrier::arrival_token token;
	if (threadIdx.x == 0)
	{
		const ConstraintView& cc = a.cc;
		unsigned b8 = (unsigned)rows * 8u, b16 = (unsigned)rows * 16u;
		cuda::device::memcpy_async_tx(sIdx, cc.idx + ta, cuda::aligned_size_t<16>(b8), bar);
		cuda::device::memcpy_async_tx(sNf, cc.nf + ta, cuda::aligned_size_t<16>(b16), bar);
		cuda::device::memcpy_async_tx(sAnchor[0], cc.anchor[0] + ta, cuda::aligned_size_t<16>(b16), bar);
		cuda::device::memcpy_async_tx(sAnchor[1], cc.anchor[1] + ta, cuda::aligned_size_t<16>(b16), bar);
		cuda::device::memcpy_async_tx(sPm[0], cc.pm[0] + ta, cuda::aligned_size_t<16>(b16), bar);
		cuda::device::memcpy_async_tx(sPm[1], cc.pm[1] + ta, cuda::aligned_size_t<16>(b16), bar);
		cuda::device::memcpy_async_tx(sLambda[0], cc.lambda[0] + ta, cuda::aligned_size_t<16>(b8), bar);
		cuda::device::memcpy_async_tx(sLambda[1], cc.lambda[1] + ta, cuda::aligned_size_t<16>(b8), bar);
		token = cuda::device::barrier_arrive_tx(bar, 1, 3 * b8 + 5 * b16);
	}
	else
	{
		token = bar.arrive();
	}
	bar.wait(std::move(token));

	int t = t0 + threadIdx.x;
	if (t < cEnd)
	{
		int r = t - ta;
		ContactStream cs;
		cs.slot = -1;
		cs.last = 0;
		cs.idx = sIdx[r];
		cs.nf = sNf[r];
		cs.la0 = sAnchor[0][r];
		cs.la1 = sAnchor[1][r];
		cs.pm0 = sPm[0][r];
		cs.pm1 = sPm[1][r];
		cs.l0 = sLambda[0][r];
		cs.l1 = sLambda[1][r];
		s2bSolveContactTgsSoftStream(a, t, cs, a.ctx.inv_h, useBias != 0);
	}
}

// one group (or the whole range): joints first, then contacts
__global__ void __launch_bounds__(S2B_BLOCK) s2bRangePassKernel(SolveArgs a, PassPtrs p, int jointOp, int contactOp, int jBegin, int jEnd,
															   int cBegin, int cEnd)
{
	int t = blockIdx.x * blockDim.x + threadIdx.x;
	int nj = jointOp != JOP_NONE ? jEnd - jBegin : 0;
	if (t < nj)
	{
		s2bRunJointOp(jointOp, a, jBegin + t, p);
	}
	else if (contactOp != COP_NONE && t - nj < cEnd - cBegin)
	{
		s2bRunContactOp(contactOp, a, cBegin + (t - nj));
	}
}

// serial overflow group: one thread walks the items in order
__global__ void s2bSerialPassKernel(SolveArgs a, PassPtrs p, int jointOp, int contactOp, int jBegin, int jEnd, int cBegin, int cEnd)
{
	if (blockIdx.x == 0 && threadIdx.x == 0)
	{
		if (jointOp != JOP_NONE)
		{
			for (int t = jBegin; t < jEnd; ++t)
			{
				s2bRunJointOp(jointOp, a, t, p);
			}
		}
		if (contactOp != COP_NONE)
		{
			for (int t = cBegin; t < cEnd; ++t)
			{
				s2bRunContactOp(contactOp, a, t);
			}
		}
	}
}

__global__ void s2bMeterWork(const int* counts, int passes, unsigned long long* work)
{
	work[0] += (unsigned long long)(counts[CNT_CONTACTS] + counts[CNT_JOINTS]) * (unsigned long long)passes;
	work[1] += 1ull;
}

// ---------------------------------------------------------------------------------------------------------------
// host driver
// ---------------------------------------------------------------------------------------------------------------

static SoftCoef makeSoft(float h, float hertz, float zeta)
{
	// reference src/solve_common.c:264-271 (contacts), src/revolute_joint.c:470-476 (joints)
	SoftCoef c;
	float omega = 2.0f * s2_pi * hertz;
	float cc = h * omega * (2.0f * zeta + h * omega);
	c.bias = omega / (2.0f * zeta + h * omega);
	c.impulse = 1.0f / (1.0f + cc);
	c.mass = cc * c.impulse;
	return c;
}

struct HostPlan
{
	// launch-by-launch mode only
	int groups = 0;
	std::vector<int> cOff, jOff;
};

static PassDesc bodyPass(int op)
{
	PassDesc d = {PASS_BODY, (unsigned char)op, JOP_NONE, COP_NONE};
	return d;
}

static PassDesc flatPass(int jop, int cop)
{
	PassDesc d = {PASS_FLAT, BOP_NONE, (unsigned char)jop, (unsigned char)cop};
	return d;
}

static PassDesc groupPass(int jop, int cop)
{
	PassDesc d = {PASS_GROUP, BOP_NONE, (unsigned char)jop, (unsigned char)cop};
	return d;
}

struct ProgramBuilder
{
	Program prog;
	ProgramBuilder()
	{
		memset(&prog, 0, sizeof(prog));
	}
	void segment(int repeat)
	{
		prog.repeat[prog.segmentCount] = repeat;
		prog.passCount[prog.segmentCount] = 0;
		prog.segmentCount += 1;
	}
	void add(PassDesc d)
	{
		int s = prog.segmentCount - 1;
		prog.passes[s][prog.passCount[s]++] = d;
	}
};

// The stage list of every variant (SURVEY.md §3.2-3.3), taken from the variant's driver in the reference. Also returns
// the number of solve passes per step that count as constraint-iterations (SURVEY.md §8d).
static Program buildProgram(int solverType, const s2bStepContext& ctx, bool gatherWarm, int* countedPasses)
{
	ProgramBuilder b;
	int S = ctx.iterations, E = ctx.extraIterations;
	bool warm = ctx.warmStart != 0;
	*countedPasses = 0;
	switch (solverType)
	{
		case 7: // s2Solve_TGS_Soft, reference src/solve_tgs_soft.c:138-280
		case 5: // s2Solve_SoftStep, reference src/solve_soft_step.c:182-311 (fixed anchors for velocity / impulse)
		{
			bool softStep = solverType == 5;
			b.segment(1);
			b.add(flatPass(JOP_PREPARE_SOFT_WARM, COP_PREPARE));
			// TGS_Soft with relax sweeps: the last sub-step's relax sweep also writes the impulses to the manifolds
			// (COP_TGS_SOFT_RELAX_STORE), so the closing store pass only has the joints left
			bool foldStore = softStep == false && E > 0 && S > 0;
			for (int part = 0; part < (foldStore ? 2 : 1); ++part)
			{
				bool last = foldStore && part == 1;
				b.segment(foldStore ? (last ? 1 : S - 1) : S);
				if (warm && gatherWarm)
				{
					b.add(bodyPass(softStep ? BOP_INTEGRATE_VELOCITIES_WARM_FIXED : BOP_INTEGRATE_VELOCITIES_WARM));
				}
				else
				{
					b.add(bodyPass(BOP_INTEGRATE_VELOCITIES));
					if (warm)
					{
						b.add(groupPass(JOP_WARM_START, softStep ? COP_WARM_START_FIXED : COP_WARM_START));
					}
				}
				b.add(groupPass(JOP_SOFT_BIAS, softStep ? COP_SOFTSTEP_BIAS : COP_TGS_SOFT_BIAS));
				b.add(bodyPass(BOP_INTEGRATE_POSITIONS));
				if (E > 0)
				{
					b.add(groupPass(JOP_SOFT_RELAX, softStep ? COP_SOFTSTEP_RELAX : (last ? COP_TGS_SOFT_RELAX_STORE : COP_TGS_SOFT_RELAX)));
				}
			}
			b.segment(1);
			b.add(bodyPass(BOP_FINALIZE_POSITIONS));
			b.add(flatPass(JOP_STORE, foldStore ? COP_NONE : COP_STORE));
			*countedPasses = S * (1 + (E > 0 ? 1 : 0));
			break;
		}
		case 1: // s2Solve_PGS, reference src/solve_pgs.c:125-213
		case 2: // s2Solve_PGS_NGS, reference src/solve_pgs_ngs.c:149-255
		case 4: // s2Solve_PGS_Soft, reference src/solve_pgs_soft.c:127-242
		case 0: // s2Solve_Jacobi, reference src/solve_jacobi.c:134-292
		{
			bool soft = solverType == 4 || solverType == 0;
			bool jacobi = solverType == 0;
			b.segment(1);
			if (jacobi)
			{
				b.add(bodyPass(BOP_JACOBI_RESET));
			}
			b.add(bodyPass(BOP_INTEGRATE_VELOCITIES));
			b.add(flatPass(soft ? JOP_PREPARE_SOFT_FLAG : JOP_PREPARE_RIGID_FLAG, COP_PREPARE));
			if (warm)
			{
				// all contacts are warm started before any joint (reference e.g. src/solve_pgs.c:166-184)
				b.add(groupPass(JOP_NONE, COP_WARM_START));
				b.add(groupPass(JOP_WARM_START, COP_NONE));
			}
			b.segment(S);
			if (solverType == 1)
			{
				b.add(groupPass(JOP_BAUMGARTE_BIAS, COP_PGS_BAUMGARTE));
			}
			else if (solverType == 2)
			{
				b.add(groupPass(JOP_RIGID, COP_PGS));
			}
			else if (solverType == 4)
			{
				b.add(groupPass(JOP_SOFT_BIAS, COP_PGS_SOFT_BIAS));
			}
			else
			{
				b.add(groupPass(JOP_SOFT_BIAS, COP_JACOBI_BIAS));
				b.add(bodyPass(BOP_JACOBI_APPLY));
			}
			b.segment(1);
			b.add(bodyPass(BOP_INTEGRATE_POSITIONS));
			if (solverType == 1)
			{
				b.add(bodyPass(BOP_FINALIZE_POSITIONS));
				b.add(flatPass(JOP_STORE, COP_STORE));
				*countedPasses = S;
			}
			else if (solverType == 2)
			{
				b.add(flatPass(JOP_NONE, COP_STORE)); // impulses are stored before the position iterations
				b.segment(E);
				b.add(groupPass(JOP_POSITION, COP_NGS));
				b.segment(1);
				b.add(bodyPass(BOP_FINALIZE_POSITIONS));
				b.add(flatPass(JOP_STORE, COP_NONE));
				*countedPasses = S + E;
			}
			else
			{
				b.segment(E);
				if (jacobi)
				{
					b.add(groupPass(JOP_SOFT_RELAX, COP_JACOBI_RELAX));
					b.add(bodyPass(BOP_JACOBI_APPLY));
				}
				else
				{
					b.add(groupPass(JOP_SOFT_RELAX, COP_PGS_SOFT_RELAX));
				}
				b.segment(1);
				b.add(bodyPass(BOP_FINALIZE_POSITIONS));
				b.add(flatPass(JOP_STORE, COP_STORE));
				*countedPasses = S + E;
			}
			break;
		}
		case 3: // s2Solve_PGS_NGS_Block, reference src/solve_pgs_ngs_block.c:892-963
		{
			b.segment(1);
			b.add(bodyPass(BOP_INTEGRATE_VELOCITIES));
			b.add(flatPass(JOP_PREPARE_RIGID_FLAG, COP_PREPARE_BLOCK));
			// s2CreateContactSolver applies the (possibly zero) stored impulses unconditionally (:264-299), before any joint
			b.add(groupPass(JOP_NONE, COP_WARM_START_FIXED));
			if (warm)
			{
				b.add(groupPass(JOP_WARM_START, COP_NONE));
			}
			b.segment(S);
			b.add(groupPass(JOP_RIGID, COP_BLOCK_VELOCITY));
			b.segment(1);
			b.add(flatPass(JOP_NONE, COP_STORE)); // before the position iterations (:934)
			b.add(bodyPass(BOP_INTEGRATE_POSITIONS));
			b.segment(E);
			// the position iterations visit the contacts BEFORE the joints (:938-952): two sweeps keep that order in
			// every schedule
			b.add(groupPass(JOP_NONE, COP_BLOCK_POSITION));
			b.add(groupPass(JOP_POSITION, COP_NONE));
			b.segment(1);
			b.add(bodyPass(BOP_FINALIZE_POSITIONS));
			b.add(flatPass(JOP_STORE, COP_NONE));
			*countedPasses = S + E;
			break;
		}
		case 8: // s2Solve_TGS_NGS, reference src/solve_tgs_ngs.c:207-317
		{
			b.segment(1);
			b.add(flatPass(JOP_PREPARE_RIGID_FLAG, COP_PREPARE));
			b.segment(S);
			if (warm && gatherWarm)
			{
				b.add(bodyPass(BOP_INTEGRATE_VELOCITIES_WARM));
			}
			else
			{
				b.add(bodyPass(BOP_INTEGRATE_VELOCITIES));
				if (warm)
				{
					b.add(groupPass(JOP_WARM_START, COP_WARM_START));
				}
			}
			b.add(groupPass(JOP_RIGID, COP_TGS));
			b.add(bodyPass(BOP_INTEGRATE_POSITIONS));
			b.add(groupPass(JOP_POSITION, COP_NGS));
			b.segment(1);
			b.add(bodyPass(BOP_FINALIZE_POSITIONS));
			b.add(flatPass(JOP_STORE, COP_STORE));
			*countedPasses = 2 * S;
			break;
		}
		case 6: // s2Solve_TGS_Sticky, reference src/solve_tgs_sticky.c:313-417
		{
			b.segment(1);
			b.add(flatPass(JOP_PREPARE_RIGID_COLD, COP_PREPARE_STICKY));
			b.segment(S);
			b.add(bodyPass(BOP_INTEGRATE_VELOCITIES));
			b.add(groupPass(JOP_BAUMGARTE_BIAS, COP_STICKY_BIAS));
			b.add(bodyPass(BOP_INTEGRATE_POSITIONS));
			b.segment(1);
			b.add(bodyPass(BOP_FINALIZE_POSITIONS));
			b.segment(E);
			b.add(groupPass(JOP_BAUMGARTE_RELAX, COP_STICKY_RELAX));
			b.segment(1);
			b.add(flatPass(JOP_STORE, COP_STORE));
			*countedPasses = S + E;
			break;
		}
		case 9: // s2Solve_XPBD, reference src/solve_xpbd.c:342-530
		{
			b.segment(1);
			b.add(flatPass(JOP_PREPARE_XPBD, COP_PREPARE_COLD));
			b.segment(S);
			b.add(bodyPass(BOP_XPBD_INTEGRATE));
			b.add(groupPass(JOP_XPBD, COP_XPBD_POSITIONS));
			b.add(bodyPass(BOP_XPBD_PROJECT));
			b.add(groupPass(JOP_NONE, COP_XPBD_VELOCITIES));
			b.segment(1);
			b.add(bodyPass(BOP_XPBD_FINALIZE));
			b.add(flatPass(JOP_STORE, COP_STORE_SCALED));
			*countedPasses = 2 * S;
			break;
		}
		default:
			break;
	}
	return b.prog;
}

static void runProgramLaunchByLaunch(s2bWorld* w, const SolveArgs& a, const PassPtrs& p, const Program& prog, const HostPlan& plan, int nJ,
									 int nC)
{
	for (int s = 0; s < prog.segmentCount; ++s)
	{
		for (int r = 0; r < prog.repeat[s]; ++r)
		{
			for (int k = 0; k < prog.passCount[s]; ++k)
			{
				PassDesc pass = prog.passes[s][k];
				if (pass.kind == PASS_BODY)
				{
					if (a.bodies.capacity > 0)
					{
						S2B_LAUNCH(w, s2bBodyPassKernel, gridFor(a.bodies.capacity, S2B_BLOCK), S2B_BLOCK, 0, a, (int)pass.bodyOp);
					}
				}
				else if (pass.kind == PASS_FLAT)
				{
					if (nJ + nC > 0)
					{
						S2B_LAUNCH(w, s2bRangePassKernel, gridFor(nJ + nC, S2B_BLOCK), S2B_BLOCK, 0, a, p, (int)pass.jointOp,
								   (int)pass.contactOp, 0, nJ, 0, nC);
					}
				}
				else
				{
					for (int g = 0; g < plan.groups; ++g)
					{
						int jb = plan.jOff[g], je = plan.jOff[g + 1], cb = plan.cOff[g], ce = plan.cOff[g + 1];
						int n = (pass.jointOp != JOP_NONE ? je - jb : 0) + (pass.contactOp != COP_NONE ? ce - cb : 0);
						if (n > 0)
						{
							S2B_LAUNCH(w, s2bRangePassKernel, gridFor(n, S2B_BLOCK), S2B_BLOCK, 0, a, p, (int)pass.jointOp,
									   (int)pass.contactOp, jb, je, cb, ce);
						}
					}
					int G = (int)plan.cOff.size() - 2; // table index of the overflow group
					int jb = plan.jOff[G], je = plan.jOff[G + 1], cb = plan.cOff[G], ce = plan.cOff[G + 1];
					int n = (pass.jointOp != JOP_NONE ? je - jb : 0) + (pass.contactOp != COP_NONE ? ce - cb : 0);
					if (n > 0)
					{
						S2B_LAUNCH(w, s2bSerialPassKernel, 1, 32, 0, a, p, (int)pass.jointOp, (int)pass.contactOp, jb, je, cb, ce);
					}
				}
			}
		}
	}
}

// wavefront levels on the host (validation schedule): level(i) = 1 + max level of earlier items sharing a movable body
static void buildWavefront(s2bWorld* w, SolverScratch* s, int nJ, int nC, HostPlan& plan)
{
	cudaStream_t st = w->stream;
	int n = nJ + nC;
	std::vector<int2> ends((size_t)std::max(n, 1));
	std::vector<int> activeSlots((size_t)std::max(nC, 1));
	std::vector<unsigned long long> keys;
	S2B_CHECK(cudaMemcpyAsync(ends.data(), s->itemBodies.p, sizeof(int2) * (size_t)n, cudaMemcpyDeviceToHost, st));
	if (nC > 0)
	{
		S2B_CHECK(cudaMemcpyAsync(activeSlots.data(), s->activeSlots.p, sizeof(int) * (size_t)nC, cudaMemcpyDeviceToHost, st));
	}
	bool hinted = w->orderHint.empty() == false && nC > 0;
	if (hinted)
	{
		keys.resize((size_t)w->contactCount);
		S2B_CHECK(cudaMemcpyAsync(keys.data(), w->contacts[w->cur].key.p, sizeof(unsigned long long) * keys.size(),
								  cudaMemcpyDeviceToHost, st));
	}
	S2B_CHECK(cudaStreamSynchronize(st));

	// sequential order of the contact constraints: natural (slot) order, or the imposed order
	std::vector<int> order((size_t)nC);
	for (int i = 0; i < nC; ++i)
	{
		order[i] = i;
	}
	if (hinted)
	{
		std::vector<std::pair<unsigned long long, int>> hint(w->orderHint.size());
		for (size_t k = 0; k < hint.size(); ++k)
		{
			hint[k] = {w->orderHint[k], (int)k};
		}
		std::sort(hint.begin(), hint.end());
		std::vector<long long> rank((size_t)nC);
		for (int i = 0; i < nC; ++i)
		{
			unsigned long long key = keys[(size_t)activeSlots[i]];
			auto it = std::lower_bound(hint.begin(), hint.end(), std::make_pair(key, -1));
			rank[i] = (it != hint.end() && it->first == key) ? (long long)it->second : (long long)hint.size() + i;
		}
		std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return rank[x] < rank[y]; });
	}

	std::vector<int> lastLevel((size_t)std::max(w->bodyCap, 1), 0);
	std::vector<int> level((size_t)std::max(n, 1), 0);
	int maxLevel = 0;
	auto place = [&](int item) {
		int2 e = ends[(size_t)item];
		int l = 0;
		if (e.x >= 0)
		{
			l = std::max(l, lastLevel[e.x]);
		}
		if (e.y >= 0)
		{
			l = std::max(l, lastLevel[e.y]);
		}
		l += 1;
		level[item] = l;
		if (e.x >= 0)
		{
			lastLevel[e.x] = l;
		}
		if (e.y >= 0)
		{
			lastLevel[e.y] = l;
		}
		maxLevel = std::max(maxLevel, l);
	};
	for (int i = 0; i < nJ; ++i)
	{
		place(i);
	}
	for (int k = 0; k < nC; ++k)
	{
		place(nJ + order[k]);
	}

	int G = maxLevel;
	plan.groups = G;
	plan.cOff.assign((size_t)G + 2, 0);
	plan.jOff.assign((size_t)G + 2, 0);
	for (int i = 0; i < nJ; ++i)
	{
		plan.jOff[(size_t)level[i]] += 1; // level l (1-based) stored at index l, shifted below
	}
	for (int i = 0; i < nC; ++i)
	{
		plan.cOff[(size_t)level[nJ + i]] += 1;
	}
	// exclusive scan with the 1-based shift: off[g] = number of items with level <= g
	for (int g = 1; g <= G; ++g)
	{
		plan.jOff[g] += plan.jOff[g - 1];
		plan.cOff[g] += plan.cOff[g - 1];
	}
	plan.jOff[G + 1] = plan.jOff[G];
	plan.cOff[G + 1] = plan.cOff[G];
	// now off[g-1]..off[g] is the range of level g  (off[0] = 0)
	std::vector<int> jPerm((size_t)std::max(nJ, 1)), cPerm((size_t)std::max(nC, 1));
	{
		std::vector<int> jc(plan.jOff.begin(), plan.jOff.end()), ccur(plan.cOff.begin(), plan.cOff.end());
		for (int i = 0; i < nJ; ++i)
		{
			jPerm[(size_t)jc[(size_t)level[i] - 1]++] = i;
		}
		for (int k = 0; k < nC; ++k)
		{
			int i = order[k];
			cPerm[(size_t)ccur[(size_t)level[nJ + i] - 1]++] = i;
		}
	}

	s->cGroupOff.reserve((size_t)G + 2, st, false);
	s->jGroupOff.reserve((size_t)G + 2, st, false);
	S2B_CHECK(cudaMemcpyAsync(s->cGroupOff.p, plan.cOff.data(), sizeof(int) * ((size_t)G + 2), cudaMemcpyHostToDevice, st));
	S2B_CHECK(cudaMemcpyAsync(s->jGroupOff.p, plan.jOff.data(), sizeof(int) * ((size_t)G + 2), cudaMemcpyHostToDevice, st));
	if (nC > 0)
	{
		S2B_CHECK(cudaMemcpyAsync(s->cPerm.p, cPerm.data(), sizeof(int) * (size_t)nC, cudaMemcpyHostToDevice, st));
	}
	if (nJ > 0)
	{
		S2B_CHECK(cudaMemcpyAsync(s->jPerm.p, jPerm.data(), sizeof(int) * (size_t)nJ, cudaMemcpyHostToDevice, st));
	}
	int counts[CNT_SIZE] = {0};
	counts[CNT_CONTACTS] = nC;
	counts[CNT_JOINTS] = nJ;
	counts[CNT_GROUPS] = G;
	S2B_CHECK(cudaMemcpyAsync(s->counts.p, counts, sizeof(counts), cudaMemcpyHostToDevice, st));
	S2B_CHECK(cudaStreamSynchronize(st));
}

// Gate of the schedule inside the stage's CUDA graph: run the gather + schedule sub-graph only when the set of live
// constraints changed since it was last built (flag raised by the narrow phase when a manifold gains its first or loses
// its last point, by body rows whose validity / movability changed, by joint uploads; anything the host knows about —
// a replaced contact table, other settings — changes the graph signature instead and is rebuilt eagerly).
// The same word block also carries what the Kempe pass (s2bKempeKernel) wants to know about the scene's recent past:
// [1] replays since the last rebuild, [2] a rebuild skipped the pass because the scene was churning, [3] the value of [1]
// when the rebuild that is about to run was asked for. A scene that has gone quiet with a skipped pass still owed gets ONE
// rebuild of its own, so that it does not keep the extra colours for good.
__global__ void s2bScheduleGate(cudaGraphConditionalHandle handle, int* dirty)
{
	int v = dirty[0];
	dirty[0] = 0;
	if (v != 0)
	{
		dirty[3] = dirty[1];
		dirty[1] = 0;
	}
	else
	{
		int quiet = dirty[1] + 1;
		dirty[1] = quiet;
		if (quiet == S2B_KEMPE_QUIET_STEPS && dirty[2] != 0)
		{
			v = 1;
			dirty[3] = quiet;
			dirty[1] = 0;
		}
	}
	cudaGraphSetConditional(handle, v != 0 ? 1u : 0u);
}

// Everything one solver stage needs to know on the host before anything is enqueued.
struct SolvePlan
{
	int solverType = 0;
	s2bStepContext ctx;
	Program program;
	int countedPasses = 0;
	bool gatherWarm = false, dataflow = false, needInc = false, usePersistent = false;
	int contactCount = 0, jointCap = 0, bodyCap = 0, maxItems = 0;
	size_t nC = 1, nJ = 1, nI = 1;
	VariantColumns cols;
	int threads = S2B_BLOCK;
	int grid = 1;	 // blocks of the persistent kernel
	int regions = 0; // region-local schedule: == grid, or 0
	HostPlan host;	 // launch-by-launch / wavefront modes
	int hostNC = 0, hostNJ = 0;
};

static void verifyProgram(int solverType, const Program& prog)
{
	for (int s = 0; s < prog.segmentCount; ++s)
	{
		for (int k = 0; k < prog.passCount[s]; ++k)
		{
			PassDesc d = prog.passes[s][k];
			bool ok = (d.bodyOp == BOP_NONE || s2bUsesBodyOp(solverType, d.bodyOp)) && (d.jointOp == JOP_NONE || s2bUsesJointOp(solverType, d.jointOp)) &&
					  (d.contactOp == COP_NONE || s2bUsesContactOp(solverType, d.contactOp));
			if (ok == false)
			{
				fprintf(stderr, "solver2d-b200: internal error: program of solver %d uses an operation its kernel was built without (%d/%d/%d)\n",
						solverType, d.bodyOp, d.jointOp, d.contactOp);
				abort();
			}
		}
	}
}

// sizes, modes and scratch of this stage (host only; may allocate, never inside a capture that matters: a re-allocation
// bumps the allocation epoch and with it the graph signature)
static void planSolve(s2bWorld* w, SolverScratch* s, SolvePlan& pl)
{
	cudaStream_t st = w->stream;
	int solverType = pl.solverType;
	const s2bStepContext& ctx = pl.ctx;
	// per-sub-step warm starting as a per-body gather (warm_gather.cuh); S2B_WARM_GATHER=0 keeps the grouped passes
	pl.gatherWarm = w->gatherWarm != 0 && ctx.warmStart != 0 && (solverType == 7 || solverType == 5 || solverType == 8);
	pl.program = buildProgram(solverType, ctx, pl.gatherWarm, &pl.countedPasses);
	verifyProgram(solverType, pl.program);
	pl.usePersistent = w->persistent != 0 && w->coopSupported != 0;
	// ticketed Gauss-Seidel passes instead of grid barriers (persistent kernel only, experimental); S2B_DATAFLOW=1 enables
	pl.dataflow = w->dataflow != 0 && pl.usePersistent;
	pl.needInc = pl.gatherWarm || pl.dataflow;
	pl.contactCount = w->contactCount;
	pl.jointCap = w->jointCap;
	pl.bodyCap = w->bodyCap;
	pl.maxItems = pl.contactCount + pl.jointCap;
	pl.cols = columnsFor(solverType);
	int contactCount = pl.contactCount, jointCap = pl.jointCap, bodyCap = pl.bodyCap, maxItems = pl.maxItems;

	// grid of the persistent kernel
	pl.threads = S2B_BLOCK;
	pl.grid = 1;
	if (pl.usePersistent)
	{
		if (w->solveGrid == 0 || w->solveGridSolver != solverType)
		{
			int blocksPerSm = 0;
			S2B_CHECK(cudaFuncSetAttribute(s2bPersistentKernel(solverType), cudaFuncAttributeMaxDynamicSharedMemorySize, S2B_DYN_SHARED_BYTES));
			S2B_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocksPerSm, s2bPersistentKernel(solverType), S2B_BLOCK, S2B_DYN_SHARED_BYTES));
			const char* env = getenv("S2B_SOLVE_BLOCKS_PER_SM");
			int want = env != nullptr ? atoi(env) : 2;
			w->solveGrid = w->smCount * std::min(std::max(blocksPerSm, 1), std::max(want, 1));
			w->solveGridSolver = solverType;
		}
		const char* env = getenv("S2B_SOLVE_THREADS");
		if (env != nullptr && atoi(env) >= 32 && atoi(env) <= S2B_BLOCK)
		{
			pl.threads = atoi(env) & ~31;
		}
		int wanted = std::max(gridFor(std::max(maxItems, bodyCap), pl.threads), 1);
		pl.grid = std::min(std::min(w->solveGrid, wanted), 511); // 511: region ids share a 16-bit key with the colour
	}
	pl.regions = (w->schedule == S2B_SCHEDULE_COLOR && pl.usePersistent && w->useRegions != 0 && pl.dataflow == false && maxItems > 0)
					 ? pl.grid
					 : 0;
	if (w->useRegions == 1 && pl.regions > 0)
	{
		if (s->regionVerdictPending)
		{
			// (the copy was enqueued a step ago, behind a schedule the host has long waited past; a stale word is only a hint)
			s->regionVerdictPending = false;
			if (w->hostMail[MAIL_REGIONS_ON] == 0)
			{
				s->regionSkip = S2B_REGION_RETRY;
			}
		}
		if (s->regionSkip > 0)
		{
			s->regionSkip -= 1;
			pl.regions = 0;
		}
	}

	// ---- reserve scratch (sizes are upper bounds known on the host: no synchronisation) ----
	size_t nC = (size_t)std::max(contactCount, 1), nJ = (size_t)std::max(jointCap, 1), nI = (size_t)std::max(maxItems, 1);
	pl.nC = nC;
	pl.nJ = nJ;
	pl.nI = nI;
	VariantColumns cols = pl.cols;
	s->counts.reserve(CNT_SIZE, st, false);
	s->activeFlag.reserve(nC, st, false);
	s->activeSlots.reserve(nC, st, false);
	s->jointFlag.reserve(nJ, st, false);
	s->jointSlots.reserve(nJ, st, false);
	s->itemBodies.reserve(nI, st, false);
	s->degree.reserve((size_t)bodyCap + 1, st, false);
	s->adjStart.reserve((size_t)bodyCap + 2, st, false);
	s->adjCursor.reserve((size_t)bodyCap + 1, st, false);
	s->adj.reserve(2 * nI, st, false);
	s->colorA.reserve(nI, st, false);
	s->colorB.reserve(nI, st, false);
	s->colorC.reserve(nI, st, false);
	s->kempeState.reserve(KS_SIZE, st, false, true);
	s->kempeClaim.reserve((size_t)bodyCap + 1, st, false, false);
	s->kempePath.reserve((size_t)S2B_KEMPE_MAX_ITEMS * S2B_KEMPE_MAX_HOPS, st, false, false);
	s->itemRegion.reserve(nI, st, false);
	s->sortKeyIn.reserve(2 * nI, st, false);
	s->sortKeyOut.reserve(2 * nI, st, false);
	s->sortValIn.reserve(2 * nI, st, false);
	s->sortValOut.reserve(2 * nI, st, false);
	s->cGroupOff.reserve(S2B_MAX_COLORS + 2, st, false);
	s->jGroupOff.reserve(S2B_MAX_COLORS + 2, st, false);
	s->cPerm.reserve(nC, st, false);
	s->jPerm.reserve(nJ, st, false);
	s->heavyBodies.reserve((size_t)bodyCap + 2, st, false);
	s->ovBodies.reserve((size_t)bodyCap + 2, st, false);
	s->longBodies.reserve((size_t)bodyCap + 2, st, false);
	s->ovBodySlot.reserve((size_t)bodyCap + 2, st, false);
	if (pl.regions > 0)
	{
		s->bodyKeyIn.reserve((size_t)bodyCap + 1, st, false);
		s->bodyKeyOut.reserve((size_t)bodyCap + 1, st, false);
		s->bodyValIn.reserve((size_t)bodyCap + 1, st, false);
		s->bodySorted.reserve((size_t)bodyCap + 1, st, false);
		s->island.reserve((size_t)bodyCap + 1, st, false);
		s->islandParent.reserve((size_t)bodyCap + 1, st, false);
		s->islandSize.reserve((size_t)bodyCap + 1, st, false);
		s->islandStart.reserve((size_t)bodyCap + 1, st, false);
		s->regCount.reserve(1024, st, false);
		s->regBodies.reserve((size_t)bodyCap + 1, st, false);
		s->bodyLocal.reserve((size_t)bodyCap + 1, st, false);
		s->bodyRegion.reserve((size_t)bodyCap + 1, st, false);
		s->regBodyStart.reserve((size_t)pl.regions + 2, st, false);
		s->cRegOff.reserve((size_t)pl.regions * S2B_REG_STRIDE, st, false);
		s->jRegOff.reserve((size_t)pl.regions * S2B_REG_STRIDE, st, false);
	}
	if (pl.needInc)
	{
		s->itemVal.reserve(nI, st, false);
		s->incWork.reserve(2 * nI, st, false);
		s->incList.reserve(2 * nI, st, false);
		s->lastTouch.reserve(nC + 2, st, false);
	}
	if (pl.dataflow)
	{
		s->flow.reserve(2 * nC + 2 * nJ, st, false);
		s->bodyTicket.reserve((size_t)bodyCap + 2, st, false);
	}
	w->solveBarrier.reserve(64, st, true, true);
	w->schedDirty.reserve(4, st, true, true);
	// (+2 rows: the bulk-staged colour kernel may read up to two rows past the last constraint)
	s->idx.reserve(nC + 2, st, false);
	s->nf.reserve(nC + 2, st, false);
	s->src.reserve(nC, st, false);
	if (pl.gatherWarm)
	{
		s->warmP.reserve(nC, st, false);
		s->warmAnchor.reserve(2 * nC, st, false);
	}
	for (int p = 0; p < 2; ++p)
	{
		s->anchor[p].reserve(nC + 2, st, false);
		s->pm[p].reserve(nC + 2, st, false);
		s->lambda[p].reserve(nC + 2, st, false);
		if (cols.r0)
		{
			s->r0[p].reserve(nC, st, false);
		}
		if (cols.sep)
		{
			s->sep[p].reserve(nC, st, false);
		}
		if (cols.sticky)
		{
			s->fanchor[p].reserve(nC, st, false);
			s->tsep[p].reserve(nC, st, false);
		}
	}
	s->jhead.reserve(nJ, st, false);
	s->janchor.reserve(nJ, st, false);
	s->jmass.reserve(nJ, st, false);
	s->jd0ax.reserve(nJ, st, false);
	s->jlim.reserve(nJ, st, false);
	s->jmotor.reserve(nJ, st, false);
	s->jcoef.reserve(nJ, st, false);
	s->jpivot.reserve(nJ, st, false);
	s->jimp.reserve(nJ, st, false);
	s->jlimp.reserve(nJ, st, false);

	// cub temp storage (compaction, scan, sorts) sized for the largest use
	size_t tempBytes = 0, need = 0;
	cub::DeviceSelect::Flagged(nullptr, need, thrust::counting_iterator<int>(0), (int*)nullptr, (int*)nullptr, (int*)nullptr,
							   (int)nI, st);
	tempBytes = std::max(tempBytes, need);
	cub::DeviceScan::ExclusiveSum(nullptr, need, (int*)nullptr, (int*)nullptr, bodyCap + 1, st);
	tempBytes = std::max(tempBytes, need);
	cub::DeviceRadixSort::SortPairs(nullptr, need, (unsigned short*)nullptr, (unsigned short*)nullptr, (int*)nullptr, (int*)nullptr, (int)nI, 0,
									16, st);
	tempBytes = std::max(tempBytes, need);
	cub::DeviceRadixSort::SortPairs(nullptr, need, (unsigned long long*)nullptr, (unsigned long long*)nullptr, (int*)nullptr, (int*)nullptr,
									bodyCap + 1, 0, 64, st);
	tempBytes = std::max(tempBytes, need);
	s->cubTemp.reserve(tempBytes + 256, st, false, false);
}

static void launchColorKernel(s2bWorld* w, SolverScratch* s, int maxItems, int* color, int maxColors, int indexRounds, int validate,
							  int abortAbove = -1, const int* hubs = nullptr, int hubDegree = 0)
{
	// work counters of the kernel (shared by the primary and the cut colouring)
	S2B_CHECK(cudaMemsetAsync(s->counts.p + CNT_REMAINING, 0, sizeof(int) * 5, w->stream));
	if (w->colorGrid == 0)
	{
		int blocksPerSm = 0;
		S2B_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocksPerSm, s2bColorKernel, 256, 0));
		w->colorGrid = w->smCount * std::min(std::max(blocksPerSm, 1), 2);
	}
	int grid = std::min(w->colorGrid, std::max(1, gridFor(maxItems, 256)));
	int* countsPtr = s->counts.p;
	const int2* ib = s->itemBodies.p;
	const int* as = s->adjStart.p;
	const int* ad = s->adj.p;
	int* tent = s->colorB.p;
	void* args[] = {&countsPtr, &ib, &as, &ad, &color, &tent, &maxColors, &indexRounds, &validate, &abortAbove, &hubs, &hubDegree};
	S2B_CHECK(cudaLaunchCooperativeKernel((void*)s2bColorKernel, dim3(grid), dim3(256), args, 0, w->stream));
	w->kernelLaunches += 1;
}

static void launchKempeKernel(s2bWorld* w, SolverScratch* s, int bodyCap)
{
	if (w->kempeGrid == 0)
	{
		int blocksPerSm = 0;
		S2B_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&blocksPerSm, s2bKempeKernel, 256, 0));
		w->kempeGrid = w->smCount * std::min(std::max(blocksPerSm, 1), 2);
	}
	int grid = w->kempeGrid;
	const int* countsPtr = s->counts.p;
	const int2* ib = s->itemBodies.p;
	const int* as = s->adjStart.p;
	const int* ad = s->adj.p;
	int* color = s->colorA.p;
	int* state = s->kempeState.p;
	int* claim = s->kempeClaim.p;
	int* paths = s->kempePath.p;
	int* sched = w->schedDirty.p;
	void* args[] = {&countsPtr, &ib, &as, &ad, &color, &state, &claim, &paths, &bodyCap, &sched};
	S2B_CHECK(cudaLaunchCooperativeKernel((void*)s2bKempeKernel, dim3(grid), dim3(256), args, 0, w->stream));
	w->kernelLaunches += 1;
}

// gather + schedule: from the contact / joint tables to the solve order, the group tables, the regions and the incidence
// lists. Everything here depends only on WHICH constraints are live (and on the settings in the graph signature), not on
// their values: while that set stands, a replayed graph skips all of it (see s2bSolve).
static void enqueueSchedule(s2bWorld* w, SolverScratch* s, SolvePlan& pl)
{
	cudaStream_t st = w->stream;
	int contactCount = pl.contactCount, jointCap = pl.jointCap, bodyCap = pl.bodyCap, maxItems = pl.maxItems;
	size_t nI = pl.nI, nC = pl.nC, nJ = pl.nJ;

	// ---- gather ----
	S2B_CHECK(cudaMemsetAsync(w->schedDirty.p, 0, sizeof(int), st)); // what follows is the rebuild the flag asks for
	S2B_CHECK(cudaMemsetAsync(s->counts.p, 0, sizeof(int) * CNT_SIZE, st));
	{
		int n = std::max(contactCount, jointCap);
		if (n > 0)
		{
			S2B_LAUNCH(w, s2bFlagActive, gridFor(n, 256), 256, 0, makeView(w->contacts[w->cur]), contactCount, jointView(w),
					   jointCap, s->activeFlag.p, s->jointFlag.p);
		}
		size_t tb = s->cubTemp.cap;
		if (contactCount > 0)
		{
			cub::DeviceSelect::Flagged(s->cubTemp.p, tb, thrust::counting_iterator<int>(0), s->activeFlag.p, s->activeSlots.p,
									   s->counts.p + CNT_CONTACTS, contactCount, st);
			w->kernelLaunches += 2;
		}
		if (jointCap > 0)
		{
			tb = s->cubTemp.cap;
			cub::DeviceSelect::Flagged(s->cubTemp.p, tb, thrust::counting_iterator<int>(0), s->jointFlag.p, s->jointSlots.p,
									   s->counts.p + CNT_JOINTS, jointCap, st);
			w->kernelLaunches += 2;
		}
	}

	bool needHostCounts = (w->schedule == S2B_SCHEDULE_WAVEFRONT) || pl.usePersistent == false;
	s->regions = 0;
	if (maxItems > 0)
	{
		bool wantAdj = w->schedule == S2B_SCHEDULE_COLOR || pl.needInc;
		if (wantAdj)
		{
			S2B_CHECK(cudaMemsetAsync(s->degree.p, 0, sizeof(int) * ((size_t)bodyCap + 1), st));
			S2B_CHECK(cudaMemsetAsync(s->adjCursor.p, 0, sizeof(int) * ((size_t)bodyCap + 1), st));
		}
		S2B_LAUNCH(w, s2bItemEndpoints, gridFor(maxItems, 256), 256, 0, s->counts.p, s->jointSlots.p, s->activeSlots.p,
				   jointView(w), makeView(w->contacts[w->cur]), bodyView(w), s->itemBodies.p, wantAdj ? s->degree.p : nullptr);
		if (wantAdj)
		{
			size_t tb = s->cubTemp.cap;
			cub::DeviceScan::ExclusiveSum(s->cubTemp.p, tb, s->degree.p, s->adjStart.p, bodyCap + 1, st);
			w->kernelLaunches += 2;
			S2B_LAUNCH(w, s2bFillAdjacency, gridFor(maxItems, 256), 256, 0, s->counts.p, s->itemBodies.p, s->adjStart.p,
					   s->adjCursor.p, s->adj.p);
		}
		S2B_CHECK(cudaMemsetAsync(s->heavyBodies.p, 0, sizeof(int), st));

		if (w->schedule == S2B_SCHEDULE_COLOR)
		{
			if (w->coopSupported == 0)
			{
				fprintf(stderr, "solver2d-b200: cooperative launch unsupported on this device\n");
				abort();
			}
			// colours: start from the persisted ones; only constraints that appeared this step are uncoloured
			S2B_LAUNCH(w, s2bSeedColors, gridFor(maxItems, 256), 256, 0, s->counts.p, s->jointSlots.p, s->activeSlots.p, w->jColor.p,
					   w->contacts[w->cur].color.p, s->colorA.p, w->maxColors);
			launchColorKernel(w, s, maxItems, s->colorA.p, w->maxColors, S2B_INDEX_PRIORITY_ROUNDS, 1, -1, nullptr, w->hubDegree);
			if (w->kempe != 0)
			{
				launchKempeKernel(w, s, bodyCap);
			}
			S2B_LAUNCH(w, s2bStoreColors, gridFor(maxItems, 256), 256, 0, s->counts.p, s->jointSlots.p, s->activeSlots.p, w->jColor.p,
					   w->contacts[w->cur].color.p, s->colorA.p);

			// regions: Hilbert order of the bodies' centres, equal chunks
			if (pl.regions > 0)
			{
				// islands (union-find over the items), then Hilbert order with the island as the major key
				S2B_LAUNCH(w, s2bIslandInitKernel, gridFor(bodyCap, 256), 256, 0, bodyCap, s->islandParent.p);
				S2B_LAUNCH(w, s2bIslandHookKernel, gridFor(maxItems, 256), 256, 0, s->counts.p, s->itemBodies.p, s->islandParent.p);
				S2B_CHECK(cudaMemsetAsync(s->islandSize.p, 0, sizeof(int) * ((size_t)bodyCap + 1), st));
				S2B_CHECK(cudaMemsetAsync(s->islandStart.p, 0x7F, sizeof(int) * ((size_t)bodyCap + 1), st));
				S2B_CHECK(cudaMemsetAsync(s->regCount.p, 0, sizeof(int) * 512, st));
				S2B_LAUNCH(w, s2bIslandFlattenKernel, gridFor(bodyCap, 256), 256, 0, bodyView(w), s->islandParent.p, s->island.p, s->islandSize.p);
				S2B_LAUNCH(w, s2bBodyBoundsKernel, gridFor(bodyCap, 256), 256, 0, bodyView(w), s->counts.p);
				S2B_LAUNCH(w, s2bBodyKeysKernel, gridFor(bodyCap, 256), 256, 0, bodyView(w), s->counts.p, s->degree.p, s->island.p, s->bodyKeyIn.p,
						   s->bodyValIn.p, s->heavyBodies.p);
				size_t tb = s->cubTemp.cap;
				cub::DeviceRadixSort::SortPairs(s->cubTemp.p, tb, s->bodyKeyIn.p, s->bodyKeyOut.p, s->bodyValIn.p, s->bodySorted.p, bodyCap, 0, 64,
												st);
				w->kernelLaunches += 10;
				S2B_LAUNCH(w, s2bIslandStartKernel, gridFor(bodyCap, 256), 256, 0, s->counts.p, s->bodySorted.p, s->island.p, s->islandStart.p);
				S2B_LAUNCH(w, s2bAssignRegionsKernel, gridFor(bodyCap, 256), 256, 0, s->counts.p, bodyCap, pl.regions, s->bodySorted.p, s->island.p,
						   s->islandStart.p, s->islandSize.p, s->bodyRegion.p, s->regCount.p, w->wholeIslandBodies);
				S2B_LAUNCH(w, s2bRegionOffsetsKernel, 1, 512, 0, pl.regions, s->regCount.p, s->regBodyStart.p, s->regCount.p + 512, s->counts.p);
				S2B_LAUNCH(w, s2bFillRegionBodiesKernel, gridFor(bodyCap, 256), 256, 0, s->counts.p, s->bodySorted.p, s->bodyRegion.p,
						   s->regCount.p + 512, s->regBodies.p, s->regBodyStart.p, s->bodyLocal.p);
				s->regions = pl.regions;
			}
			S2B_LAUNCH(w, s2bClassifyItemsKernel, gridFor(maxItems, 256), 256, 0, s->counts.p, s->itemBodies.p, s->bodyRegion.p, s->colorA.p,
					   pl.regions > 0 ? 1 : 0, s->itemRegion.p, s->colorC.p);
			int regionCutLimit = -1;
			if (pl.regions > 0)
			{
				// the cut set is coloured among itself, from scratch, with hashed priorities (a handful of rounds)
				regionCutLimit = w->useRegions >= 2 ? S2B_MAX_COLORS : w->regionCutLimit;
				launchColorKernel(w, s, maxItems, s->colorC.p, S2B_MAX_COLORS, 0, 0, regionCutLimit < S2B_MAX_COLORS ? regionCutLimit - 1 : -1, s->heavyBodies.p);
				S2B_LAUNCH(w, s2bCutColorCountKernel, gridFor(maxItems, 256), 256, 0, s->counts.p, s->colorC.p);
			}

			// solve order: stable 16-bit radix sort of (key, natural index), joints and contacts separately
			unsigned short* jKeysIn = s->sortKeyIn.p;
			unsigned short* cKeysIn = s->sortKeyIn.p + nI;
			unsigned short* jKeysOut = s->sortKeyOut.p;
			unsigned short* cKeysOut = s->sortKeyOut.p + nI;
			int* jValsIn = s->sortValIn.p;
			int* cValsIn = s->sortValIn.p + nI;
			// entries beyond the live counts keep key 0xFFFF: they sort behind every live entry and are never read
			S2B_CHECK(cudaMemsetAsync(s->sortKeyIn.p, 0xFF, sizeof(unsigned short) * 2 * nI, st));
			S2B_LAUNCH(w, s2bMakeSortKeys, gridFor(maxItems, 256), 256, 0, s->counts.p, s->colorA.p, s->itemRegion.p, s->colorC.p, regionCutLimit,
					   jKeysIn, jValsIn, cKeysIn, cValsIn);
			// the sorts run over the host-known upper-bound sizes, so no device count has to be read back
			size_t tb = s->cubTemp.cap;
			if (contactCount > 0)
			{
				tb = s->cubTemp.cap;
				cub::DeviceRadixSort::SortPairs(s->cubTemp.p, tb, cKeysIn, cKeysOut, cValsIn, s->cPerm.p, contactCount, 0, 16, st);
				w->kernelLaunches += 3;
			}
			if (jointCap > 0)
			{
				tb = s->cubTemp.cap;
				cub::DeviceRadixSort::SortPairs(s->cubTemp.p, tb, jKeysIn, jKeysOut, jValsIn, s->jPerm.p, jointCap, 0, 16, st);
				w->kernelLaunches += 3;
			}
			int entries = pl.regions * S2B_REG_STRIDE + S2B_MAX_COLORS + 2;
			S2B_LAUNCH(w, s2bBuildTablesKernel, gridFor(entries, 256), 256, 0, pl.regions, jKeysOut, jointCap, cKeysOut, contactCount, s->jRegOff.p,
					   s->cRegOff.p, s->jGroupOff.p, s->cGroupOff.p);
			S2B_LAUNCH(w, s2bFinishGroups, 1, 1, 0, s->counts.p, s->cGroupOff.p, s->jGroupOff.p, s->heavyBodies.p,
					   (pl.regions > 0 && pl.solverType == 7 && pl.gatherWarm && w->residentRegions != 0) ? S2B_RES_MAX_BODIES : 0);
			// bodies of the serial overflow group (hub bodies' constraints beyond the colour limit), for its shared-memory walk
			S2B_CHECK(cudaMemsetAsync(s->ovBodySlot.p, 0xFF, sizeof(int) * ((size_t)bodyCap + 1), st));
			S2B_CHECK(cudaMemsetAsync(s->ovBodies.p, 0, sizeof(int), st));
			S2B_LAUNCH(w, s2bOverflowBodiesKernel, gridFor(maxItems, 256), 256, 0, s->counts.p, s->jGroupOff.p, s->cGroupOff.p, s->jPerm.p,
					   s->cPerm.p, s->jointSlots.p, s->activeSlots.p, jointView(w), makeView(w->contacts[w->cur]), s->ovBodySlot.p, s->ovBodies.p);
		}

		if (needHostCounts)
		{
			int hostCounts[CNT_SIZE];
			S2B_CHECK(cudaMemcpyAsync(hostCounts, s->counts.p, sizeof(hostCounts), cudaMemcpyDeviceToHost, st));
			S2B_CHECK(cudaStreamSynchronize(st));
			pl.hostNC = hostCounts[CNT_CONTACTS];
			pl.hostNJ = hostCounts[CNT_JOINTS];
			if (w->schedule == S2B_SCHEDULE_WAVEFRONT)
			{
				buildWavefront(w, s, pl.hostNJ, pl.hostNC, pl.host);
			}
			else
			{
				pl.host.groups = hostCounts[CNT_GROUPS];
				pl.host.cOff.resize(S2B_MAX_COLORS + 2);
				pl.host.jOff.resize(S2B_MAX_COLORS + 2);
				S2B_CHECK(cudaMemcpy(pl.host.cOff.data(), s->cGroupOff.p, sizeof(int) * (S2B_MAX_COLORS + 2), cudaMemcpyDeviceToHost));
				S2B_CHECK(cudaMemcpy(pl.host.jOff.data(), s->jGroupOff.p, sizeof(int) * (S2B_MAX_COLORS + 2), cudaMemcpyDeviceToHost));
			}
			s->hostContacts = pl.hostNC;
			s->hostJoints = pl.hostNJ;
			s->hostGroups = pl.host.groups;
			s->hostCGroupOff = pl.host.cOff;
			s->hostJGroupOff = pl.host.jOff;
			s->hostCountsValid = true;
		}
		else
		{
			s->hostCountsValid = false;
		}

		if (contactCount > 0)
		{
			S2B_LAUNCH(w, s2bBuildSources, gridFor(contactCount, 256), 256, 0, s->counts.p, s->cPerm.p, s->activeSlots.p, s->src.p);
		}

		if (pl.needInc)
		{
			// incidence lists of the movable bodies in solve order (+ the ticket ordinals of every constraint)
			if (w->schedule == S2B_SCHEDULE_COLOR)
			{
				S2B_LAUNCH(w, s2bItemOrderFromKeysKernel, gridFor(maxItems, 256), 256, 0, s->counts.p, s->cPerm.p, s->jPerm.p, s->sortKeyIn.p,
						   s->sortKeyIn.p + nI, s->itemVal.p);
			}
			else
			{
				S2B_LAUNCH(w, s2bItemOrderKernel, gridFor(maxItems, 256), 256, 0, s->counts.p, s->cPerm.p, s->jPerm.p, s->cGroupOff.p,
						   s->jGroupOff.p, std::max(pl.host.groups, 1), s->itemVal.p);
			}
			int2 *cfa = nullptr, *cfb = nullptr, *jfa = nullptr, *jfb = nullptr;
			if (pl.dataflow)
			{
				S2B_CHECK(cudaMemsetAsync(s->flow.p, 0xFF, sizeof(int2) * (2 * nC + 2 * nJ), st));
				cfa = s->flow.p;
				cfb = s->flow.p + nC;
				jfa = s->flow.p + 2 * nC;
				jfb = s->flow.p + 2 * nC + nJ;
			}
			// without regions the hub bodies (gathered by a whole block) are registered here; with regions s2bBodyKeysKernel did it
			int* heavy = (pl.gatherWarm && pl.usePersistent && pl.regions == 0) ? s->heavyBodies.p : nullptr;
			S2B_CHECK(cudaMemsetAsync(s->longBodies.p, 0, sizeof(int), st));
			S2B_LAUNCH(w, s2bSortIncidenceKernel, gridFor(bodyCap, 128), 128, 0, bodyCap, s->adjStart.p, s->adj.p, s->itemBodies.p,
					   s->itemVal.p, s->incWork.p, s->incList.p, cfa, cfb, jfa, jfb, heavy, s->longBodies.p);
			S2B_LAUNCH(w, s2bSortLongIncidenceKernel, 64, 256, 0, s->longBodies.p, s->adjStart.p, s->adj.p, s->itemBodies.p, s->itemVal.p,
					   s->incWork.p, s->incList.p, cfa, cfb, jfa, jfb);
			if (contactCount > 0)
			{
				S2B_CHECK(cudaMemsetAsync(s->lastTouch.p, 0, sizeof(int) * (size_t)contactCount, st));
				S2B_LAUNCH(w, s2bLastTouchKernel, gridFor(bodyCap, 256), 256, 0, bodyCap, s->adjStart.p, s->incList.p, s->lastTouch.p);
			}
		}
	}
	else
	{
		if (pl.needInc)
		{
			S2B_CHECK(cudaMemsetAsync(s->adjStart.p, 0, sizeof(int) * ((size_t)bodyCap + 2), st));
		}
		S2B_CHECK(cudaMemsetAsync(s->heavyBodies.p, 0, sizeof(int), st));
		// no constraints at all: bodies still integrate
		pl.host.groups = 0;
		pl.host.cOff.assign(S2B_MAX_COLORS + 2, 0);
		pl.host.jOff.assign(S2B_MAX_COLORS + 2, 0);
		S2B_CHECK(cudaMemsetAsync(s->cGroupOff.p, 0, sizeof(int) * (S2B_MAX_COLORS + 2), st));
		S2B_CHECK(cudaMemsetAsync(s->jGroupOff.p, 0, sizeof(int) * (S2B_MAX_COLORS + 2), st));
		s->hostContacts = s->hostJoints = s->hostGroups = 0;
		s->hostCGroupOff = pl.host.cOff;
		s->hostJGroupOff = pl.host.jOff;
		s->hostCountsValid = true;
	}
}

// the argument block + the iteration itself (persistent kernel or launch by launch) + the work meter
static void enqueueIterate(s2bWorld* w, SolverScratch* s, SolvePlan& pl, bool capturing)
{
	cudaStream_t st = w->stream;
	int solverType = pl.solverType;
	const s2bStepContext& ctx = pl.ctx;
	VariantColumns cols = pl.cols;
	size_t nC = pl.nC, nJ = pl.nJ;
	int bodyCap = pl.bodyCap;

	SolveArgs a;
	memset(&a, 0, sizeof(a));
	a.bodies = bodyView(w);
	a.contacts = makeView(w->contacts[w->cur]);
	a.joints = jointView(w);
	a.cc.idx = s->idx.p;
	a.cc.nf = s->nf.p;
	a.cc.src = s->src.p;
	a.cc.warmP = pl.gatherWarm ? s->warmP.p : nullptr;
	a.cc.warmAnchor = pl.gatherWarm ? s->warmAnchor.p : nullptr;
	a.cc.lastTouch = (pl.gatherWarm && pl.solverType == 7 && w->fusePositions != 0 && pl.dataflow == false) ? s->lastTouch.p : nullptr;
	for (int p = 0; p < 2; ++p)
	{
		a.cc.anchor[p] = s->anchor[p].p;
		a.cc.pm[p] = s->pm[p].p;
		a.cc.lambda[p] = s->lambda[p].p;
		a.cc.r0[p] = cols.r0 ? s->r0[p].p : nullptr;
		a.cc.sep[p] = cols.sep ? s->sep[p].p : nullptr;
		a.cc.fanchor[p] = cols.sticky ? s->fanchor[p].p : nullptr;
		a.cc.tsep[p] = cols.sticky ? s->tsep[p].p : nullptr;
	}
	a.jc.head = s->jhead.p;
	a.jc.anchor = s->janchor.p;
	a.jc.mass = s->jmass.p;
	a.jc.d0ax = s->jd0ax.p;
	a.jc.lim = s->jlim.p;
	a.jc.motor = s->jmotor.p;
	a.jc.coef = s->jcoef.p;
	a.jc.pivot = s->jpivot.p;
	a.jc.imp = s->jimp.p;
	a.jc.limp = s->jlimp.p;
	a.counts = s->counts.p;
	a.ctx = ctx;
	a.gravity = w->gravity;
	a.solverType = solverType;
	a.sticky = w->sticky ? 1 : 0;

	// hertz clamps of the variant: TGS_Soft (reference src/solve_tgs_soft.c:185-186), SoftStep (src/solve_soft_step.c:216-217),
	// PGS_Soft / Jacobi (src/solve_pgs_soft.c:162-163, src/solve_jacobi.c:169-170); unused by the rigid variants
	float contactHertz = S2_MIN(s2_contactHertz, 0.25f * ctx.inv_h);
	float jointHertz = S2_MIN(s2_jointHertz, 0.125f * ctx.inv_h);
	if (solverType == 5)
	{
		jointHertz = S2_MIN(s2_jointHertz, 0.25f * ctx.inv_h);
	}
	else if (solverType == 4 || solverType == 0)
	{
		contactHertz = S2_MIN(s2_contactHertz, 0.333f * ctx.inv_h);
		jointHertz = S2_MIN(s2_jointHertz, 0.5f * ctx.inv_h);
	}
	// XPBD recomputes its inverse sub-step as 1 / h (reference src/solve_xpbd.c:399-400), not inv_dt * iterations
	a.xpbdInvH = ctx.h != 0.0f ? 1.0f / ctx.h : 0.0f;
	a.contactHertz = contactHertz;
	a.jointHertz = jointHertz;
	a.softDynamic = makeSoft(ctx.h, contactHertz, 10.0f);
	a.softStatic = makeSoft(ctx.h, 2.0f * contactHertz, 10.0f);
	a.softJoint = makeSoft(ctx.h, jointHertz, 10.0f);

	PassPtrs pp = {s->jointSlots.p, s->jPerm.p};
	a.cGroupOff = s->cGroupOff.p;
	a.jGroupOff = s->jGroupOff.p;
	a.incStart = pl.gatherWarm ? s->adjStart.p : nullptr;
	a.incList = pl.gatherWarm ? s->incList.p : nullptr;
	// hub bodies: with regions the list drives their body passes (every variant); without, only the block-wide gather
	a.heavyBodies = (pl.regions > 0 || (pl.gatherWarm && pl.maxItems > 0 && pl.usePersistent)) ? s->heavyBodies.p : nullptr;
	a.regions = pl.regions;
	a.bodyLocal = (pl.regions > 0 && pl.solverType == 7 && pl.gatherWarm && w->residentRegions != 0) ? s->bodyLocal.p : nullptr;
	a.regBodyStart = s->regBodyStart.p;
	a.regBodies = s->regBodies.p;
	a.jRegOff = s->jRegOff.p;
	a.cRegOff = s->cRegOff.p;
	a.barrier = w->solveBarrier.p;
	bool stagedOverflow = w->schedule == S2B_SCHEDULE_COLOR && pl.usePersistent && pl.maxItems > 0;
	a.ovBodies = stagedOverflow ? s->ovBodies.p : nullptr;
	a.ovBodySlot = stagedOverflow ? s->ovBodySlot.p : nullptr;
	if (pl.dataflow)
	{
		S2B_CHECK(cudaMemsetAsync(s->bodyTicket.p, 0, sizeof(int) * ((size_t)bodyCap + 2), st));
		a.bodyTicket = s->bodyTicket.p;
		a.flowError = s->bodyTicket.p + bodyCap + 1;
		s->flowErrorOffset = bodyCap + 1;
		a.cFlowA = s->flow.p;
		a.cFlowB = s->flow.p + nC;
		a.jFlowA = s->flow.p + 2 * nC;
		a.jFlowB = s->flow.p + 2 * nC + nJ;
	}
	s->lastArgs = a;
	s->lastJointSlots = pp.jointSlots;
	s->lastJPerm = pp.jPerm;
	s->lastArgsValid = true;
	if (pl.usePersistent)
	{
		// wavefront tables hold CNT_GROUPS levels and no overflow group; the overflow counts are zero so the kernel
		// never indexes past them
		{
			const char* env = getenv("S2B_FLOW_SLEEP_NS");
			a.flowSleepNs = env != nullptr ? atoi(env) : 0;
		}
		if (s->traceCap > 0)
		{
			s->trace.reserve((size_t)s->traceCap, st, false);
			S2B_CHECK(cudaMemsetAsync(s->trace.p, 0, sizeof(unsigned long long), st));
			a.trace = s->trace.p;
			a.traceCap = s->traceCap;
		}
		void* args[] = {&a, &pp, &pl.program};
		if (w->solveKernelStart == nullptr)
		{
			S2B_CHECK(cudaEventCreate(&w->solveKernelStart));
			S2B_CHECK(cudaEventCreate(&w->solveKernelEnd));
		}
		// (inside a capture the time stamps become external event-record nodes so that they are taken on every replay)
		unsigned evFlags = capturing ? cudaEventRecordExternal : cudaEventRecordDefault;
		S2B_CHECK(cudaEventRecordWithFlags(w->solveKernelStart, st, evFlags));
		S2B_CHECK(cudaLaunchCooperativeKernel(s2bPersistentKernel(solverType), dim3(pl.grid), dim3(pl.threads), args, S2B_DYN_SHARED_BYTES, st));
		S2B_CHECK(cudaEventRecordWithFlags(w->solveKernelEnd, st, evFlags));
		w->solveKernelTimed = true;
		w->kernelLaunches += 1;
	}
	else
	{
		runProgramLaunchByLaunch(w, a, pp, pl.program, pl.host, pl.hostNJ, pl.hostNC);
		w->solveKernelTimed = false;
	}

	// work meter: constraint-iterations of this step = (contact constraints + joints) x solve passes (SURVEY §8d)
	{
		w->dWork.reserve(4, st, true);
		S2B_LAUNCH(w, s2bMeterWork, 1, 1, 0, s->counts.p, pl.countedPasses, w->dWork.p);
	}
}

void s2bSolve(s2bWorld* w, int solverType, const s2bStepContext* ctxIn)
{
	SolverScratch* s = s2bGetSolverScratch(w);
	cudaStream_t st = w->stream;
	s2bStepContext ctx = *ctxIn;

	if (solverType < 0 || solverType > 9)
	{
		fprintf(stderr, "solver2d-b200: solver type %d is not implemented on the device — there is no CPU fallback\n", solverType);
		abort();
	}
	if (solverType == 9 && (ctx.iterations == 0 || ctx.dt == 0.0f))
	{
		return; // s2Solve_XPBD leaves early (reference src/solve_xpbd.c:345-353)
	}
	// ---- CUDA graph of the stage ----
	// A steady scene runs the SAME ~40 launches with the SAME arguments every step (counts live in device memory). The
	// second consecutive step with an unchanged signature is captured into a graph; after that the stage is one
	// cudaGraphLaunch until the signature changes (a contact table rebuilt by the pair pass, a re-allocation, other step
	// parameters). S2B_GRAPH=0 disables it.
	bool graphable = w->schedule == S2B_SCHEDULE_COLOR && w->persistent != 0 && w->coopSupported != 0 && s->graphDisabled == false &&
					 s->traceCap == 0 && w->contactCount + w->jointCap > 0 && w->useGraph != 0;
	std::vector<unsigned char> sig;
	if (graphable)
	{
		auto put = [&sig](const void* ptr, size_t n) {
			const unsigned char* b = (const unsigned char*)ptr;
			sig.insert(sig.end(), b, b + n);
		};
		unsigned long long epoch = s2bAllocEpoch();
		int ints[] = {solverType,	 w->contactCount, w->jointCap, w->bodyCap,		  w->cur,
					  w->maxColors, w->gatherWarm,	  w->dataflow, w->sticky ? 1 : 0, w->useRegions * 256 + w->regionCutLimit};
		put(&ctx, sizeof(ctx));
		put(ints, sizeof(ints));
		put(&epoch, sizeof(epoch));
		put(&w->contactTableVersion, sizeof(w->contactTableVersion));
		put(&w->scheduleEpoch, sizeof(w->scheduleEpoch));
		put(&w->gravity, sizeof(w->gravity));
		if (s->graphExec != nullptr && sig == s->graphSig)
		{
			if (s->scheduleSig != sig)
			{
				// the schedule buffers were last built for another configuration (a solve with other settings in between)
				int one = 1;
				S2B_CHECK(cudaMemcpyAsync(w->schedDirty.p, &one, sizeof(int), cudaMemcpyHostToDevice, st));
				s->scheduleSig = sig;
			}
			S2B_CHECK(cudaGraphLaunch(s->graphExec, st));
			s->stepsSinceEager += 1;
			w->kernelLaunches += s->graphLaunches;
			w->solveKernelTimed = true;
			s->hostCountsValid = false;
			s->graphReplays += 1;
			return;
		}
	}
	if (graphable && s->graphExec != nullptr && getenv("S2B_GRAPH_DEBUG") != nullptr)
	{
		// which part of the signature moved? layout: ctx | 10 ints | epoch | table version | schedule epoch | gravity
		size_t n = std::min(sig.size(), s->graphSig.size());
		for (size_t k = 0; k < n; ++k)
		{
			if (sig[k] != s->graphSig[k])
			{
				fprintf(stderr, "solver2d-b200: graph signature changed at byte %zu (ctx %zu B, ints from %zu, epoch at %zu)\n", k, sizeof(ctx),
						sizeof(ctx), sizeof(ctx) + 10 * sizeof(int));
				break;
			}
		}
	}

	SolvePlan pl;
	pl.solverType = solverType;
	pl.ctx = ctx;
	planSolve(w, s, pl);
	if (graphable)
	{
		// planSolve may have (re)allocated: the signature carries the allocation epoch
		unsigned long long epoch = s2bAllocEpoch();
		memcpy(sig.data() + sizeof(ctx) + 10 * sizeof(int), &epoch, sizeof(epoch));
	}

	bool capturing = graphable && sig == s->graphCandidate;
	int launchesBefore = w->kernelLaunches;
	s->graphCandidate = sig;
	s->scheduleSig = sig;
	if (capturing == false)
	{
		// (no gate in front of this rebuild: the host says how quiet the scene has been — every byte 0 or 0x7F)
		S2B_CHECK(cudaMemsetAsync(w->schedDirty.p + 3, s->stepsSinceEager >= S2B_KEMPE_QUIET_STEPS ? 0x7F : 0, sizeof(int), st));
		s->stepsSinceEager = 0;
		enqueueSchedule(w, s, pl);
		if (w->useRegions == 1 && pl.regions > 0)
		{
			S2B_CHECK(cudaMemcpyAsync(w->hostMail + MAIL_REGIONS_ON, s->counts.p + CNT_REGIONS_ON, sizeof(int), cudaMemcpyDeviceToHost, st));
			s->regionVerdictPending = true;
		}
		enqueueIterate(w, s, pl, false);
		return;
	}
	s->stepsSinceEager += 1;

	// ---- build the graph: gate -> IF (gather + schedule) -> iterate ----
	if (s->graphExec != nullptr)
	{
		cudaGraphExecDestroy(s->graphExec);
		s->graphExec = nullptr;
	}
	w->capturing = true;
	cudaGraph_t graph = nullptr;
	cudaError_t err = cudaGraphCreate(&graph, 0);
	cudaGraphNode_t gateNode = nullptr, ifNode = nullptr;
	cudaGraph_t body = nullptr;
	bool conditional = getenv("S2B_GRAPH_CONDITIONAL") == nullptr || atoi(getenv("S2B_GRAPH_CONDITIONAL")) != 0;
	if (err == cudaSuccess && conditional)
	{
		cudaGraphConditionalHandle handle;
		err = cudaGraphConditionalHandleCreate(&handle, graph, 1, cudaGraphCondAssignDefault);
		if (err == cudaSuccess)
		{
			cudaKernelNodeParams kp = {};
			int* dirty = w->schedDirty.p;
			void* args[] = {&handle, &dirty};
			kp.func = (void*)s2bScheduleGate;
			kp.gridDim = dim3(1);
			kp.blockDim = dim3(1);
			kp.kernelParams = args;
			err = cudaGraphAddKernelNode(&gateNode, graph, nullptr, 0, &kp);
		}
		if (err == cudaSuccess)
		{
			cudaGraphNodeParams np = {cudaGraphNodeTypeConditional};
			np.conditional.handle = handle;
			np.conditional.type = cudaGraphCondTypeIf;
			np.conditional.size = 1;
			err = cudaGraphAddNode(&ifNode, graph, &gateNode, 1, &np);
			if (err == cudaSuccess)
			{
				body = np.conditional.phGraph_out[0];
			}
		}
		if (err == cudaSuccess)
		{
			err = cudaStreamBeginCaptureToGraph(st, body, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal);
			if (err == cudaSuccess)
			{
				enqueueSchedule(w, s, pl);
				cudaGraph_t out = nullptr;
				err = cudaStreamEndCapture(st, &out);
			}
		}
		if (err == cudaSuccess)
		{
			err = cudaStreamBeginCaptureToGraph(st, graph, &ifNode, nullptr, 1, cudaStreamCaptureModeThreadLocal);
			if (err == cudaSuccess)
			{
				enqueueIterate(w, s, pl, true);
				cudaGraph_t out = nullptr;
				err = cudaStreamEndCapture(st, &out);
			}
		}
		w->kernelLaunches += 1; // the gate
	}
	else if (err == cudaSuccess)
	{
		// plain capture of the whole stage (S2B_GRAPH_CONDITIONAL=0): the schedule is rebuilt on every replay
		err = cudaStreamBeginCaptureToGraph(st, graph, nullptr, nullptr, 0, cudaStreamCaptureModeThreadLocal);
		if (err == cudaSuccess)
		{
			enqueueSchedule(w, s, pl);
			enqueueIterate(w, s, pl, true);
			cudaGraph_t out = nullptr;
			err = cudaStreamEndCapture(st, &out);
		}
	}
	w->capturing = false;
	if (err == cudaSuccess)
	{
		err = cudaGraphInstantiate(&s->graphExec, graph, 0);
	}
	if (graph != nullptr)
	{
		cudaGraphDestroy(graph);
	}
	if (err != cudaSuccess || s->graphExec == nullptr)
	{
		// not possible on this driver: nothing ran, so run this step eagerly and stop trying
		(void)cudaGetLastError();
		fprintf(stderr, "solver2d-b200: building the CUDA graph of the solver stage failed (%s); continuing without graphs\n",
				cudaGetErrorString(err));
		s->graphExec = nullptr;
		s->graphDisabled = true;
		s->graphCandidate.clear();
		w->kernelLaunches = launchesBefore;
		s2bSolve(w, solverType, ctxIn);
		return;
	}
	s->graphSig = sig;
	s->graphLaunches = w->kernelLaunches - launchesBefore;
	s->graphCaptures += 1;
	// the schedule of the previous (eager) step is still valid unless the flag says otherwise: the gate decides
	S2B_CHECK(cudaGraphLaunch(s->graphExec, st));
}

extern "C" void s2b_get_work(s2bWorld* w, uint64_t out[2], int reset)
{
	S2B_CHECK(cudaSetDevice(w->device));
	S2B_CHECK(cudaStreamSynchronize(w->stream));
	out[0] = out[1] = 0;
	if (w->dWork.p != nullptr)
	{
		S2B_CHECK(cudaMemcpy(out, w->dWork.p, sizeof(uint64_t) * 2, cudaMemcpyDeviceToHost));
		if (reset)
		{
			S2B_CHECK(cudaMemset(w->dWork.p, 0, sizeof(uint64_t) * 2));
		}
	}
}

extern "C" float s2b_last_solve_kernel_ms(s2bWorld* w)
{
	S2B_CHECK(cudaSetDevice(w->device));
	if (w->solveKernelTimed == false)
	{
		return 0.0f;
	}
	S2B_CHECK(cudaEventSynchronize(w->solveKernelEnd));
	float ms = 0.0f;
	S2B_CHECK(cudaEventElapsedTime(&ms, w->solveKernelStart, w->solveKernelEnd));
	return ms;
}

extern "C" int s2b_download_solve_order(s2bWorld* w, int32_t* items, int maxItems, int32_t* groupSizes, int maxGroups,
										int32_t* groupCount)
{
	S2B_CHECK(cudaSetDevice(w->device));
	SolverScratch* s = s2bGetSolverScratch(w);
	S2B_CHECK(cudaStreamSynchronize(w->stream));
	int counts[CNT_SIZE];
	S2B_CHECK(cudaMemcpy(counts, s->counts.p, sizeof(counts), cudaMemcpyDeviceToHost));
	int nC = counts[CNT_CONTACTS], nJ = counts[CNT_JOINTS], groups = counts[CNT_GROUPS];
	bool wavefront = w->schedule == S2B_SCHEDULE_WAVEFRONT;
	int regions = (wavefront || counts[CNT_REGIONS_ON] == 0) ? 0 : s->regions;
	int tableLen = (wavefront ? groups : S2B_MAX_COLORS) + 2;
	std::vector<int> cOff((size_t)tableLen), jOff((size_t)tableLen), src((size_t)std::max(nC, 1)), jPerm((size_t)std::max(nJ, 1)),
		jointSlots((size_t)std::max(nJ, 1));
	S2B_CHECK(cudaMemcpy(cOff.data(), s->cGroupOff.p, sizeof(int) * (size_t)tableLen, cudaMemcpyDeviceToHost));
	S2B_CHECK(cudaMemcpy(jOff.data(), s->jGroupOff.p, sizeof(int) * (size_t)tableLen, cudaMemcpyDeviceToHost));
	std::vector<int> cReg((size_t)std::max(regions, 1) * S2B_REG_STRIDE), jReg((size_t)std::max(regions, 1) * S2B_REG_STRIDE);
	if (regions > 0)
	{
		S2B_CHECK(cudaMemcpy(cReg.data(), s->cRegOff.p, sizeof(int) * (size_t)regions * S2B_REG_STRIDE, cudaMemcpyDeviceToHost));
		S2B_CHECK(cudaMemcpy(jReg.data(), s->jRegOff.p, sizeof(int) * (size_t)regions * S2B_REG_STRIDE, cudaMemcpyDeviceToHost));
	}
	if (nC > 0)
	{
		S2B_CHECK(cudaMemcpy(src.data(), s->src.p, sizeof(int) * (size_t)nC, cudaMemcpyDeviceToHost));
	}
	if (nJ > 0)
	{
		S2B_CHECK(cudaMemcpy(jPerm.data(), s->jPerm.p, sizeof(int) * (size_t)nJ, cudaMemcpyDeviceToHost));
		S2B_CHECK(cudaMemcpy(jointSlots.data(), s->jointSlots.p, sizeof(int) * (size_t)nJ, cudaMemcpyDeviceToHost));
	}
	// a group = joints [jb, je) then contacts [cb, ce) of the two streams. Serial order of the region-local schedule
	// (persistent.cuh): region by region, colour by colour inside a region; then the device-wide groups (cut colours /
	// colours / wavefront levels); the serial overflow group (colour schedule only, table index S2B_MAX_COLORS) comes last.
	int written = 0, groupsOut = 0;
	auto emit = [&](int jb, int je, int cb, int ce) {
		int size = 0;
		for (int t = jb; t < je; ++t, ++size)
		{
			if (written < maxItems && items != nullptr)
			{
				items[written] = -1 - jointSlots[(size_t)jPerm[(size_t)t]];
			}
			written += 1;
		}
		for (int t = cb; t < ce; ++t, ++size)
		{
			if (written < maxItems && items != nullptr)
			{
				items[written] = src[(size_t)t];
			}
			written += 1;
		}
		if (size > 0)
		{
			if (groupSizes != nullptr && groupsOut < maxGroups)
			{
				groupSizes[groupsOut] = size;
			}
			groupsOut += 1;
		}
	};
	for (int r = 0; r < regions; ++r)
	{
		for (int c = 0; c < S2B_MAX_COLORS; ++c)
		{
			size_t e = (size_t)r * S2B_REG_STRIDE + c;
			emit(jReg[e], jReg[e + 1], cReg[e], cReg[e + 1]);
		}
	}
	for (int g = 0; g < groups; ++g)
	{
		emit(jOff[(size_t)g], jOff[(size_t)g + 1], cOff[(size_t)g], cOff[(size_t)g + 1]);
	}
	if (wavefront == false)
	{
		emit(jOff[S2B_MAX_COLORS], jOff[S2B_MAX_COLORS + 1], cOff[S2B_MAX_COLORS], cOff[S2B_MAX_COLORS + 1]);
	}
	if (groupCount != nullptr)
	{
		*groupCount = groupsOut;
	}
	return written;
}

// Islands of the constraint graph of the last solve (see s2bIslandHookKernel): label per body slot = smallest body slot of
// its island (a body without constraints, or a static body, is an island of its own); -1 for free slots.
extern "C" int s2b_download_islands(s2bWorld* w, int32_t* islandOfBody, int capacity)
{
	S2B_CHECK(cudaSetDevice(w->device));
	S2bEpochFreeze freeze; // scratch of this query is not referenced by the solver's graph
	SolverScratch* s = s2bGetSolverScratch(w);
	cudaStream_t st = w->stream;
	int bodyCap = w->bodyCap;
	if (bodyCap <= 0 || s->counts.p == nullptr)
	{
		return 0;
	}
	int maxItems = w->contactCount + w->jointCap;
	DevArray<int> parent, label, size;
	parent.reserve((size_t)bodyCap + 1, st, false);
	label.reserve((size_t)bodyCap + 1, st, false);
	size.reserve((size_t)bodyCap + 1, st, false, true);
	S2B_LAUNCH(w, s2bIslandInitKernel, gridFor(bodyCap, 256), 256, 0, bodyCap, parent.p);
	if (maxItems > 0 && s->itemBodies.p != nullptr)
	{
		S2B_LAUNCH(w, s2bIslandHookKernel, gridFor(maxItems, 256), 256, 0, s->counts.p, s->itemBodies.p, parent.p);
	}
	S2B_LAUNCH(w, s2bIslandFlattenKernel, gridFor(bodyCap, 256), 256, 0, bodyView(w), parent.p, label.p, size.p);
	std::vector<int> host((size_t)bodyCap);
	std::vector<uint8_t> flags((size_t)bodyCap);
	S2B_CHECK(cudaMemcpyAsync(host.data(), label.p, sizeof(int) * (size_t)bodyCap, cudaMemcpyDeviceToHost, st));
	S2B_CHECK(cudaMemcpyAsync(flags.data(), w->bFlags.p, (size_t)bodyCap, cudaMemcpyDeviceToHost, st));
	S2B_CHECK(cudaStreamSynchronize(st));
	parent.release();
	label.release();
	size.release();
	int islands = 0;
	for (int i = 0; i < bodyCap; ++i)
	{
		bool valid = (flags[(size_t)i] & S2B_BODY_VALID) != 0;
		if (valid && host[(size_t)i] == i)
		{
			islands += 1;
		}
		if (i < capacity && islandOfBody != nullptr)
		{
			islandOfBody[i] = valid ? host[(size_t)i] : -1;
		}
	}
	return islands;
}

extern "C" void s2b_get_counters(s2bWorld* w, s2bCounters* out)
{
	S2B_CHECK(cudaSetDevice(w->device));
	S2B_CHECK(cudaStreamSynchronize(w->stream));
	memset(out, 0, sizeof(*out));
	out->bodyCapacity = w->bodyCap;
	out->shapeCapacity = w->shapeCap;
	out->jointCapacity = w->jointCap;
	out->contactCount = w->contactCount;
	if (w->scratch != nullptr && w->scratch->counts.p != nullptr)
	{
		int counts[CNT_SIZE];
		S2B_CHECK(cudaMemcpy(counts, w->scratch->counts.p, sizeof(counts), cudaMemcpyDeviceToHost));
		out->constraintCount = counts[CNT_CONTACTS];
		out->jointCount = counts[CNT_JOINTS];
		// colours of the constraint graph under the colour schedule, levels under the wavefront schedule
		out->groupCount = w->schedule == S2B_SCHEDULE_COLOR ? counts[CNT_COLORS] : counts[CNT_GROUPS];
		// (cut statistics are reported whenever regions were tried; regionCount says whether the solve order used them)
		out->cutGroupCount = w->scratch->regions > 0 ? counts[CNT_CUT_COLORS] : 0;
		out->cutCount = w->scratch->regions > 0 ? counts[CNT_CUT] : 0;
		out->regionCount = counts[CNT_REGIONS_ON] != 0 ? w->scratch->regions : 0;
		out->overflowCount = counts[CNT_OVERFLOW_C] + counts[CNT_OVERFLOW_J];
		if (w->scratch->kempeState.p != nullptr)
		{
			int ks[4];
			S2B_CHECK(cudaMemcpy(ks, w->scratch->kempeState.p, sizeof(ks), cudaMemcpyDeviceToHost));
			out->recolouredCount = ks[KS_FIXED];
		}
		if (w->scratch->bodyTicket.p != nullptr && w->scratch->flowErrorOffset > 0)
		{
			int flag = 0;
			S2B_CHECK(cudaMemcpy(&flag, w->scratch->bodyTicket.p + w->scratch->flowErrorOffset, sizeof(int), cudaMemcpyDeviceToHost));
			if (flag != 0)
			{
				fprintf(stderr, "solver2d-b200: a ticketed solver pass ran into its spin limit (internal error)\n");
				abort();
			}
		}
	}
	out->treeHeight = w->treeHeight;
	out->largeLeafCount = w->largeLeafCount;
	out->pairRebuildCount = w->pairRebuildCount;
	out->movedCount = w->hostMail[MAIL_MOVED];
	out->pairPassCount = w->pairPassCount;
	out->kernelLaunches = w->kernelLaunches;
	out->graphReplays = w->scratch != nullptr ? w->scratch->graphReplays : 0;
	out->graphCaptures = w->scratch != nullptr ? w->scratch->graphCaptures : 0;
}

extern "C" void s2b_set_solve_trace(s2bWorld* w, int capacity)
{
	s2bGetSolverScratch(w)->traceCap = capacity > 0 ? capacity + 1 : 0;
}

extern "C" int s2b_get_solve_trace(s2bWorld* w, uint64_t* out, int maxEntries)
{
	S2B_CHECK(cudaSetDevice(w->device));
	S2B_CHECK(cudaStreamSynchronize(w->stream));
	SolverScratch* s = s2bGetSolverScratch(w);
	if (s->trace.p == nullptr || s->traceCap == 0)
	{
		return 0;
	}
	unsigned long long n = 0;
	S2B_CHECK(cudaMemcpy(&n, s->trace.p, sizeof(n), cudaMemcpyDeviceToHost));
	int count = (int)std::min<unsigned long long>(n, (unsigned long long)maxEntries);
	if (count > 0)
	{
		S2B_CHECK(cudaMemcpy(out, s->trace.p + 1, sizeof(uint64_t) * (size_t)count, cudaMemcpyDeviceToHost));
	}
	return count;
}

extern "C" void s2b_flush_l2(s2bWorld* w);

// Roofline probe of THE hot kernel in isolation: the TGS_Soft relax pass over the largest colour of the current constraint
// set, one launch per repetition, L2 evicted before every launch so that the constraint stream and the bodies come from
// HBM. The preceding solve is run launch by launch to have the group table on the host; the world's state advances by
// that one solver stage plus `reps` extra relax passes of one colour (a probe, not a simulation step).
extern "C" float s2b_time_color_kernel(s2bWorld* w, const s2bStepContext* context, int reps, int* constraints)
{
	S2B_CHECK(cudaSetDevice(w->device));
	if (constraints)
	{
		*constraints = 0;
	}
	int persistentBefore = w->persistent;
	w->persistent = 0;
	s2bSolve(w, 7, context);
	w->persistent = persistentBefore;
	SolverScratch* s = s2bGetSolverScratch(w);
	if (s->lastArgsValid == false || s->hostCountsValid == false || s->hostGroups == 0)
	{
		return 0.0f;
	}
	int best = 0, bestCount = 0;
	for (int g = 0; g < s->hostGroups; ++g)
	{
		int n = s->hostCGroupOff[g + 1] - s->hostCGroupOff[g];
		if (n > bestCount)
		{
			bestCount = n;
			best = g;
		}
	}
	if (bestCount == 0)
	{
		return 0.0f;
	}
	int cb = s->hostCGroupOff[best], ce = s->hostCGroupOff[best + 1];
	SolveArgs a = s->lastArgs;
	// S2B_COLOR_KERNEL=bulk selects the version that stages the stream through shared memory with TMA bulk copies; measured
	// slightly SLOWER than ordinary coalesced loads (5.13 vs 5.29 TB/s at 1.5 M constraints), so it is not the default
	const char* which = getenv("S2B_COLOR_KERNEL");
	bool bulk = which != nullptr && strcmp(which, "bulk") == 0;
	// (the bulk version may stage up to two rows past the colour; the stream columns are reserved with two spare rows for that)
	cudaEvent_t e0, e1;
	S2B_CHECK(cudaEventCreate(&e0));
	S2B_CHECK(cudaEventCreate(&e1));
	float total = 0.0f;
	for (int r = 0; r < reps + 2; ++r)
	{
		s2b_flush_l2(w);
		S2B_CHECK(cudaEventRecord(e0, w->stream));
		if (bulk)
		{
			S2B_LAUNCH(w, s2bTgsSoftColorKernelBulk, gridFor(bestCount, S2B_BULK_BLOCK), S2B_BULK_BLOCK, 0, a, cb, ce, 0);
		}
		else
		{
			S2B_LAUNCH(w, s2bTgsSoftColorKernel, gridFor(bestCount, S2B_BLOCK), S2B_BLOCK, 0, a, cb, ce, 0);
		}
		S2B_CHECK(cudaEventRecord(e1, w->stream));
		S2B_CHECK(cudaEventSynchronize(e1));
		float ms = 0.0f;
		S2B_CHECK(cudaEventElapsedTime(&ms, e0, e1));
		if (r >= 2)
		{
			total += ms; // the first two repetitions warm the instruction cache and the TLB
		}
	}
	cudaEventDestroy(e0);
	cudaEventDestroy(e1);
	if (constraints)
	{
		*constraints = bestCount;
	}
	return reps > 0 ? total / (float)reps : 0.0f;
}
