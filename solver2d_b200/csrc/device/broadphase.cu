// solver2d-b200 — stages 1+2 (and the destroy half of stage 3) of s2World_Step on the device.
//
// Replaces s2UpdateBroadPhasePairs / s2FindPairs / s2PairQueryCallback (reference src/broad_phase.c:166-367), the three
// incrementally-updated dynamic AABB trees (src/dynamic_tree.c) with their rebuild (broad_phase.c:381-385), the pair
// hash set (src/table.c) and the fat-AABB overlap test + s2DestroyContact of world.c:149-166.
//
// B200-first design instead of a port of the pointer-chasing tree:
//   * the proxies are sorted in Morton order, fully in parallel, only on steps where some proxy left its fat AABB (or the
//     host created/destroyed something); a shallow 16-wide hierarchy over that order (node i of level l covers sorted
//     leaves [i*16^l, (i+1)*16^l)) is refitted every pass, and the few scene-sized proxies are kept out of it in a short
//     list that every query tests directly;
//   * one thread per *moved* proxy walks the hierarchy and applies the reference's pair rules (both-moved de-duplication by
//     proxy key, body-type rules of the three-tree query, existing pair, same body, filter, joint override, shape-type
//     table) — so the set of created contacts equals the reference's;
//   * existing contacts whose fat AABBs stopped overlapping are dropped, survivors and new pairs are merged by a radix
//     sort on the 64-bit shape-pair key and all contact columns are gathered into the other column set.
// The contact table is therefore always sorted by pair key: the device's natural (wavefront) constraint order.
#include "s2b_internal.cuh"

#include <cub/cub.cuh>
#include <thrust/iterator/counting_iterator.h>

#include <algorithm>

struct BroadScratch
{
	DevArray<int> validFlag;	   // per shape slot
	DevArray<int> leafShape;	   // compacted valid shapes
	DevArray<unsigned> mortonIn, mortonOut;
	DevArray<int> leafIn, leafOut; // sorted leaf -> index into leafShape
	DevArray<int> sortedShape;	   // sorted leaf -> shape slot (leafShape[leafOut[k]], composed at the rebuild)
	DevArray<int> counters;		   // BC_*
	DevArray<int> boundsBits;	   // 8 ordered-int encoded floats: box centres min.x min.y max.x max.y, boxes min.x min.y max.x max.y
	DevArray<float4> nodeBox;	   // sorted leaf boxes [0, n), then the levels of the hierarchy (s2bLevels)
	DevArray<int> movedShapes;	   // shapes of the moved proxies, in Morton order
	DevArray<int> movedFlag;
	DevArray<int> largeShapes;	   // shapes of moved proxies with scene-sized boxes
	DevArray<unsigned long long> newKey;
	DevArray<int2> newShapes;
	DevArray<int> keepFlag, keepSlots;
	DevArray<unsigned long long> mergeKeyIn, mergeKeyOut;
	DevArray<int> mergeSrcIn, mergeSrcOut;
	DevArray<char> cubTemp;
	int newPairCap = 0;
	// the hierarchy of the last pass: while no shape was created, destroyed or re-uploaded its TOPOLOGY is reused and only
	// the boxes are refitted (boxes drift a little per step; a periodic rebuild keeps the tree tight)
	bool treeValid = false;
	int treeShapeCap = 0;
	int treeReuses = 0;
	// open-addressing hash set of the shape-pair keys of the current contact table ("does this pair already exist?")
	DevArray<unsigned long long> pairHash;
	unsigned long long hashMask = 0;
	unsigned long long hashVersion = ~0ull; // contact table version the set was built from
	// pair search started behind the previous step (s2bPrefetchPairSearch)
	bool prefetched = false;	   // a search is in flight / finished and not consumed yet
	bool lastPassRan = false;	   // the last pass found moved proxies (the scene is in motion)
	bool searchTimed = false;
	unsigned long long prefetchEpoch = 0, searchedVersion = 0;
	int searchedCount = 0;
	size_t prefetchTempBytes = 0;
	cudaEvent_t evSearch[2] = {nullptr, nullptr};
	cudaEvent_t searchDone = nullptr;
};

#define S2B_TREE_REUSE_LIMIT 16

static BroadScratch* getBroad(s2bWorld* w)
{
	if (w->broad == nullptr)
	{
		w->broad = new BroadScratch();
	}
	return w->broad;
}

void s2bFreeBroadScratch(s2bWorld* w)
{
	BroadScratch* b = w->broad;
	if (b == nullptr)
	{
		return;
	}
	b->validFlag.release();
	b->leafShape.release();
	b->mortonIn.release();
	b->mortonOut.release();
	b->leafIn.release();
	b->leafOut.release();
	b->sortedShape.release();
	b->counters.release();
	b->boundsBits.release();
	b->nodeBox.release();
	b->movedShapes.release();
	b->movedFlag.release();
	b->newKey.release();
	b->newShapes.release();
	b->keepFlag.release();
	b->keepSlots.release();
	b->mergeKeyIn.release();
	b->mergeKeyOut.release();
	b->mergeSrcIn.release();
	b->mergeSrcOut.release();
	b->cubTemp.release();
	b->largeShapes.release();
	b->pairHash.release();
	for (int i = 0; i < 2; ++i)
	{
		if (b->evSearch[i] != nullptr)
		{
			cudaEventDestroy(b->evSearch[i]);
		}
	}
	if (b->searchDone != nullptr)
	{
		cudaEventDestroy(b->searchDone);
	}
	delete b;
	w->broad = nullptr;
}

// BC_LEAVES and BC_LARGE_LEAVES describe the sorted order and live as long as it is reused; the others are cleared by
// every pass
enum
{
	BC_LEAVES = 0,
	BC_LARGE_LEAVES = 1, // scene-sized leaves kept out of the hierarchy at the last rebuild (may exceed the list's capacity)
	BC_NEW_PAIRS = 2,
	BC_KEPT = 3,
	BC_MOVED = 4,
	BC_HEIGHT = 5,
	BC_LARGE = 6,		// moved proxies handled by the leaf-side query
	BC_REFIT_DONE = 7,	// blocks of s2bRefit that finished their part
	BC_SIZE = 8
};

// ---------------------------------------------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------------------------------------------

__device__ __forceinline__ int s2bFloatToOrdered(float f)
{
	int i = __float_as_int(f);
	return i >= 0 ? i : i ^ 0x7FFFFFFF;
}

__device__ __forceinline__ float s2bOrderedToFloat(int i)
{
	return __int_as_float(i >= 0 ? i : i ^ 0x7FFFFFFF);
}

__device__ __forceinline__ unsigned s2bExpandBits(unsigned v)
{
	// 16 bits -> every other bit of 32
	v &= 0xFFFFu;
	v = (v | (v << 8)) & 0x00FF00FFu;
	v = (v | (v << 4)) & 0x0F0F0F0Fu;
	v = (v | (v << 2)) & 0x33333333u;
	v = (v | (v << 1)) & 0x55555555u;
	return v;
}

__device__ __forceinline__ bool s2bBoxesOverlap(float4 a, float4 b)
{
	// s2AABB_Overlaps (reference include/solver2d/aabb.h:111-123): closed test
	float d1x = b.x - a.z, d1y = b.y - a.w;
	float d2x = a.x - b.z, d2y = a.y - b.w;
	if (d1x > 0.0f || d1y > 0.0f)
	{
		return false;
	}
	if (d2x > 0.0f || d2y > 0.0f)
	{
		return false;
	}
	return true;
}

// s2ShouldShapesCollide (reference src/contact.h:70-79)
__device__ __forceinline__ bool s2bShouldShapesCollide(int4 fa, int4 fb)
{
	if (fa.z == fb.z && fa.z != 0)
	{
		return fa.z > 0;
	}
	return ((unsigned)fa.y & (unsigned)fb.x) != 0 && ((unsigned)fa.x & (unsigned)fb.y) != 0;
}

// joints with collideConnected == false override collision (replaces the joint-list walk of s2ShouldBodiesCollide,
// reference src/body.c:386-417) — binary search in the sorted body-pair keys uploaded by the host
__device__ __forceinline__ bool s2bJointOverride(const unsigned long long* keys, int count, int bodyA, int bodyB)
{
	if (count == 0)
	{
		return false;
	}
	unsigned long long lo = (unsigned long long)(bodyA < bodyB ? bodyA : bodyB);
	unsigned long long hi = (unsigned long long)(bodyA < bodyB ? bodyB : bodyA);
	unsigned long long key = (lo << 32) | hi;
	int l = 0, r = count;
	while (l < r)
	{
		int m = (l + r) >> 1;
		if (keys[m] < key)
		{
			l = m + 1;
		}
		else
		{
			r = m;
		}
	}
	return l < count && keys[l] == key;
}

// pair-key hash set (replaces an 18-step binary search per candidate pair by one or two probes)
__device__ __forceinline__ unsigned long long s2bMix64(unsigned long long x)
{
	x ^= x >> 33;
	x *= 0xff51afd7ed558ccdull;
	x ^= x >> 33;
	x *= 0xc4ceb9fe1a85ec53ull;
	x ^= x >> 33;
	return x;
}

__global__ void s2bBuildPairHash(const unsigned long long* keys, int count, unsigned long long* table, unsigned long long mask)
{
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= count)
	{
		return;
	}
	unsigned long long key = keys[i];
	unsigned long long slot = s2bMix64(key) & mask;
	for (;;)
	{
		unsigned long long prev = atomicCAS(table + slot, ~0ull, key);
		if (prev == ~0ull || prev == key)
		{
			return;
		}
		slot = (slot + 1) & mask;
	}
}

__device__ __forceinline__ bool s2bPairInHash(const unsigned long long* table, unsigned long long mask, unsigned long long key)
{
	unsigned long long slot = s2bMix64(key) & mask;
	for (;;)
	{
		unsigned long long v = table[slot];
		if (v == key)
		{
			return true;
		}
		if (v == ~0ull)
		{
			return false;
		}
		slot = (slot + 1) & mask;
	}
}

__device__ __forceinline__ bool s2bKeyExists(const unsigned long long* keys, int count, unsigned long long key)
{
	int l = 0, r = count;
	while (l < r)
	{
		int m = (l + r) >> 1;
		if (keys[m] < key)
		{
			l = m + 1;
		}
		else
		{
			r = m;
		}
	}
	return l < count && keys[l] == key;
}

// manifold function table of the reference (src/contact.c:139-154): is (typeA, typeB) a primary pair, a flipped pair,
// or not collidable at all (segment vs segment)?
// returns 0 = none, 1 = primary, 2 = flip
__device__ __forceinline__ int s2bPairKind(int t1, int t2)
{
	// primary pairs: (circle,circle) (capsule,circle) (capsule,capsule) (polygon,circle) (polygon,capsule)
	// (polygon,polygon) (segment,circle) (segment,capsule) (segment,polygon)
	const int CAP = S2B_SHAPE_CAPSULE, CIR = S2B_SHAPE_CIRCLE, POL = S2B_SHAPE_POLYGON, SEG = S2B_SHAPE_SEGMENT;
	if (t1 == SEG && t2 == SEG)
	{
		return 0;
	}
	bool primary = (t1 == CIR && t2 == CIR) || (t1 == CAP && t2 == CIR) || (t1 == CAP && t2 == CAP) || (t1 == POL && t2 == CIR) ||
				   (t1 == POL && t2 == CAP) || (t1 == POL && t2 == POL) || (t1 == SEG && t2 != SEG);
	return primary ? 1 : 2;
}

// ---------------------------------------------------------------------------------------------------------------
// hierarchy
// ---------------------------------------------------------------------------------------------------------------

// A fixed-fanout hierarchy over the Morton-sorted leaves: node i of level l covers sorted leaves [i*16^l, (i+1)*16^l), so
// the topology is implicit in the order and a rebuild is the sort alone. At 100 k leaves a query descends 5 levels of
// independent 16-box tests instead of the dozens of dependent levels of a binary radix tree.
#define S2B_FANOUT 16
#define S2B_MAX_LEVELS 8 // 16^8 leaves

// Leaves whose fat box is scene-sized (the pyramid's ground is 547 m wide) would make every ancestor scene-sized and drag
// every query down their chain. At a rebuild up to S2B_MAX_LARGE_LEAVES of them sort behind the hierarchy's leaves
// (sorted leaves [n - large, n)); every query tests them directly. Any beyond the capacity stay in the hierarchy. Each leaf
// is on exactly one side, so every (query, leaf) overlap is still considered exactly once.
#define S2B_MAX_LARGE_LEAVES 64

// Offsets into nodeBox and node counts of the levels over the first nh sorted leaves: level 0 (the leaves) at 0, level 1 at
// n, each next level right behind the previous one. Returns the top level: the first whose node count is <= 16 (0 when
// the leaves themselves are that few). s2bRefit and s2bFindPairs both lay the levels out with this.
__device__ __forceinline__ int s2bLevels(int n, int nh, int* offset, int* count)
{
	offset[0] = 0;
	count[0] = nh;
	int top = 0, off = n;
	while (count[top] > S2B_FANOUT && top + 1 < S2B_MAX_LEVELS)
	{
		int c = (count[top] + S2B_FANOUT - 1) / S2B_FANOUT;
		top += 1;
		offset[top] = off;
		count[top] = c;
		off += c;
	}
	return top;
}

__device__ __forceinline__ float4 s2bEmptyBox()
{
	return make_float4(3.0e38f, 3.0e38f, -3.0e38f, -3.0e38f);
}

__device__ __forceinline__ float4 s2bUnion(float4 a, float4 b)
{
	return make_float4(fminf(a.x, b.x), fminf(a.y, b.y), fmaxf(a.z, b.z), fmaxf(a.w, b.w));
}

// union over the 16 lanes of each half warp (every lane of the warp has to call this)
__device__ __forceinline__ float4 s2bUnion16(float4 box)
{
	for (int o = S2B_FANOUT / 2; o > 0; o >>= 1)
	{
		box.x = fminf(box.x, __shfl_xor_sync(0xFFFFFFFFu, box.x, o));
		box.y = fminf(box.y, __shfl_xor_sync(0xFFFFFFFFu, box.y, o));
		box.z = fmaxf(box.z, __shfl_xor_sync(0xFFFFFFFFu, box.z, o));
		box.w = fmaxf(box.w, __shfl_xor_sync(0xFFFFFFFFu, box.w, o));
	}
	return box;
}

__global__ void s2bFlagValidShapes(ShapeView s, int* validFlag)
{
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < s.capacity)
	{
		validFlag[i] = (s.head[i].x & S2B_ROW_VALID) ? 1 : 0;
	}
}

// bounds of the box centres (Morton quantisation) and of the boxes themselves (what counts as scene-sized)
__global__ void s2bSceneBounds(ShapeView s, const int* leafShape, const int* counters, int* boundsBits)
{
	int n = counters[BC_LEAVES];
	int k = blockIdx.x * blockDim.x + threadIdx.x;
	float c[4] = {3.0e38f, 3.0e38f, -3.0e38f, -3.0e38f};
	float4 box = s2bEmptyBox();
	if (k < n)
	{
		box = s.fat[leafShape[k]];
		float cx = 0.5f * (box.x + box.z), cy = 0.5f * (box.y + box.w);
		c[0] = c[2] = cx;
		c[1] = c[3] = cy;
	}
	float v[8] = {c[0], c[1], c[2], c[3], box.x, box.y, box.z, box.w};
	for (int o = 16; o > 0; o >>= 1)
	{
		for (int j = 0; j < 8; ++j)
		{
			float u = __shfl_xor_sync(0xFFFFFFFFu, v[j], o);
			v[j] = (j & 2) ? fmaxf(v[j], u) : fminf(v[j], u);
		}
	}
	if ((threadIdx.x & 31) == 0)
	{
		for (int j = 0; j < 8; ++j)
		{
			if (j & 2)
			{
				atomicMax(boundsBits + j, s2bFloatToOrdered(v[j]));
			}
			else
			{
				atomicMin(boundsBits + j, s2bFloatToOrdered(v[j]));
			}
		}
	}
}

__global__ void s2bMortonCodes(ShapeView s, const int* leafShape, int* counters, const int* boundsBits, unsigned* morton,
							   int* leafIndex, int capacity)
{
	int n = counters[BC_LEAVES];
	int k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= capacity)
	{
		return;
	}
	leafIndex[k] = k;
	if (k >= n)
	{
		morton[k] = 0xFFFFFFFFu; // padding sorts last (behind the large leaves: the sort is stable)
		return;
	}
	float minx = s2bOrderedToFloat(boundsBits[0]), miny = s2bOrderedToFloat(boundsBits[1]);
	float maxx = s2bOrderedToFloat(boundsBits[2]), maxy = s2bOrderedToFloat(boundsBits[3]);
	float4 f = s.fat[leafShape[k]];
	if (n >= 256)
	{
		float sceneSide = fmaxf(s2bOrderedToFloat(boundsBits[6]) - s2bOrderedToFloat(boundsBits[4]),
								s2bOrderedToFloat(boundsBits[7]) - s2bOrderedToFloat(boundsBits[5]));
		float side = fmaxf(f.z - f.x, f.w - f.y);
		if (side * 16.0f > sceneSide && atomicAdd(counters + BC_LARGE_LEAVES, 1) < S2B_MAX_LARGE_LEAVES)
		{
			morton[k] = 0xFFFFFFFFu; // ordinary codes are below 2^31
			return;
		}
	}
	float cx = 0.5f * (f.x + f.z), cy = 0.5f * (f.y + f.w);
	float ex = fmaxf(maxx - minx, 1.0e-6f), ey = fmaxf(maxy - miny, 1.0e-6f);
	float ux = fminf(fmaxf((cx - minx) / ex, 0.0f), 1.0f);
	float uy = fminf(fmaxf((cy - miny) / ey, 0.0f), 1.0f);
	unsigned qx = (unsigned)(ux * 32767.0f), qy = (unsigned)(uy * 32767.0f);
	morton[k] = (s2bExpandBits(qx) | (s2bExpandBits(qy) << 1)) & 0x7FFFFFFFu;
}

__global__ void s2bSortedShapes(const int* leafShape, const int* leafOut, const int* counters, int* sortedShape)
{
	int k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k < counters[BC_LEAVES])
	{
		sortedShape[k] = leafShape[leafOut[k]];
	}
}

// ---------------------------------------------------------------------------------------------------------------
// pair queries
// ---------------------------------------------------------------------------------------------------------------

// append `value` to list[] (length in *count) for every thread with take == true: one atomic per BLOCK, and the block's
// entries keep their thread order (every thread of the block has to call this)
__device__ __forceinline__ void s2bBlockAppend(bool take, int value, int* list, int* count)
{
	__shared__ int warpOffset[32];
	__shared__ int blockBase;
	unsigned takers = __ballot_sync(0xFFFFFFFFu, take);
	int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	if (lane == 0)
	{
		warpOffset[warp] = __popc(takers);
	}
	__syncthreads();
	if (threadIdx.x == 0)
	{
		int total = 0;
		int warps = (blockDim.x + 31) >> 5;
		for (int k = 0; k < warps; ++k)
		{
			int c = warpOffset[k];
			warpOffset[k] = total;
			total += c;
		}
		blockBase = total > 0 ? atomicAdd(count, total) : 0;
	}
	__syncthreads();
	if (take)
	{
		list[blockBase + warpOffset[warp] + __popc(takers & ((1u << lane) - 1u))] = value;
	}
}

// The queries of this pass are the proxies that moved (BC_MOVED, movedShapes), in Morton order — neighbours stay
// neighbours in the list, a warp's queries share the nodes they test — except up to S2B_MAX_LARGE_MOVERS proxies with
// LARGE boxes (a container wall spanning the scene overlaps thousands of leaves: one thread testing them all takes
// milliseconds), which go to largeShapes (BC_LARGE) and are tested the other way round: every leaf against that short
// list (s2bFindPairsLarge). "Large" is measured against the scene box of the last rebuild.
#define S2B_MAX_LARGE_MOVERS 64

// Refit of the hierarchy and collection of the queries in one launch (256 threads a block). Thread k copies the box of
// sorted leaf k; the 16-lane groups reduce level 1, each block reduces its level-2 node, and the last block to finish
// reduces the levels above. The pass clears BC_REFIT_DONE before this runs.
__global__ void __launch_bounds__(256) s2bRefit(ShapeView s, const int* sortedShape, int* counters, const int* boundsBits,
												 float4* nodeBox, int* movedShapes, int* largeShapes)
{
	int n = counters[BC_LEAVES];
	int nh = n - min(counters[BC_LARGE_LEAVES], S2B_MAX_LARGE_LEAVES);
	int k = blockIdx.x * blockDim.x + threadIdx.x;
	bool moved = false;
	int shape = -1;
	float4 box = s2bEmptyBox();
	if (k < n)
	{
		shape = sortedShape[k];
		box = s.fat[shape];
		nodeBox[k] = box;
		moved = (s.head[shape].x & S2B_SHAPE_MOVED) != 0;
		if (moved && n >= 256)
		{
			float sceneArea = (s2bOrderedToFloat(boundsBits[6]) - s2bOrderedToFloat(boundsBits[4])) *
							  (s2bOrderedToFloat(boundsBits[7]) - s2bOrderedToFloat(boundsBits[5]));
			float area = (box.z - box.x) * (box.w - box.y);
			if (area * 256.0f > sceneArea)
			{
				int slot = atomicAdd(counters + BC_LARGE, 1);
				if (slot < S2B_MAX_LARGE_MOVERS)
				{
					largeShapes[slot] = shape;
					moved = false;
				}
			}
		}
	}
	s2bBlockAppend(moved, shape, movedShapes, counters + BC_MOVED);

	int offset[S2B_MAX_LEVELS], count[S2B_MAX_LEVELS];
	int top = s2bLevels(n, nh, offset, count);
	__shared__ float4 level1[256 / S2B_FANOUT];
	__shared__ bool lastBlock;
	float4 group = s2bUnion16(k < nh ? box : s2bEmptyBox());
	if ((threadIdx.x & (S2B_FANOUT - 1)) == 0)
	{
		if (top >= 1 && k < nh)
		{
			nodeBox[offset[1] + k / S2B_FANOUT] = group;
		}
		level1[threadIdx.x / S2B_FANOUT] = group;
	}
	__syncthreads();
	if (threadIdx.x < 32)
	{
		float4 node = s2bUnion16(threadIdx.x < 256 / S2B_FANOUT ? level1[threadIdx.x] : s2bEmptyBox());
		if (threadIdx.x == 0 && top >= 2 && blockIdx.x * 256 < nh)
		{
			nodeBox[offset[2] + blockIdx.x] = node;
		}
	}
	if (threadIdx.x == 0)
	{
		__threadfence();
		lastBlock = atomicAdd(counters + BC_REFIT_DONE, 1) == (int)gridDim.x - 1;
	}
	__syncthreads();
	if (lastBlock == false)
	{
		return;
	}
	__threadfence();
	for (int l = 3; l <= top; ++l)
	{
		const float4* below = nodeBox + offset[l - 1];
		for (int i = threadIdx.x; i < count[l]; i += blockDim.x)
		{
			int first = i * S2B_FANOUT, last = min(first + S2B_FANOUT, count[l - 1]);
			float4 r = s2bEmptyBox();
			for (int j = first; j < last; ++j)
			{
				// L2 reads: level 2 was written by the other blocks
				r = s2bUnion(r, __ldcg(below + j));
			}
			nodeBox[offset[l] + i] = r;
		}
		__syncthreads();
	}
	if (threadIdx.x == 0)
	{
		counters[BC_HEIGHT] = top + 1;
	}
}

// what the query of proxy Q does with an overlapping proxy `other` (reference s2PairQueryCallback, src/broad_phase.c:166-258)
struct PairQuery
{
	int shapeQ, bodyQ, keyQ;
	unsigned typeBodyQ;
	int4 headQ, filterQ;
};

__device__ __forceinline__ void s2bConsiderPair(const PairQuery& q, int other, const ShapeView& s, const BodyView& b, int* counters,
												 const unsigned long long* pairHash, unsigned long long hashMask,
												 const unsigned long long* jointKeys, int jointKeyCount, unsigned long long* newKey,
												 int2* newShapes, int newCap)
{
	int shapeQ = q.shapeQ;
	if (other == shapeQ)
	{
		return;
	}
	int4 headO = s.head[other];
	int bodyO = headO.y;
	int keyO = headO.z;
	unsigned typeBodyO = S2B_BODY_TYPE((unsigned)b.flags[bodyO]);
	// a kinematic proxy only queries the dynamic tree
	if (q.typeBodyQ == S2B_BODY_KINEMATIC && typeBodyO != S2B_BODY_DYNAMIC)
	{
		return;
	}
	// both proxies moved: the one with the smaller key reports the pair
	if ((headO.x & S2B_SHAPE_MOVED) && keyO > q.keyQ)
	{
		// ... unless the other one cannot see us in its own query
		bool otherSeesUs = !(typeBodyO == S2B_BODY_KINEMATIC && q.typeBodyQ != S2B_BODY_DYNAMIC) && typeBodyO != S2B_BODY_STATIC;
		if (otherSeesUs)
		{
			return;
		}
	}
	if (bodyO == q.bodyQ)
	{
		return;
	}
	unsigned long long lo = (unsigned long long)(other < shapeQ ? other : shapeQ);
	unsigned long long hi = (unsigned long long)(other < shapeQ ? shapeQ : other);
	unsigned long long pairKey = (lo << 32) | hi;
	// "this pair already has a contact" — unless one of the shapes was (re)created since the table was built: the table's
	// contact then belongs to the shape that used to live in that slot and is dropped by this very pass (s2bCollectKeptContacts),
	// so the pair has to be reported again (the reference removes the key from its pair set when the old shape is destroyed,
	// src/contact.c:231-292, and creates the contact on the next update)
	bool recreated = ((q.headQ.x | headO.x) & S2B_SHAPE_FRESH) != 0;
	if (recreated == false && s2bPairInHash(pairHash, hashMask, pairKey))
	{
		return;
	}
	int shapeA, shapeB;
	if (keyO < q.keyQ)
	{
		shapeA = other;
		shapeB = shapeQ;
	}
	else
	{
		shapeA = shapeQ;
		shapeB = other;
	}
	int4 filterO = s.filter[other];
	if (s2bShouldShapesCollide(shapeA == shapeQ ? q.filterQ : filterO, shapeA == shapeQ ? filterO : q.filterQ) == false)
	{
		return;
	}
	if (s2bJointOverride(jointKeys, jointKeyCount, q.bodyQ, bodyO))
	{
		return;
	}
	int typeA = ((shapeA == shapeQ ? q.headQ.x : headO.x) >> 1) & 0x7;
	int typeB = ((shapeA == shapeQ ? headO.x : q.headQ.x) >> 1) & 0x7;
	int kind = s2bPairKind(typeA, typeB);
	if (kind == 0)
	{
		return;
	}
	if (kind == 2)
	{
		int tmp = shapeA;
		shapeA = shapeB;
		shapeB = tmp;
	}
	int slot = atomicAdd(counters + BC_NEW_PAIRS, 1);
	if (slot < newCap)
	{
		newKey[slot] = pairKey;
		newShapes[slot] = make_int2(shapeA, shapeB);
	}
}

__device__ __forceinline__ bool s2bMakeQuery(PairQuery& q, int shapeQ, const ShapeView& s, const BodyView& b)
{
	q.shapeQ = shapeQ;
	q.headQ = s.head[shapeQ];
	q.filterQ = s.filter[shapeQ];
	q.bodyQ = q.headQ.y;
	q.keyQ = q.headQ.z;
	q.typeBodyQ = S2B_BODY_TYPE((unsigned)b.flags[q.bodyQ]);
	return q.typeBodyQ != S2B_BODY_STATIC; // static proxies never query (reference src/broad_phase.c:284-299)
}

#define S2B_QUERY_BATCH 16

// bit j set: child box j of the `count` (<= 16) boxes at `boxes` overlaps q; the loads are independent
__device__ __forceinline__ unsigned s2bOverlapMask(const float4* __restrict__ boxes, int count, float4 q)
{
	unsigned mask = 0;
#pragma unroll
	for (int j = 0; j < S2B_FANOUT; ++j)
	{
		if (j < count && s2bBoxesOverlap(q, __ldg(boxes + j)))
		{
			mask |= 1u << j;
		}
	}
	return mask;
}

// survivors: both shapes alive and not re-created, fat AABBs still overlap (reference src/world.c:149-166), and no joint
// created since forbids the pair (reference src/joint.c:214-217)
// The survivors' slots are appended to keepSlots (BC_KEPT): their order does not matter, the merged table is sorted by pair key.
__device__ __forceinline__ void s2bCollectKeptContacts(int i, const ContactView& c, int contactCount, const ShapeView& s,
														const unsigned long long* jointKeys, int jointKeyCount, int* keepSlots, int* counters)
{
	bool keep = false;
	if (i < contactCount)
	{
		int2 sh = c.shapes[i];
		int4 ha = s.head[sh.x], hb = s.head[sh.y];
		bool alive = (ha.x & S2B_ROW_VALID) && (hb.x & S2B_ROW_VALID) && (ha.x & S2B_SHAPE_FRESH) == 0 && (hb.x & S2B_SHAPE_FRESH) == 0;
		keep = alive && s2bBoxesOverlap(s.fat[sh.x], s.fat[sh.y]) && s2bJointOverride(jointKeys, jointKeyCount, ha.y, hb.y) == false;
	}
	s2bBlockAppend(keep, i, keepSlots, counters + BC_KEPT);
}

// Blocks [0, queryBlocks): one thread per moved proxy with an ordinary box walks the hierarchy and tests the large-leaf
// list. The blocks behind them collect the survivors of the current table, which is independent of the queries and runs in
// the shadow of their tail.
__global__ void __launch_bounds__(128) s2bFindPairs(ShapeView s, BodyView b, const int* sortedShape, int* counters, const int* movedShapes,
													const float4* __restrict__ nodeBox, int queryBlocks, ContactView cur, int contactCount,
													const unsigned long long* destroyKeys, int destroyKeyCount, int* keepSlots,
													const unsigned long long* pairHash, unsigned long long hashMask,
													const unsigned long long* jointKeys, int jointKeyCount, unsigned long long* newKey,
													int2* newShapes, int newCap)
{
	if ((int)blockIdx.x >= queryBlocks)
	{
		s2bCollectKeptContacts(((int)blockIdx.x - queryBlocks) * blockDim.x + threadIdx.x, cur, contactCount, s, destroyKeys,
							   destroyKeyCount, keepSlots, counters);
		return;
	}
	int n = counters[BC_LEAVES];
	int large = min(counters[BC_LARGE_LEAVES], S2B_MAX_LARGE_LEAVES);
	int nh = n - large;
	int movedCount = counters[BC_MOVED];
	int qi = blockIdx.x * blockDim.x + threadIdx.x;
	if (qi >= movedCount)
	{
		return;
	}
	PairQuery q;
	if (s2bMakeQuery(q, movedShapes[qi], s, b) == false)
	{
		return;
	}
	float4 boxQ = s.fat[q.shapeQ];

	// Depth-first over the levels with one pending child mask per level. Overlapping LEAVES are only collected during the
	// walk and examined in batches afterwards: the walk (box tests) and the pair rules (shape header, hash probe, filters)
	// are two different instruction streams, and a warp whose lanes hit leaves at different moments would otherwise
	// execute both serially for every lane (10 of 32 lanes active, ncu round 1).
	int offset[S2B_MAX_LEVELS], count[S2B_MAX_LEVELS];
	int top = s2bLevels(n, nh, offset, count);
	unsigned pending[S2B_MAX_LEVELS];
	int base[S2B_MAX_LEVELS];
	int found[S2B_QUERY_BATCH + S2B_FANOUT];
	int nFound = 0;
	int level = top;
	bool walking = nh > 0;
	if (walking)
	{
		pending[top] = s2bOverlapMask(nodeBox + offset[top], count[top], boxQ);
		base[top] = 0;
	}
	while (walking || nFound > 0)
	{
		while (walking && nFound < S2B_QUERY_BATCH)
		{
			unsigned m = pending[level];
			if (level == 0 || m == 0)
			{
				for (; m != 0; m &= m - 1)
				{
					found[nFound++] = base[0] + __ffs(m) - 1;
				}
				level += 1;
				walking = level <= top;
				continue;
			}
			pending[level] = m & (m - 1);
			int first = (base[level] + __ffs(m) - 1) * S2B_FANOUT;
			pending[level - 1] = s2bOverlapMask(nodeBox + offset[level - 1] + first, min(S2B_FANOUT, count[level - 1] - first), boxQ);
			base[level - 1] = first;
			level -= 1;
		}
		for (int k = 0; k < nFound; ++k)
		{
			s2bConsiderPair(q, sortedShape[found[k]], s, b, counters, pairHash, hashMask, jointKeys, jointKeyCount, newKey, newShapes,
							newCap);
		}
		nFound = 0;
	}
	for (int i = nh; i < n; ++i)
	{
		if (s2bBoxesOverlap(boxQ, nodeBox[i]))
		{
			s2bConsiderPair(q, sortedShape[i], s, b, counters, pairHash, hashMask, jointKeys, jointKeyCount, newKey, newShapes, newCap);
		}
	}
}

// every leaf against the short list of large movers (s2bRefit). Same rules, same pairs; the order new pairs are
// emitted in never matters (they are sorted).
__global__ void s2bFindPairsLarge(ShapeView s, BodyView b, const int* leafShape, int* counters, const int* largeShapes,
								  const unsigned long long* pairHash, unsigned long long hashMask, const unsigned long long* jointKeys,
								  int jointKeyCount, unsigned long long* newKey, int2* newShapes, int newCap)
{
	int n = counters[BC_LEAVES];
	int large = min(counters[BC_LARGE], S2B_MAX_LARGE_MOVERS);
	int k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k >= n || large == 0)
	{
		return;
	}
	int other = leafShape[k];
	float4 boxO = s.fat[other];
	for (int i = 0; i < large; ++i)
	{
		int shapeQ = largeShapes[i];
		if (s2bBoxesOverlap(s.fat[shapeQ], boxO) == false)
		{
			continue;
		}
		PairQuery q;
		if (s2bMakeQuery(q, shapeQ, s, b))
		{
			s2bConsiderPair(q, other, s, b, counters, pairHash, hashMask, jointKeys, jointKeyCount, newKey, newShapes, newCap);
		}
	}
}

// The sort key is the pair key squeezed to 2 x shapeBits bits (lo << shapeBits | hi) so the radix sort runs only over
// significant digits.
__device__ __forceinline__ unsigned long long s2bSqueezeKey(unsigned long long pairKey, int shapeBits)
{
	return ((pairKey >> 32) << shapeBits) | (pairKey & 0xFFFFFFFFull);
}

__global__ void s2bMergeKeys(const int* counters, const int* keepSlots, const unsigned long long* oldKeys,
							 const unsigned long long* newKey, unsigned long long* mergeKey, int* mergeSrc, int capacity, int shapeBits)
{
	int kept = counters[BC_KEPT], fresh = counters[BC_NEW_PAIRS];
	int t = blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= capacity)
	{
		return;
	}
	if (t < kept)
	{
		mergeKey[t] = s2bSqueezeKey(oldKeys[keepSlots[t]], shapeBits);
		mergeSrc[t] = keepSlots[t]; // >= 0: old slot
	}
	else if (t < kept + fresh)
	{
		mergeKey[t] = s2bSqueezeKey(newKey[t - kept], shapeBits);
		mergeSrc[t] = -1 - (t - kept); // < 0: new pair index
	}
	else
	{
		mergeKey[t] = ~0ull;
		mergeSrc[t] = 0;
	}
}

// s2CreateContact for new pairs (reference src/contact.c:156-229: empty manifold, empty cache, mixed friction), plain
// copy for survivors
__global__ void s2bGatherContactsSorted(const int* counters, const unsigned long long* sortedKey, const int* sortedSrc, ContactView src,
										ContactView dst, const int2* newShapes, ShapeView s, int sticky, int shapeBits)
{
	int total = counters[BC_KEPT] + counters[BC_NEW_PAIRS];
	int t = blockIdx.x * blockDim.x + threadIdx.x;
	if (t >= total)
	{
		return;
	}
	int from = sortedSrc[t];
	unsigned long long squeezed = sortedKey[t];
	dst.key[t] = ((squeezed >> shapeBits) << 32) | (squeezed & ((1ull << shapeBits) - 1ull));
	if (from >= 0)
	{
		dst.shapes[t] = src.shapes[from];
		dst.bodies[t] = src.bodies[from];
		dst.info[t] = src.info[from];
		dst.nf[t] = src.nf[from];
		dst.color[t] = src.color[from];
		for (int p = 0; p < 2; ++p)
		{
			dst.anchor[p][t] = src.anchor[p][from];
			dst.impulse[p][t] = src.impulse[p][from];
			if (sticky)
			{
				dst.fanchor[p][t] = src.fanchor[p][from];
				dst.fnormal[p][t] = src.fnormal[p][from];
			}
		}
	}
	else
	{
		int2 sh = newShapes[-1 - from];
		dst.shapes[t] = sh;
		dst.bodies[t] = make_int2(s.head[sh.x].y, s.head[sh.y].y);
		dst.info[t] = make_int4(0, 0, 0, 0);
		// s2MixFriction (reference src/contact.c:42-45)
		float friction = sqrtf(s.fr[sh.x].x * s.fr[sh.y].x);
		dst.nf[t] = make_float4(0.0f, 0.0f, friction, 0.0f);
		dst.color[t] = -1;
		for (int p = 0; p < 2; ++p)
		{
			dst.anchor[p][t] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
			dst.impulse[p][t] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
			if (sticky)
			{
				dst.fanchor[p][t] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
				dst.fnormal[p][t] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
			}
		}
	}
}

__global__ void s2bClearMovedFlags(ShapeView s, int* movedCounter)
{
	int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i < s.capacity)
	{
		int4 h = s.head[i];
		if (h.x & (S2B_SHAPE_MOVED | S2B_SHAPE_FRESH))
		{
			s.head[i] = make_int4(h.x & ~(S2B_SHAPE_MOVED | S2B_SHAPE_FRESH), h.y, h.z, h.w);
		}
	}
	if (i == 0)
	{
		movedCounter[0] = 0;
	}
}

// ---------------------------------------------------------------------------------------------------------------
// host driver
// ---------------------------------------------------------------------------------------------------------------

// mailbox slots of the pair pass (pinned host memory, written by asynchronous copies)
#define MAIL_BC_BASE 16

// scratch sizes of a pass (host only; the pass itself never allocates between its kernels)
static size_t bpReserve(s2bWorld* w, BroadScratch* B)
{
	cudaStream_t st = w->stream;
	int shapeCap = w->shapeCap;
	int oldCount = w->contactCount;
	size_t nS = (size_t)shapeCap;
	B->validFlag.reserve(nS, st, false);
	B->leafShape.reserve(nS, st, false);
	B->mortonIn.reserve(nS, st, false);
	B->mortonOut.reserve(nS, st, false);
	B->leafIn.reserve(nS, st, false);
	B->leafOut.reserve(nS, st, false);
	B->sortedShape.reserve(nS, st, false);
	B->counters.reserve(BC_SIZE, st, false);
	B->boundsBits.reserve(8, st, false);
	B->nodeBox.reserve(nS + nS / 8 + 64, st, false); // leaves + levels: n (1 + 1/16 + 1/256 + ...) + one per level
	B->movedShapes.reserve(nS, st, false);
	B->movedFlag.reserve(nS, st, false);
	B->largeShapes.reserve(S2B_MAX_LARGE_MOVERS, st, false);
	B->keepFlag.reserve((size_t)std::max(oldCount, 1), st, false);
	B->keepSlots.reserve((size_t)std::max(oldCount, 1), st, false);
	if (B->newPairCap == 0)
	{
		B->newPairCap = 8 * shapeCap + 1024;
	}
	size_t need = 0, tempBytes = 0;
	cub::DeviceSelect::Flagged(nullptr, need, thrust::counting_iterator<int>(0), (int*)nullptr, (int*)nullptr, (int*)nullptr,
							   std::max(shapeCap, oldCount), st);
	tempBytes = std::max(tempBytes, need);
	cub::DeviceRadixSort::SortPairs(nullptr, need, (unsigned*)nullptr, (unsigned*)nullptr, (int*)nullptr, (int*)nullptr, shapeCap, 0,
									32, st);
	tempBytes = std::max(tempBytes, need);
	B->newKey.reserve((size_t)B->newPairCap, st, false);
	B->newShapes.reserve((size_t)B->newPairCap, st, false);
	B->cubTemp.reserve(tempBytes + 256, st, false, false);
	return tempBytes;
}

// First half of a pass, no host synchronisation: sorted order (re-used or rebuilt) and refit, pair-key hash of the current
// table, queries from the moved proxies -> candidate pairs (newKey / newShapes), survivors of the current table (keepSlots),
// and the counters of all that copied to the pinned mailbox.
static void bpSearch(s2bWorld* w, BroadScratch* B)
{
	cudaStream_t st = w->stream;
	int shapeCap = w->shapeCap;
	int oldCount = w->contactCount;
	ShapeView sv = shapeView(w);
	BodyView bv = bodyView(w);
	ContactColumns& cur = w->contacts[w->cur];
	int newCap = B->newPairCap;

	// the sorted order (and with it the hierarchy's topology and the large-leaf list) is reused while no shape was
	// created, destroyed or re-uploaded; boxes drift a little per step, a periodic re-sort keeps the nodes tight
	bool reuseTree = B->treeValid && w->pairsDirty == false && B->treeShapeCap == shapeCap && B->treeReuses < S2B_TREE_REUSE_LIMIT;
	if (reuseTree)
	{
		// keep BC_LEAVES / BC_LARGE_LEAVES; clear the per-pass counters
		S2B_CHECK(cudaMemsetAsync(B->counters.p + BC_NEW_PAIRS, 0, sizeof(int) * (BC_SIZE - BC_NEW_PAIRS), st));
		B->treeReuses += 1;
	}
	else
	{
		S2B_CHECK(cudaMemsetAsync(B->counters.p, 0, sizeof(int) * BC_SIZE, st));

		// ---- leaves ----
		S2B_LAUNCH(w, s2bFlagValidShapes, gridFor(shapeCap, 256), 256, 0, sv, B->validFlag.p);
		size_t tb = B->cubTemp.cap;
		cub::DeviceSelect::Flagged(B->cubTemp.p, tb, thrust::counting_iterator<int>(0), B->validFlag.p, B->leafShape.p,
								   B->counters.p + BC_LEAVES, shapeCap, st);
		w->kernelLaunches += 2;

		// ---- Morton order, large leaves last ----
		// ordered encoding: +FLT_MAX -> 0x7F7FFFFF, -FLT_MAX -> 0xFF7FFFFF ^ 0x7FFFFFFF = 0x80800000
		const int lo = 0x7F7FFFFF, hi = (int)0x80800000;
		int initBounds[8] = {lo, lo, hi, hi, lo, lo, hi, hi};
		S2B_CHECK(cudaMemcpyAsync(B->boundsBits.p, initBounds, sizeof(initBounds), cudaMemcpyHostToDevice, st));
		S2B_LAUNCH(w, s2bSceneBounds, gridFor(shapeCap, 256), 256, 0, sv, B->leafShape.p, B->counters.p, B->boundsBits.p);
		S2B_LAUNCH(w, s2bMortonCodes, gridFor(shapeCap, 256), 256, 0, sv, B->leafShape.p, B->counters.p, B->boundsBits.p,
				   B->mortonIn.p, B->leafIn.p, shapeCap);
		tb = B->cubTemp.cap;
		cub::DeviceRadixSort::SortPairs(B->cubTemp.p, tb, B->mortonIn.p, B->mortonOut.p, B->leafIn.p, B->leafOut.p, shapeCap, 0, 32, st);
		w->kernelLaunches += 5;
		S2B_LAUNCH(w, s2bSortedShapes, gridFor(shapeCap, 256), 256, 0, B->leafShape.p, B->leafOut.p, B->counters.p, B->sortedShape.p);
		B->treeValid = true;
		B->treeShapeCap = shapeCap;
		B->treeReuses = 0;
		w->pairRebuildCount += 1;
	}

	// ---- refit, and the moved proxies ----
	S2B_LAUNCH(w, s2bRefit, gridFor(shapeCap, 256), 256, 0, sv, B->sortedShape.p, B->counters.p, B->boundsBits.p, B->nodeBox.p,
			   B->movedShapes.p, B->largeShapes.p);

	// ---- pair-key hash set of the current contact table (rebuilt only when the table changed) ----
	if (B->hashVersion != w->contactTableVersion || B->pairHash.p == nullptr)
	{
		unsigned long long size = 1024;
		while (size < 2ull * (unsigned long long)std::max(oldCount, 1))
		{
			size <<= 1;
		}
		B->pairHash.reserve((size_t)size, st, false, false);
		B->hashMask = size - 1;
		S2B_CHECK(cudaMemsetAsync(B->pairHash.p, 0xFF, sizeof(unsigned long long) * (size_t)size, st));
		if (oldCount > 0)
		{
			S2B_LAUNCH(w, s2bBuildPairHash, gridFor(oldCount, 256), 256, 0, cur.key.p, oldCount, B->pairHash.p, B->hashMask);
		}
		B->hashVersion = w->contactTableVersion;
	}

	// ---- queries from moved proxies, and the survivors ----
	int queryBlocks = gridFor(shapeCap, 128);
	S2B_LAUNCH(w, s2bFindPairs, queryBlocks + (oldCount > 0 ? gridFor(oldCount, 128) : 0), 128, 0, sv, bv, B->sortedShape.p,
			   B->counters.p, B->movedShapes.p, B->nodeBox.p, queryBlocks, makeView(cur), oldCount, w->jointDestroyKeys.p,
			   w->jointDestroyCount, B->keepSlots.p, B->pairHash.p, B->hashMask, w->jointPairKeys.p, w->jointPairCount, B->newKey.p,
			   B->newShapes.p, newCap);
	S2B_LAUNCH(w, s2bFindPairsLarge, gridFor(shapeCap, 256), 256, 0, sv, bv, B->leafShape.p, B->counters.p, B->largeShapes.p,
			   B->pairHash.p, B->hashMask, w->jointPairKeys.p, w->jointPairCount, B->newKey.p, B->newShapes.p, newCap);
	S2B_CHECK(cudaMemcpyAsync(w->hostMail + MAIL_BC_BASE, B->counters.p, sizeof(int) * BC_SIZE, cudaMemcpyDeviceToHost, st));
	B->searchedCount = oldCount;
	B->searchedVersion = w->contactTableVersion;
}

// Second half: the host knows how many candidate pairs and survivors the search found. Merge them into the other column
// set (or leave the table as it is), clear the MOVED / FRESH flags.
static void bpCommit(s2bWorld* w, BroadScratch* B, int fresh, int kept, size_t tempBytes)
{
	cudaStream_t st = w->stream;
	int shapeCap = w->shapeCap;
	int oldCount = w->contactCount;
	ShapeView sv = shapeView(w);
	ContactColumns& cur = w->contacts[w->cur];
	ContactColumns& nxt = w->contacts[w->cur ^ 1];
	int total = kept + fresh;
	if (fresh == 0 && kept == oldCount)
	{
		// the moved proxies still overlap exactly the shapes they overlapped before: the contact table stands as it is
		// (the usual outcome on a slowly settling pile)
	}
	else
	{
		nxt.reserve((size_t)std::max(total, 1), st, w->sticky, false);
		if (total > 0)
		{
			size_t need = 0;
			B->mergeKeyIn.reserve((size_t)total, st, false);
			B->mergeKeyOut.reserve((size_t)total, st, false);
			B->mergeSrcIn.reserve((size_t)total, st, false);
			B->mergeSrcOut.reserve((size_t)total, st, false);
			cub::DeviceRadixSort::SortPairs(nullptr, need, (unsigned long long*)nullptr, (unsigned long long*)nullptr, (int*)nullptr,
											(int*)nullptr, total, 0, 64, st);
			B->cubTemp.reserve(std::max(tempBytes, need) + 256, st, false, false);
			int shapeBits = 1;
			while ((1 << shapeBits) < shapeCap && shapeBits < 31)
			{
				shapeBits += 1;
			}
			S2B_LAUNCH(w, s2bMergeKeys, gridFor(total, 256), 256, 0, B->counters.p, B->keepSlots.p, cur.key.p, B->newKey.p,
					   B->mergeKeyIn.p, B->mergeSrcIn.p, total, shapeBits);
			size_t tb = B->cubTemp.cap;
			cub::DeviceRadixSort::SortPairs(B->cubTemp.p, tb, B->mergeKeyIn.p, B->mergeKeyOut.p, B->mergeSrcIn.p, B->mergeSrcOut.p,
											total, 0, 2 * shapeBits, st);
			w->kernelLaunches += 9;
			S2B_LAUNCH(w, s2bGatherContactsSorted, gridFor(total, 128), 128, 0, B->counters.p, B->mergeKeyOut.p, B->mergeSrcOut.p,
					   makeView(cur), makeView(nxt), B->newShapes.p, sv, w->sticky ? 1 : 0, shapeBits);
		}
		w->cur ^= 1;
		w->contactCount = total;
		w->contactTableVersion += 1;
		// size what the NEXT pass needs for this table now, while a re-allocation is already being paid for: the survivor
		// flags and the pair-key hash set (built lazily by that pass)
		B->keepFlag.reserve((size_t)std::max(total, 1), st, false);
		B->keepSlots.reserve((size_t)std::max(total, 1), st, false);
		{
			unsigned long long size = 1024;
			while (size < 2ull * (unsigned long long)std::max(total, 1))
			{
				size <<= 1;
			}
			B->pairHash.reserve((size_t)size, st, false, false);
		}
	}
	S2B_LAUNCH(w, s2bClearMovedFlags, gridFor(shapeCap, 256), 256, 0, sv, w->dMovedFlag.p);
	w->hostMail[MAIL_MOVED] = 0;
	w->pairsDirty = false;
	w->pairPassCount += 1;
}

// Start the pair search of the NEXT step behind this one (called after finalize): its inputs — fat AABBs, MOVED flags, the
// contact table — are final once finalize has run, and its counters then reach the host together with the end of the step,
// which the caller waits for anyway before it reads results. The next s2b_update_pairs picks the result up without having to
// stop in the middle of the pass (DESIGN.md §3.3). Anything the host uploads in between invalidates the search (uploadEpoch).
void s2bPrefetchPairSearch(s2bWorld* w)
{
	S2bEpochFreeze freeze;
	BroadScratch* B = getBroad(w);
	B->prefetched = false;
	// only scenes in motion: on a settled scene nothing is enqueued and the next pass is skipped from the moved counter alone
	if (w->prefetchPairs == 0 || w->shapeCap == 0 || B->lastPassRan == false || w->pairsDirty)
	{
		return;
	}
	if (B->evSearch[0] == nullptr)
	{
		S2B_CHECK(cudaEventCreate(&B->evSearch[0]));
		S2B_CHECK(cudaEventCreate(&B->evSearch[1]));
		S2B_CHECK(cudaEventCreateWithFlags(&B->searchDone, cudaEventDisableTiming));
	}
	B->prefetchTempBytes = bpReserve(w, B);
	S2B_CHECK(cudaEventRecord(B->evSearch[0], w->stream));
	bpSearch(w, B);
	S2B_CHECK(cudaEventRecord(B->evSearch[1], w->stream));
	S2B_CHECK(cudaEventRecord(B->searchDone, w->stream));
	B->prefetched = true;
	B->prefetchEpoch = w->uploadEpoch;
	B->searchTimed = true;
}

float s2bLastPairSearchMs(s2bWorld* w)
{
	BroadScratch* B = w->broad;
	if (B == nullptr || B->searchTimed == false)
	{
		return 0.0f;
	}
	float ms = 0.0f;
	if (cudaEventQuery(B->evSearch[1]) == cudaSuccess)
	{
		cudaEventElapsedTime(&ms, B->evSearch[0], B->evSearch[1]);
	}
	return ms;
}

void s2bBroadphaseUpdatePairs(s2bWorld* w)
{
	// scratch of this pass is not referenced by the solver's graph; a REPLACED contact table is, and shows up in the graph
	// signature through w->cur / w->contactCount / w->contactTableVersion
	S2bEpochFreeze freeze;
	cudaStream_t st = w->stream;
	BroadScratch* B = getBroad(w);
	w->dMovedFlag.reserve(4, st, true);

	// ---- the search was started behind the previous step: its counters are (about to be) in the mailbox ----
	if (B->prefetched)
	{
		B->prefetched = false;
		bool valid = w->pairsDirty == false && B->prefetchEpoch == w->uploadEpoch && B->searchedVersion == w->contactTableVersion &&
					 B->searchedCount == w->contactCount && w->prefetchPairs == 1; // (2: search but never use the result — debugging)
		if (valid)
		{
			S2B_CHECK(cudaEventSynchronize(B->searchDone));
			S2B_CHECK(cudaEventRecord(w->timer.ev[0], st));
			const int* hc = w->hostMail + MAIL_BC_BASE;
			int fresh = hc[BC_NEW_PAIRS], kept = hc[BC_KEPT];
			if (fresh <= B->newPairCap)
			{
				w->treeHeight = hc[BC_HEIGHT];
				w->largeLeafCount = std::min(hc[BC_LARGE_LEAVES], S2B_MAX_LARGE_LEAVES);
				B->lastPassRan = hc[BC_MOVED] > 0 || hc[BC_LARGE] > 0;
				bpCommit(w, B, fresh, kept, B->prefetchTempBytes);
				return;
			}
			B->newPairCap = fresh + fresh / 2 + 1024; // rare: redo the pass below with a larger pair buffer
		}
		// (something was uploaded since: the search is stale — e.g. new shapes — and is redone)
	}

	// Did anything move in the last finalize? The counter was copied to the pinned mailbox at the end of the previous
	// step; wait for that copy (normally long done) and read it.
	bool run = w->pairsDirty;
	if (run == false)
	{
		// (wait for THAT copy only — not for whatever the caller has enqueued since: force uploads, row scatters — so that the
		// kernels of this step can be queued behind them without the host idling)
		if (w->movedEvent != nullptr)
		{
			S2B_CHECK(cudaEventSynchronize(w->movedEvent));
		}
		else
		{
			S2B_CHECK(cudaStreamSynchronize(st));
		}
		run = w->hostMail[MAIL_MOVED] > 0;
	}
	S2B_CHECK(cudaEventRecord(w->timer.ev[0], st));
	B->lastPassRan = run && w->shapeCap > 0;
	if (run == false || w->shapeCap == 0)
	{
		return;
	}

	for (int attempt = 0; attempt < 4; ++attempt)
	{
		size_t tempBytes = bpReserve(w, B);
		bpSearch(w, B);
		// the new table size has to be known on the host (column reservation): one small synchronising read-back, paid only
		// when the search could not be started behind the previous step (first steps, after uploads, settled scenes)
		S2B_CHECK(cudaStreamSynchronize(st));
		const int* hc = w->hostMail + MAIL_BC_BASE;
		int fresh = hc[BC_NEW_PAIRS], kept = hc[BC_KEPT];
		if (fresh > B->newPairCap)
		{
			B->newPairCap = fresh + fresh / 2 + 1024;
			continue; // rare: redo the pass with a larger pair buffer
		}
		w->treeHeight = hc[BC_HEIGHT];
		w->largeLeafCount = std::min(hc[BC_LARGE_LEAVES], S2B_MAX_LARGE_LEAVES);
		bpCommit(w, B, fresh, kept, tempBytes);
		break;
	}
}
