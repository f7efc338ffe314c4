// tinybvh_b200/csrc/build_sah.cu - binned-SAH BVH construction on sm_100a.
//
// Replaces BVH::PrepareBuild (tiny_bvh.h:2261-2329) + BVH::Build(nodeIdx,depth) (:2332-2461).  The result is the
// reference's own tree, byte for byte: same split decisions (8 bins x 3 axes, fp32 SAH in the oracle's operation
// order, first strict minimum over axis 0..2 / plane 0..6), same child bounds (bin unions), same primIdx order
// (the reference's in-place swap partition is reproduced by a closed-form parallel permutation, see
// partition_dest()), same node numbering as the single-threaded reference (children of the k-th interior node in
// DFS preorder at 2+2k, 3+2k; node 1 unused) - tests/test_build_gpu.py memcmp()s nodes and primIdx against it.
//
// Structure (DESIGN.md "build"):
//   k_fragments     per-triangle AABB + root AABB (block reduce -> ordered-int atomics)
//   large phase     nodes with more than SMALL_T primitives, level-synchronous over 256-primitive chunks:
//                   k_bin (shared-memory bin tables per CTA -> global per-node tables), k_sweep (one warp per node:
//                   21 candidate planes on 21 lanes, warp argmin), k_flags + exclusive scan + k_posbl + k_scatter
//                   (the swap-partition permutation into the ping-pong index buffer)
//   k_build_small   one warp per subtree of <= SMALL_T primitives, whole subtree built out of shared memory
//   relayout        DFS-preorder numbering from (first, depth) of every interior node: rank = #interior nodes that
//                   start earlier + position in the chain of nodes starting at the same primitive
#include "common.cuh"
#include <stdlib.h>
#include <string.h>
#include <vector>

#define BINS 8
#define SMALL_T 128          // capacity of the warp kernel: subtrees of at most this many primitives (run-time switch point <= this)
#define CHUNK 256            // primitives per CTA in the large phase
#define BUILD_CTAS_PER_SM 4  // resident CTAs per SM of the persistent large phase (k_large_phase)
#define BIN_WORDS 168        // 3 axes x 8 bins x (3 min keys, 3 max keys, count)
#define BIN_STRIDE 192       // + 3 x 8 counts of the PARTITION's own bin function (BuildAVX flavour, see bin_part_avx)
__device__ __forceinline__ uint32_t bin_init_word( const uint32_t k ) { return (k < BIN_WORDS && (k % 7) < 3) ? 0xffffffffu : 0u; }
#define SCAN_TILE 2048

struct LargeNode { uint32_t tmp, first, count, depth; };
struct SmallRoot { uint32_t tmp, first, count, depth_buf; }; // depth | buf << 16
struct SplitInfo { uint32_t did, axis, pos, L; };
struct Counters
{
	uint32_t tmp_nodes;      // temp node records allocated (pairs)
	uint32_t next_large;     // nodes appended to the next level's list
	uint32_t small_roots;    // subtree roots for k_build_small
	uint32_t max_depth;
	uint32_t total_chunks;   // chunks of the current level list
	uint32_t lvl_num[2];     // persistent large phase: nodes / chunks of the level with parity 0 / 1
	uint32_t lvl_chunks[2];
	uint32_t levels;         // persistent large phase: levels run
	uint32_t root_key[6];    // root AABB as ordered keys: min xyz, max xyz
	uint32_t pad[4];
};

struct BuildArgs
{
	const float4* verts;
	const float4* aabbs;     // TLAS build (BVH::Build( BLASInstance*, .. ) :2243-2255): fragment i = box (aabbs[2i], aabbs[2i+1]) instead of a triangle's
	float4* frag_min; float4* frag_max;
	uint32_t* idx[2]; uint32_t* idx_final;
	uint16_t* bin_ids;
	uint32_t* flags; uint32_t* scan; uint32_t* pos_bl;
	uint32_t* chunk_pre;     // persistent large phase: exclusive prefix of the per-chunk flag totals (chunks + 1 entries)
	float4* tmp_nodes; uint32_t* node_first; uint32_t* node_depth;
	LargeNode* lvl[2]; uint32_t* chunk_start; uint32_t* chunk_start_next; uint32_t* bins; SplitInfo* split;
	SmallRoot* small;
	Counters* ctr;
	uint32_t n;
	uint32_t flavour;        // 0 = BVH::Build (scalar reference builder), 1 = BVH::BuildAVX (what BuildDefault runs on x86)
	uint32_t small_t;        // runtime switch point large phase -> warp subtrees (<= SMALL_T; the context's small_t)
	uint32_t level0;         // persistent large phase: the level it starts at (the launch-per-stage path may have run the first ones)
	float c_trav, c_int;
};

// ---------------------------------------------------------------------------------------------- shared math

// (int)(((bmin+bmax)*0.5f - nmin) * rpd) clamped to [0,7]  (tiny_bvh.h:2362-2369; gcc fuses the *0.5f - nmin)
__device__ __forceinline__ uint32_t bin_of( const float bmin, const float bmax, const float nmin, const float rpd )
{
	const float f = __fmul_rn( __fmaf_rn( __fadd_rn( bmin, bmax ), 0.5f, -nmin ), rpd );
	// x86 cvttss2si returns INT_MIN for NaN / out-of-range -> clamps to 0; cvt.rzi saturates, so send those to 0 by hand
	int bi = (f >= 2147483648.0f) ? 0 : __float2int_rz( f );
	return (uint32_t)min( max( bi, 0 ), BINS - 1 );
}

// BuildAVX flavour (tiny_bvh.h:6500-6502, :6557-6559): nmin2 = 2 * node min, rpd = (8 * 0.49999f) / extent (0 on a zero extent);
// binning bin = clamp( cvtps2dq( fma( (bmax+bmin) - nmin2, rpd, -0.5 ) ), 0, 7 )  (round to nearest even; INT_MIN when out of range)
__device__ __forceinline__ float rpd_avx( const float ext ) { return ext == 0 ? 0.0f : __fdiv_rn( __fmul_rn( 8.0f, 0.49999f ), ext ); }
__device__ __forceinline__ uint32_t bin_of_avx( const float bmin, const float bmax, const float nmin2, const float rpd )
{
	const float f = __fmaf_rn( __fsub_rn( __fadd_rn( bmax, bmin ), nmin2 ), rpd, -0.5f );
	const int bi = (f >= 2147483648.0f) ? 0 : __float2int_rn( f );
	return (uint32_t)min( max( bi, 0 ), BINS - 1 );
}
// the partition's own bin (:6629): (uint32_t)((bmax + bmin - nmin2) * rpd) through a 64-bit truncation, not clamped; only
// "<= bestPos" (bestPos <= 6) is ever asked of it, so 7 stands for everything above
__device__ __forceinline__ uint32_t bin_part_avx( const float bmin, const float bmax, const float nmin2, const float rpd )
{
	const float f = __fmul_rn( __fsub_rn( __fadd_rn( bmax, bmin ), nmin2 ), rpd );
	const long long v = (f != f || f >= 9223372036854775808.0f || f < -9223372036854775808.0f) ? (long long)0x8000000000000000ull : __float2ll_rz( f );
	return min( (uint32_t)v, 7u );
}

// BVHBase::SA / tinybvh_half_area in the oracle's pairing (tiny_bvh.h:8477, :460)
__device__ __forceinline__ float half_area( const float ex, const float ey, const float ez )
{
	return __fmaf_rn( ez, ex, __fmaf_rn( ey, ex, __fmul_rn( ey, ez ) ) );
}

struct SweepResult { bool split; uint32_t axis, pos, lN; float l1[3], l2[3], r1[3], r2[3]; };

// One warp evaluates the 21 candidate planes of a node from its bin table (ordered keys + counts) - the sweep,
// termination test and child bounds of tiny_bvh.h:2380-2412.  All lanes return the same result.
__device__ __forceinline__ SweepResult sweep_node( uint32_t* bins /* BIN_WORDS, shared or global; decoded in place */, const float4 nmin, const float4 nmax,
	const uint32_t count, const float3 min_dim, const float c_trav, const float c_int, const uint32_t flavour )
{
	const uint32_t lane = threadIdx.x & 31;
	// decode pass: lanes 0..23 turn the six ordered keys of "their" bin back into floats, once, instead of every one of
	// the 7 candidate lanes of an axis decoding all 8 bins again
	if (lane < 3 * BINS)
	{
		uint32_t* w = bins + lane * 7;
		if (w[6] != 0)
		{
			#pragma unroll
			for (int k = 0; k < 6; k++) w[k] = __float_as_uint( key2f( w[k] ) );
		}
	}
	__syncwarp();
	// lanes 0..20: axis a, plane i.  The lane index is also the tie-break priority: planes 0..6 for BVH::Build (:2396-2404),
	// 3,2,4,5,1,0,6 for BuildAVX (:6614-6620).
	const uint32_t a = lane / 7, i = flavour ? ((0x6015423u >> (4 * (lane % 7))) & 7u) : lane % 7;
	float l1[3] = { BVH_FAR, BVH_FAR, BVH_FAR }, l2[3] = { -BVH_FAR, -BVH_FAR, -BVH_FAR };
	float r1[3] = { BVH_FAR, BVH_FAR, BVH_FAR }, r2[3] = { -BVH_FAR, -BVH_FAR, -BVH_FAR };
	uint32_t lN = 0, rN = 0;
	float C = 3e30f;
	if (lane < 21)
	{
		const float ext = a == 0 ? __fsub_rn( nmax.x, nmin.x ) : a == 1 ? __fsub_rn( nmax.y, nmin.y ) : __fsub_rn( nmax.z, nmin.z );
		const float md = a == 0 ? min_dim.x : a == 1 ? min_dim.y : min_dim.z;
		if (ext > md)
		{
			for (uint32_t b = 0; b < BINS; b++)
			{
				const uint32_t* w = bins + (a * BINS + b) * 7;
				const uint32_t c = w[6];
				if (c == 0) continue; // empty bin: the reference's +-BVH_FAR initial box, no effect on a union
				const float mnx = __uint_as_float( w[0] ), mny = __uint_as_float( w[1] ), mnz = __uint_as_float( w[2] );
				const float mxx = __uint_as_float( w[3] ), mxy = __uint_as_float( w[4] ), mxz = __uint_as_float( w[5] );
				if (b <= i)
				{
					l1[0] = fminf( l1[0], mnx ), l1[1] = fminf( l1[1], mny ), l1[2] = fminf( l1[2], mnz );
					l2[0] = fmaxf( l2[0], mxx ), l2[1] = fmaxf( l2[1], mxy ), l2[2] = fmaxf( l2[2], mxz ), lN += c;
				}
				else
				{
					r1[0] = fminf( r1[0], mnx ), r1[1] = fminf( r1[1], mny ), r1[2] = fminf( r1[2], mnz );
					r2[0] = fmaxf( r2[0], mxx ), r2[1] = fmaxf( r2[1], mxy ), r2[2] = fmaxf( r2[2], mxz ), rN += c;
				}
			}
			const float aL = half_area( __fsub_rn( l2[0], l1[0] ), __fsub_rn( l2[1], l1[1] ), __fsub_rn( l2[2], l1[2] ) );
			const float aR = half_area( __fsub_rn( r2[0], r1[0] ), __fsub_rn( r2[1], r1[1] ), __fsub_rn( r2[2], r1[2] ) );
			if (flavour)
			{
				// PROCESS_PLANE (:6394-6396): both sides non-empty, cost = fma( lN, areaL, areaR * rN )
				if (lN != 0 && rN != 0) C = __fmaf_rn( __uint2float_rn( lN ), aL, __fmul_rn( aR, __uint2float_rn( rN ) ) );
			}
			else
			{
				const float ANL = lN == 0 ? BVH_FAR : __fmul_rn( aL, __uint2float_rn( lN ) );
				const float ANR = rN == 0 ? BVH_FAR : __fmul_rn( aR, __uint2float_rn( rN ) );
				C = __fadd_rn( ANL, ANR );
			}
			if (flavour)
			{
				// the partition decides the child sizes with its own bin function: left count = its histogram up to plane i
				uint32_t pl = 0;
				for (uint32_t b = 0; b <= i; b++) pl += bins[BIN_WORDS + a * BINS + b];
				lN = pl;
			}
		}
	}
	// first strict minimum below BVH_FAR in (axis, plane) order == lowest lane holding the warp minimum
	float mC = C;
	for (int o = 16; o > 0; o >>= 1) mC = fminf( mC, __shfl_xor_sync( 0xffffffffu, mC, o ) );
	const bool found = mC < BVH_FAR;
	const uint32_t win = found ? (uint32_t)(__ffs( __ballot_sync( 0xffffffffu, C == mC ) ) - 1) : 0;
	const float splitCostIn = found ? mC : BVH_FAR;
	const float rSAV = __fdiv_rn( 1.0f, half_area( __fsub_rn( nmax.x, nmin.x ), __fsub_rn( nmax.y, nmin.y ), __fsub_rn( nmax.z, nmin.z ) ) );
	const float splitCost = __fmaf_rn( __fmul_rn( c_int, rSAV ), splitCostIn, c_trav );
	const float noSplitCost = __fmul_rn( __uint2float_rn( count ), c_int );
	SweepResult R;
	R.axis = win / 7, R.pos = __shfl_sync( 0xffffffffu, i, win );
	R.lN = __shfl_sync( 0xffffffffu, lN, win );
	// BuildAVX: if its partition puts everything on one side the reference leaves the node a leaf (:6639; it has by then
	// permuted primIdx and burnt two node slots - "should not happen", not reproduced)
	R.split = found && !(splitCost >= noSplitCost) && R.lN != 0 && R.lN != count;
	#pragma unroll
	for (int k = 0; k < 3; k++)
	{
		R.l1[k] = __shfl_sync( 0xffffffffu, l1[k], win ), R.l2[k] = __shfl_sync( 0xffffffffu, l2[k], win );
		R.r1[k] = __shfl_sync( 0xffffffffu, r1[k], win ), R.r2[k] = __shfl_sync( 0xffffffffu, r2[k], win );
	}
	return R;
}

// The reference partitions in place with a sequential swap-to-end loop (tiny_bvh.h:2414-2422).  Its result is a fixed
// permutation of the node's range, reproduced here in closed form.  With n = range length, L = number of "left"
// elements, F = positions [0,L), B = positions [L,n) read backwards, m = number of right elements in F (= number of
// left elements in B), BL_k = position of the k-th left element of B in backward order:
//   left element in F                      stays;
//   k-th right element of F (FR_k)          goes to n-1 (k=0) or BL_{k-1}-1, and its slot receives the element at BL_k;
//   the element at position L, if right     behaves as FR_m;
//   any other right element of B at rel     goes to n-1-r,  r = min(l+1, mx) + (n-1-rel) - l,
//                                           l = left elements behind it (positions > rel), mx = m (+1 if FR_m exists).
// (tools/partition_check.py proves the equivalence against the sequential loop by exhaustive random testing.)
// Returns the destination (relative) of the element at `rel`; *pull is the relative position whose element moves INTO
// `rel` when rel is a front-right slot (else 0xffffffff); returns 0xffffffff when the element is moved by its puller.
__device__ __forceinline__ uint32_t partition_dest( const uint32_t rel, const uint32_t n, const uint32_t L, const bool is_left,
	const uint32_t lefts_before /* in [0,rel) */, const uint32_t m, const bool extra /* element at L is right */,
	const uint32_t* pos_bl /* relative positions of BL_k */, uint32_t* pull )
{
	*pull = 0xffffffffu;
	if (rel < L)
	{
		if (is_left) return rel;
		const uint32_t k = rel - lefts_before; // rights before rel in F
		*pull = pos_bl[k];
		return k == 0 ? n - 1 : pos_bl[k - 1] - 1;
	}
	if (is_left) return 0xffffffffu; // a back-left is pulled by its front-right slot
	if (rel == L) return m == 0 ? n - 1 : pos_bl[m - 1] - 1;
	const uint32_t l = L - lefts_before; // lefts at positions > rel (rel itself is right)
	const uint32_t mx = m + (extra ? 1u : 0u);
	const uint32_t r = min( l + 1, mx ) + (n - 1 - rel) - l;
	return n - 1 - r;
}

// Warp-aggregated update of a bin table held in shared memory: lanes that fall into the same bin first reduce their
// six box keys with REDUX (match.any + redux.sync.min/max), then ONE lane per distinct bin issues the seven shared
// atomics.  Neighbouring primitives usually share a bin, so this cuts the shared-atomic traffic (the limiter of the
// per-primitive version: 73 % L1TEX at 7 % issue, profiles/r1_build_ncu.txt) by an order of magnitude.
// Lanes without a primitive pass valid = false (they join the votes with neutral values).
__device__ __forceinline__ void bin_update_aggregated( uint32_t* bins /* one axis: BINS * 7 words */, const bool valid, const uint32_t bin,
	const uint32_t kmn0, const uint32_t kmn1, const uint32_t kmn2, const uint32_t kmx0, const uint32_t kmx1, const uint32_t kmx2 )
{
	const uint32_t key = valid ? bin : 0xffu;
	const uint32_t m = __match_any_sync( 0xffffffffu, key );
	const uint32_t a0 = __reduce_min_sync( m, kmn0 ), a1 = __reduce_min_sync( m, kmn1 ), a2 = __reduce_min_sync( m, kmn2 );
	const uint32_t b0 = __reduce_max_sync( m, kmx0 ), b1 = __reduce_max_sync( m, kmx1 ), b2 = __reduce_max_sync( m, kmx2 );
	if (valid && (threadIdx.x & 31) == (uint32_t)(__ffs( m ) - 1))
	{
		uint32_t* w = bins + bin * 7;
		atomicMin( w + 0, a0 ), atomicMin( w + 1, a1 ), atomicMin( w + 2, a2 );
		atomicMax( w + 3, b0 ), atomicMax( w + 4, b1 ), atomicMax( w + 5, b2 );
		atomicAdd( w + 6, (uint32_t)__popc( m ) );
	}
}

// ---------------------------------------------------------------------------------------------- fragments

__global__ void __launch_bounds__( 256 ) k_fragments( BuildArgs A )
{
	// PrepareBuild :2300-2308: bmin = min(v0, min(v1, v2)), bmax likewise; root box = union; primIdx[i] = i
	const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
	float mn[3] = { BVH_FAR, BVH_FAR, BVH_FAR }, mx[3] = { -BVH_FAR, -BVH_FAR, -BVH_FAR };
	if (i < A.n && A.aabbs)
	{
		const float4 lo = __ldg( A.aabbs + (size_t)i * 2 ), hi = __ldg( A.aabbs + (size_t)i * 2 + 1 );
		mn[0] = lo.x, mn[1] = lo.y, mn[2] = lo.z, mx[0] = hi.x, mx[1] = hi.y, mx[2] = hi.z;
		A.frag_min[i] = make_float4( mn[0], mn[1], mn[2], 0 ), A.frag_max[i] = make_float4( mx[0], mx[1], mx[2], 0 );
		A.idx[0][i] = i;
	}
	else if (i < A.n)
	{
		const float4 v0 = __ldg( A.verts + (size_t)i * 3 ), v1 = __ldg( A.verts + (size_t)i * 3 + 1 ), v2 = __ldg( A.verts + (size_t)i * 3 + 2 );
		mn[0] = fminf( v0.x, fminf( v1.x, v2.x ) ), mn[1] = fminf( v0.y, fminf( v1.y, v2.y ) ), mn[2] = fminf( v0.z, fminf( v1.z, v2.z ) );
		mx[0] = fmaxf( v0.x, fmaxf( v1.x, v2.x ) ), mx[1] = fmaxf( v0.y, fmaxf( v1.y, v2.y ) ), mx[2] = fmaxf( v0.z, fmaxf( v1.z, v2.z ) );
		A.frag_min[i] = make_float4( mn[0], mn[1], mn[2], 0 ), A.frag_max[i] = make_float4( mx[0], mx[1], mx[2], 0 );
		A.idx[0][i] = i;
	}
	#pragma unroll
	for (int k = 0; k < 3; k++) for (int o = 16; o > 0; o >>= 1)
		mn[k] = fminf( mn[k], __shfl_xor_sync( 0xffffffffu, mn[k], o ) ), mx[k] = fmaxf( mx[k], __shfl_xor_sync( 0xffffffffu, mx[k], o ) );
	__shared__ uint32_t s_key[6];
	if (threadIdx.x < 3) s_key[threadIdx.x] = 0xffffffffu; else if (threadIdx.x < 6) s_key[threadIdx.x] = 0;
	__syncthreads();
	if ((threadIdx.x & 31) == 0)
		for (int k = 0; k < 3; k++) atomicMin( &s_key[k], f2key( mn[k] ) ), atomicMax( &s_key[3 + k], f2key( mx[k] ) );
	__syncthreads();
	if (threadIdx.x < 3) atomicMin( &A.ctr->root_key[threadIdx.x], s_key[threadIdx.x] );
	else if (threadIdx.x < 6) atomicMax( &A.ctr->root_key[threadIdx.x], s_key[threadIdx.x] );
}

__global__ void k_init_counters( BuildArgs A )
{
	Counters* c = A.ctr;
	c->tmp_nodes = 2, c->next_large = 0, c->small_roots = 0, c->max_depth = 0, c->total_chunks = 0, c->lvl_num[0] = c->lvl_num[1] = 0, c->lvl_chunks[0] = c->lvl_chunks[1] = 0, c->levels = 0;
	for (int k = 0; k < 3; k++) c->root_key[k] = 0xffffffffu, c->root_key[3 + k] = 0;
}

__global__ void k_init_root( BuildArgs A )
{
	Counters* c = A.ctr;
	const float4 mn = make_float4( key2f( c->root_key[0] ), key2f( c->root_key[1] ), key2f( c->root_key[2] ), __uint_as_float( 0u ) );
	const float4 mx = make_float4( key2f( c->root_key[3] ), key2f( c->root_key[4] ), key2f( c->root_key[5] ), __uint_as_float( A.n ) );
	A.tmp_nodes[0] = mn, A.tmp_nodes[1] = mx;
	A.tmp_nodes[2] = make_float4( 0, 0, 0, 0 ), A.tmp_nodes[3] = make_float4( 0, 0, 0, 0 ); // node 1 stays unused (:2285)
	A.node_first[0] = 0, A.node_depth[0] = 0, A.node_first[1] = 0, A.node_depth[1] = 0;
	if (A.n > A.small_t)
	{
		A.lvl[0][0] = LargeNode{ 0, 0, A.n, 0 };
		A.chunk_start[0] = 0, A.chunk_start[1] = (A.n + CHUNK - 1) / CHUNK;
		c->total_chunks = (A.n + CHUNK - 1) / CHUNK, c->lvl_num[0] = 1, c->lvl_chunks[0] = (A.n + CHUNK - 1) / CHUNK;
		for (int k = threadIdx.x; k < BIN_STRIDE; k += blockDim.x) A.bins[k] = bin_init_word( k );
	}
	else if (threadIdx.x == 0)
	{
		A.small[0] = SmallRoot{ 0, 0, A.n, 0 };
		c->small_roots = 1;
	}
}

// ---------------------------------------------------------------------------------------------- large phase

// chunk c of the current level -> (slot j in the node list, first offset inside the node)
__device__ __forceinline__ uint32_t find_slot( const uint32_t* chunk_start, const uint32_t num, const uint32_t c )
{
	uint32_t lo = 0, hi = num; // largest j with chunk_start[j] <= c
	while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (chunk_start[mid] <= c) lo = mid; else hi = mid; }
	return lo;
}

// The per-chunk / per-node bodies of the large phase are device functions over a VIRTUAL block index `vb`: the launch-per-stage
// path calls them with blockIdx.x, the persistent path (k_large_phase) loops them over the level's chunks between grid-wide
// barriers.  Inside the persistent kernel the arrays they read were written earlier in the same launch, so none of these loads
// may take the read-only (.nc) path: LD() is a plain load there.
#define LD( p ) (*(p))
__device__ __forceinline__ void bin_chunk( const BuildArgs& A, const uint32_t* cs, const LargeNode* cur, const uint32_t num, const uint32_t* idx_in, const uint32_t vb, uint32_t* s_bins, uint32_t& s_slot )
{
	// binning :2357-2376 for one 256-primitive chunk of one node: shared-memory table, then one flush per CTA
	__syncthreads(); // the previous user of s_bins / s_slot (an earlier chunk of this CTA) is done
	if (threadIdx.x == 0) s_slot = find_slot( cs, num, vb );
	for (int k = threadIdx.x; k < BIN_STRIDE; k += CHUNK) s_bins[k] = bin_init_word( k );
	__syncthreads();
	const uint32_t j = s_slot;
	const LargeNode nd = cur[j];
	const uint32_t off = (vb - LD( cs + j )) * CHUNK + threadIdx.x;
	const bool valid = off < nd.count;
	uint32_t b3[3] = { 0, 0, 0 }, kmn[3] = { 0xffffffffu, 0xffffffffu, 0xffffffffu }, kmx[3] = { 0, 0, 0 };
	if (valid)
	{
		const float4 nmin = LD( A.tmp_nodes + (size_t)nd.tmp * 2 ), nmax = LD( A.tmp_nodes + (size_t)nd.tmp * 2 + 1 );
		const uint32_t p = nd.first + off, fi = LD( idx_in + p );
		const float4 fmn = __ldg( A.frag_min + fi ), fmx = __ldg( A.frag_max + fi ); // fragments are written by an earlier launch
		if (A.flavour)
		{
			const float rx = rpd_avx( __fsub_rn( nmax.x, nmin.x ) ), ry = rpd_avx( __fsub_rn( nmax.y, nmin.y ) ), rz = rpd_avx( __fsub_rn( nmax.z, nmin.z ) );
			const float mx2 = __fmul_rn( nmin.x, 2.0f ), my2 = __fmul_rn( nmin.y, 2.0f ), mz2 = __fmul_rn( nmin.z, 2.0f );
			b3[0] = bin_of_avx( fmn.x, fmx.x, mx2, rx ), b3[1] = bin_of_avx( fmn.y, fmx.y, my2, ry ), b3[2] = bin_of_avx( fmn.z, fmx.z, mz2, rz );
			// the partition's bins: what k_flags compares with the split plane, and what sizes the children
			const uint32_t p0 = bin_part_avx( fmn.x, fmx.x, mx2, rx ), p1 = bin_part_avx( fmn.y, fmx.y, my2, ry ), p2 = bin_part_avx( fmn.z, fmx.z, mz2, rz );
			A.bin_ids[p] = (uint16_t)(p0 | (p1 << 3) | (p2 << 6));
			atomicAdd( s_bins + BIN_WORDS + p0, 1u ), atomicAdd( s_bins + BIN_WORDS + BINS + p1, 1u ), atomicAdd( s_bins + BIN_WORDS + 2 * BINS + p2, 1u );
		}
		else
		{
			b3[0] = bin_of( fmn.x, fmx.x, nmin.x, __fdiv_rn( (float)BINS, __fsub_rn( nmax.x, nmin.x ) ) );
			b3[1] = bin_of( fmn.y, fmx.y, nmin.y, __fdiv_rn( (float)BINS, __fsub_rn( nmax.y, nmin.y ) ) );
			b3[2] = bin_of( fmn.z, fmx.z, nmin.z, __fdiv_rn( (float)BINS, __fsub_rn( nmax.z, nmin.z ) ) );
			A.bin_ids[p] = (uint16_t)(b3[0] | (b3[1] << 3) | (b3[2] << 6));
		}
		kmn[0] = f2key( fmn.x ), kmn[1] = f2key( fmn.y ), kmn[2] = f2key( fmn.z ), kmx[0] = f2key( fmx.x ), kmx[1] = f2key( fmx.y ), kmx[2] = f2key( fmx.z );
	}
	#pragma unroll
	for (int a = 0; a < 3; a++) bin_update_aggregated( s_bins + a * BINS * 7, valid, b3[a], kmn[0], kmn[1], kmn[2], kmx[0], kmx[1], kmx[2] );
	__syncthreads();
	if (threadIdx.x < BIN_WORDS)
	{
		const uint32_t k = threadIdx.x, bin = k / 7, f = k % 7;
		if (s_bins[bin * 7 + 6] != 0)
		{
			uint32_t* g = A.bins + (size_t)j * BIN_STRIDE + k;
			if (f < 3) atomicMin( g, s_bins[k] ); else if (f < 6) atomicMax( g, s_bins[k] ); else atomicAdd( g, s_bins[k] );
		}
	}
	else if (threadIdx.x < BIN_STRIDE && A.flavour && s_bins[threadIdx.x] != 0) atomicAdd( A.bins + (size_t)j * BIN_STRIDE + threadIdx.x, s_bins[threadIdx.x] );
}
__global__ void __launch_bounds__( CHUNK ) k_bin( BuildArgs A, const LargeNode* cur, const uint32_t num, const uint32_t* idx_in )
{
	__shared__ uint32_t s_bins[BIN_STRIDE];
	__shared__ uint32_t s_slot;
	bin_chunk( A, A.chunk_start, cur, num, idx_in, blockIdx.x, s_bins, s_slot );
}

// append the two children of a split node: bigger than SMALL_T -> next level's list, else -> warp-built subtree
__device__ __forceinline__ void emit_child( const BuildArgs& A, LargeNode* next, const uint32_t tmp, const uint32_t first, const uint32_t count, const uint32_t depth, const uint32_t out_buf )
{
	if (count > A.small_t) next[atomicAdd( &A.ctr->next_large, 1u )] = LargeNode{ tmp, first, count, depth };
	else A.small[atomicAdd( &A.ctr->small_roots, 1u )] = SmallRoot{ tmp, first, count, depth | (out_buf << 16) };
}

__device__ __forceinline__ void sweep_one( const BuildArgs& A, const LargeNode* cur, LargeNode* next, const uint32_t j, const uint32_t* idx_in, const uint32_t out_buf )
{
	const uint32_t lane = threadIdx.x & 31;
	const LargeNode nd = cur[j];
	const float4 nmin = A.tmp_nodes[(size_t)nd.tmp * 2], nmax = A.tmp_nodes[(size_t)nd.tmp * 2 + 1];
	const float4 rmin = A.tmp_nodes[0], rmax = A.tmp_nodes[1];
	const float mdf = A.flavour ? 1e-7f : 1e-20f; // minDim (:2346 / :6555)
	const float3 min_dim = make_float3( __fmul_rn( __fsub_rn( rmax.x, rmin.x ), mdf ), __fmul_rn( __fsub_rn( rmax.y, rmin.y ), mdf ), __fmul_rn( __fsub_rn( rmax.z, rmin.z ), mdf ) );
	const SweepResult R = sweep_node( A.bins + (size_t)j * BIN_STRIDE, nmin, nmax, nd.count, min_dim, A.c_trav, A.c_int, A.flavour );
	if (!R.split)
	{
		// leaf: its range is final (tiny_bvh.h:2409-2412); publish the order it has in the current buffer
		if (lane == 0) A.split[j] = SplitInfo{ 0, 0, 0, 0 };
		for (uint32_t k = lane; k < nd.count; k += 32) A.idx_final[nd.first + k] = idx_in[nd.first + k];
		return;
	}
	if (lane == 0)
	{
		const uint32_t n = atomicAdd( &A.ctr->tmp_nodes, 2u ), d = nd.depth + 1;
		A.tmp_nodes[(size_t)n * 2] = make_float4( R.l1[0], R.l1[1], R.l1[2], __uint_as_float( nd.first ) );
		A.tmp_nodes[(size_t)n * 2 + 1] = make_float4( R.l2[0], R.l2[1], R.l2[2], __uint_as_float( R.lN ) );
		A.tmp_nodes[(size_t)n * 2 + 2] = make_float4( R.r1[0], R.r1[1], R.r1[2], __uint_as_float( nd.first + R.lN ) );
		A.tmp_nodes[(size_t)n * 2 + 3] = make_float4( R.r2[0], R.r2[1], R.r2[2], __uint_as_float( nd.count - R.lN ) );
		A.node_first[n] = nd.first, A.node_first[n + 1] = nd.first + R.lN, A.node_depth[n] = d, A.node_depth[n + 1] = d;
		// parent becomes interior: leftFirst = child pair, triCount = 0 (:2432)
		A.tmp_nodes[(size_t)nd.tmp * 2].w = __uint_as_float( n ), A.tmp_nodes[(size_t)nd.tmp * 2 + 1].w = __uint_as_float( 0u );
		atomicMax( &A.ctr->max_depth, d );
		A.split[j] = SplitInfo{ 1, R.axis, R.pos, R.lN };
		emit_child( A, next, n, nd.first, R.lN, d, out_buf );
		emit_child( A, next, n + 1, nd.first + R.lN, nd.count - R.lN, d, out_buf );
	}
}
__global__ void __launch_bounds__( 256 ) k_sweep( BuildArgs A, const LargeNode* cur, LargeNode* next, const uint32_t num, const uint32_t* idx_in, const uint32_t out_buf )
{
	const uint32_t j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
	if (j < num) sweep_one( A, cur, next, j, idx_in, out_buf );
}

__device__ __forceinline__ uint32_t flag_of( const BuildArgs& A, const uint32_t* cs, const LargeNode* cur, const uint32_t num, const uint32_t vb, uint32_t& s_slot )
{
	__syncthreads();
	if (threadIdx.x == 0) s_slot = find_slot( cs, num, vb );
	__syncthreads();
	const uint32_t j = s_slot;
	const LargeNode nd = cur[j];
	const SplitInfo sp = A.split[j];
	const uint32_t off = (vb - LD( cs + j )) * CHUNK + threadIdx.x;
	// flags live in CHUNK SPACE (index = chunk * CHUNK + lane): the scan then costs O(active primitives) per level, and a
	// node's flags stay contiguous because its chunks are; padding lanes of a node's last chunk carry 0
	const uint32_t p = nd.first + off;
	return (off < nd.count && sp.did && ((((uint32_t)A.bin_ids[p]) >> (3 * sp.axis)) & 7u) <= sp.pos) ? 1u : 0u;
}
__global__ void __launch_bounds__( CHUNK ) k_flags( BuildArgs A, const LargeNode* cur, const uint32_t num )
{
	__shared__ uint32_t s_slot;
	A.flags[(size_t)blockIdx.x * CHUNK + threadIdx.x] = flag_of( A, A.chunk_start, cur, num, blockIdx.x, s_slot );
}

// exclusive scan of flags[0..n) into scan[0..n] (scan[n] = total): tile sums, one-block spine, apply
__global__ void __launch_bounds__( 256 ) k_scan_tiles( const uint32_t* __restrict__ in, uint32_t* __restrict__ tile_sum, const uint32_t n )
{
	__shared__ uint32_t s[8];
	const uint32_t base = blockIdx.x * SCAN_TILE;
	uint32_t v = 0;
	for (uint32_t k = threadIdx.x; k < SCAN_TILE; k += 256) if (base + k < n) v += in[base + k];
	for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync( 0xffffffffu, v, o );
	if ((threadIdx.x & 31) == 0) s[threadIdx.x >> 5] = v;
	__syncthreads();
	if (threadIdx.x == 0) { uint32_t t = 0; for (int k = 0; k < 8; k++) t += s[k]; tile_sum[blockIdx.x] = t; }
}

__global__ void __launch_bounds__( 1024 ) k_scan_spine( uint32_t* tile_sum, const uint32_t tiles )
{
	// in-place exclusive scan of tile sums by one block
	__shared__ uint32_t s_warp[32];
	__shared__ uint32_t s_carry;
	if (threadIdx.x == 0) s_carry = 0;
	__syncthreads();
	for (uint32_t base = 0; base < tiles; base += 1024)
	{
		const uint32_t i = base + threadIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
		const uint32_t v = i < tiles ? tile_sum[i] : 0;
		uint32_t x = v;
		for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync( 0xffffffffu, x, o ); if (lane >= o) x += y; }
		if (lane == 31) s_warp[w] = x;
		__syncthreads();
		if (w == 0)
		{
			uint32_t t = s_warp[lane];
			for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync( 0xffffffffu, t, o ); if (lane >= o) t += y; }
			s_warp[lane] = t; // inclusive over warps
		}
		__syncthreads();
		const uint32_t carry = s_carry, wbase = w ? s_warp[w - 1] : 0;
		if (i < tiles) tile_sum[i] = carry + wbase + x - v;
		__syncthreads();
		if (threadIdx.x == 1023) s_carry = carry + wbase + x;
		__syncthreads();
	}
}

__global__ void __launch_bounds__( 256 ) k_scan_apply( const uint32_t* __restrict__ in, const uint32_t* __restrict__ tile_sum, uint32_t* __restrict__ out, const uint32_t n )
{
	// each thread owns 8 consecutive elements of the 2048-element tile
	__shared__ uint32_t s_warp[8];
	const uint32_t base = blockIdx.x * SCAN_TILE + threadIdx.x * 8, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
	uint32_t v[8], t = 0;
	#pragma unroll
	for (int k = 0; k < 8; k++) { v[k] = base + k < n ? in[base + k] : 0; t += v[k]; }
	uint32_t x = t;
	for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync( 0xffffffffu, x, o ); if (lane >= o) x += y; }
	if (lane == 31) s_warp[w] = x;
	__syncthreads();
	uint32_t wbase = 0;
	for (uint32_t k = 0; k < w; k++) wbase += s_warp[k];
	uint32_t run = tile_sum[blockIdx.x] + wbase + x - t;
	#pragma unroll
	for (int k = 0; k < 8; k++) { if (base + k < n) out[base + k] = run; run += v[k]; }
	if (base < n && base + 8 >= n) out[n] = run; // the thread holding the last element publishes the total
}

// exclusive prefix of the flags at chunk-space index i.  PERSIST = false: A.scan holds the global scan (exclusive_scan);
// PERSIST = true: A.scan holds the prefix inside each chunk and A.chunk_pre the exclusive prefix over chunk totals.
template <bool PERSIST> __device__ __forceinline__ uint32_t scan_at( const BuildArgs& A, const size_t i )
{
	return PERSIST ? A.chunk_pre[i / CHUNK] + A.scan[i] : A.scan[i];
}
template <bool PERSIST> __device__ __forceinline__ void posbl_chunk( const BuildArgs& A, const uint32_t* cs, const LargeNode* cur, const uint32_t num, const uint32_t vb, uint32_t& s_slot )
{
	__syncthreads();
	if (threadIdx.x == 0) s_slot = find_slot( cs, num, vb );
	__syncthreads();
	const uint32_t j = s_slot;
	const LargeNode nd = cur[j];
	const SplitInfo sp = A.split[j];
	const uint32_t off = (vb - LD( cs + j )) * CHUNK + threadIdx.x;
	if (!sp.did || off >= nd.count || off < sp.L) return;
	const size_t sb = (size_t)LD( cs + j ) * CHUNK; // this node's base in chunk space
	if (A.flags[sb + off]) A.pos_bl[nd.first + (scan_at<PERSIST>( A, sb + nd.count ) - scan_at<PERSIST>( A, sb + off + 1 ))] = off; // BL_k, k = lefts behind it
}
__global__ void __launch_bounds__( CHUNK ) k_posbl( BuildArgs A, const LargeNode* cur, const uint32_t num )
{
	__shared__ uint32_t s_slot;
	posbl_chunk<false>( A, A.chunk_start, cur, num, blockIdx.x, s_slot );
}

template <bool PERSIST> __device__ __forceinline__ void scatter_chunk( const BuildArgs& A, const uint32_t* cs, const LargeNode* cur, const uint32_t num, const uint32_t* idx_in, uint32_t* idx_out, const uint32_t vb, uint32_t& s_slot )
{
	__syncthreads();
	if (threadIdx.x == 0) s_slot = find_slot( cs, num, vb );
	__syncthreads();
	const uint32_t j = s_slot;
	const LargeNode nd = cur[j];
	const SplitInfo sp = A.split[j];
	const uint32_t off = (vb - LD( cs + j )) * CHUNK + threadIdx.x;
	if (!sp.did || off >= nd.count) return;
	const size_t sb = (size_t)LD( cs + j ) * CHUNK; // this node's base in chunk space
	const uint32_t p = nd.first + off, s0 = scan_at<PERSIST>( A, sb );
	const uint32_t lefts_before = scan_at<PERSIST>( A, sb + off ) - s0, lefts_in_F = scan_at<PERSIST>( A, sb + sp.L ) - s0;
	const uint32_t m = sp.L - lefts_in_F;
	const bool extra = sp.L < nd.count && A.flags[sb + sp.L] == 0;
	uint32_t pull;
	const uint32_t dest = partition_dest( off, nd.count, sp.L, A.flags[sb + off] != 0, lefts_before, m, extra, A.pos_bl + nd.first, &pull );
	if (dest != 0xffffffffu) idx_out[nd.first + dest] = idx_in[p];
	if (pull != 0xffffffffu) idx_out[p] = idx_in[nd.first + pull];
}
__global__ void __launch_bounds__( CHUNK ) k_scatter( BuildArgs A, const LargeNode* cur, const uint32_t num, const uint32_t* idx_in, uint32_t* idx_out )
{
	__shared__ uint32_t s_slot;
	scatter_chunk<false>( A, A.chunk_start, cur, num, idx_in, idx_out, blockIdx.x, s_slot );
}

// next level: chunk offsets (exclusive scan of ceil(count/CHUNK)) and fresh bin tables, by one block
__global__ void __launch_bounds__( 1024 ) k_prepare_level( BuildArgs A, const LargeNode* __restrict__ next )
{
	__shared__ uint32_t s_warp[32];
	__shared__ uint32_t s_carry;
	const uint32_t num = A.ctr->next_large;
	if (threadIdx.x == 0) s_carry = 0;
	__syncthreads();
	for (uint32_t base = 0; base < num; base += 1024)
	{
		const uint32_t i = base + threadIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5;
		const uint32_t v = i < num ? (next[i].count + CHUNK - 1) / CHUNK : 0;
		uint32_t x = v;
		for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync( 0xffffffffu, x, o ); if (lane >= o) x += y; }
		if (lane == 31) s_warp[w] = x;
		__syncthreads();
		if (w == 0)
		{
			uint32_t t = s_warp[lane];
			for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync( 0xffffffffu, t, o ); if (lane >= o) t += y; }
			s_warp[lane] = t;
		}
		__syncthreads();
		const uint32_t carry = s_carry, wbase = w ? s_warp[w - 1] : 0;
		if (i < num) A.chunk_start[i] = carry + wbase + x - v;
		__syncthreads();
		if (threadIdx.x == 1023) s_carry = carry + wbase + x;
		__syncthreads();
	}
	if (threadIdx.x == 0) A.chunk_start[num] = s_carry, A.ctr->total_chunks = s_carry;
}

__global__ void k_bins_init( uint32_t* bins, const uint32_t words )
{
	const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
	if (k < words) bins[k] = bin_init_word( k % BIN_STRIDE );
}

// ---------------------------------------------------------------------------------------------- persistent large phase
// The whole level loop in ONE cooperative launch: every stage of a level is a grid-stride loop over the level's chunks / nodes,
// stages are separated by grid-wide barriers (cooperative groups), and the level bookkeeping that the launch-per-stage path
// reads back to the host (how many nodes / chunks the next level has) stays in device memory.  A level costs six barriers
// instead of eleven launches and a host round trip.
#include <cooperative_groups.h>
namespace cg = cooperative_groups;

// block-wide exclusive scan helper for 256 threads: returns the exclusive prefix of v and, in `total`, the block total
__device__ __forceinline__ uint32_t block_exscan_256( const uint32_t v, uint32_t* s_warp /* 8 */, uint32_t& total )
{
	const uint32_t lane = threadIdx.x & 31, w = threadIdx.x >> 5;
	uint32_t x = v;
	for (int o = 1; o < 32; o <<= 1) { const uint32_t y = __shfl_up_sync( 0xffffffffu, x, o ); if (lane >= o) x += y; }
	__syncthreads();
	if (lane == 31) s_warp[w] = x;
	__syncthreads();
	uint32_t wbase = 0, t = 0;
	#pragma unroll
	for (uint32_t k = 0; k < 8; k++) { const uint32_t sw = s_warp[k]; if (k < w) wbase += sw; t += sw; }
	total = t;
	return wbase + x - v;
}

__global__ void __launch_bounds__( CHUNK ) k_large_phase( BuildArgs A )
{
	cg::grid_group grid = cg::this_grid();
	__shared__ uint32_t s_bins[BIN_STRIDE];
	__shared__ uint32_t s_slot, s_carry;
	__shared__ uint32_t s_warp[8];
	Counters* C = A.ctr;
	uint32_t* const chunk_start0 = A.chunk_start;
	const uint32_t warps_per_block = CHUNK / 32, gwarp = blockIdx.x * warps_per_block + (threadIdx.x >> 5), gwarps = gridDim.x * warps_per_block;
	for (uint32_t level = 0; level < 4096; level++)
	{
		// level state is kept per parity (this level reads [level & 1], stage 4 writes [(level + 1) & 1]): no hand-over stage
		const uint32_t par = level & 1;
		const uint32_t num = C->lvl_num[par], chunks = C->lvl_chunks[par];
		if (num == 0) break; // uniform over the grid: written before the last barrier
		const uint32_t* const cs = par ? A.chunk_start_next : chunk_start0;
		uint32_t* const chunk_start_out = par ? chunk_start0 : A.chunk_start_next;
		const uint32_t lp = (A.level0 + level) & 1; // parity of the ping-pong node lists / index buffers (absolute level)
		const LargeNode* cur = A.lvl[lp];
		LargeNode* next = A.lvl[lp ^ 1];
		const uint32_t* idx_in = A.idx[lp];
		uint32_t* idx_out = A.idx[lp ^ 1];
		// ---- 1. bin tables of the level's nodes
		for (uint32_t c = blockIdx.x; c < chunks; c += gridDim.x) bin_chunk( A, cs, cur, num, idx_in, c, s_bins, s_slot );
		grid.sync();
		// ---- 2. one warp per node: sweep, termination, children
		for (uint32_t j = gwarp; j < num; j += gwarps) sweep_one( A, cur, next, j, idx_in, lp ^ 1 );
		grid.sync();
		// ---- 3. left / right flags in chunk space + their prefix inside each chunk + the chunk totals
		for (uint32_t c = blockIdx.x; c < chunks; c += gridDim.x)
		{
			const uint32_t f = flag_of( A, cs, cur, num, c, s_slot );
			uint32_t total;
			const uint32_t pre = block_exscan_256( f, s_warp, total );
			A.flags[(size_t)c * CHUNK + threadIdx.x] = f, A.scan[(size_t)c * CHUNK + threadIdx.x] = pre;
			if (threadIdx.x == 0) A.chunk_pre[c] = total;
		}
		grid.sync();
		// ---- 4. block 0: exclusive prefix over the chunk totals; block 1 (or 0): the next level's chunk offsets; all: fresh bin tables
		const uint32_t num_next = C->next_large;
		if (blockIdx.x == 0)
		{
			if (threadIdx.x == 0) s_carry = 0;
			__syncthreads();
			for (uint32_t base = 0; base < chunks; base += CHUNK)
			{
				const uint32_t i = base + threadIdx.x;
				const uint32_t v = i < chunks ? A.chunk_pre[i] : 0;
				uint32_t total;
				const uint32_t pre = block_exscan_256( v, s_warp, total );
				const uint32_t carry = s_carry;
				if (i < chunks) A.chunk_pre[i] = carry + pre;
				__syncthreads();
				if (threadIdx.x == 0) s_carry = carry + total;
				__syncthreads();
			}
			if (threadIdx.x == 0) A.chunk_pre[chunks] = s_carry, A.scan[(size_t)chunks * CHUNK] = 0; // scan_at( chunks * CHUNK ) = total
		}
		if (blockIdx.x == (gridDim.x > 1 ? 1u : 0u))
		{
			// chunk offsets of the next level: exclusive scan of ceil( count / CHUNK ) into a second array (the current one is
			// still needed by stages 5 and 6); swapped in after the last barrier of the level
			__syncthreads();
			if (threadIdx.x == 0) s_carry = 0;
			__syncthreads();
			for (uint32_t base = 0; base < num_next; base += CHUNK)
			{
				const uint32_t i = base + threadIdx.x;
				const uint32_t v = i < num_next ? (next[i].count + CHUNK - 1) / CHUNK : 0;
				uint32_t total;
				const uint32_t pre = block_exscan_256( v, s_warp, total );
				const uint32_t carry = s_carry;
				if (i < num_next) chunk_start_out[i] = carry + pre;
				__syncthreads();
				if (threadIdx.x == 0) s_carry = carry + total;
				__syncthreads();
			}
			if (threadIdx.x == 0) chunk_start_out[num_next] = s_carry, C->lvl_num[par ^ 1] = num_next, C->lvl_chunks[par ^ 1] = s_carry, C->levels = level + 1;
		}
		// the bin tables were consumed in stage 2: re-arm them for the next level's nodes
		for (uint32_t k = blockIdx.x * CHUNK + threadIdx.x; k < num_next * BIN_STRIDE; k += gridDim.x * CHUNK) A.bins[k] = bin_init_word( k % BIN_STRIDE );
		grid.sync();
		// ---- 5. positions of the lefts behind the split point (every block has read next_large by now: re-arm it for the next level's sweep)
		if (blockIdx.x == 0 && threadIdx.x == 0) C->next_large = 0;
		for (uint32_t c = blockIdx.x; c < chunks; c += gridDim.x) posbl_chunk<true>( A, cs, cur, num, c, s_slot );
		grid.sync();
		// ---- 6. the swap partition as a permutation into the other index buffer
		for (uint32_t c = blockIdx.x; c < chunks; c += gridDim.x) scatter_chunk<true>( A, cs, cur, num, idx_in, idx_out, c, s_slot );
		grid.sync();
	}
}

// ---------------------------------------------------------------------------------------------- small subtrees

#define SMALL_WARPS 8
struct SmallSmem
{
	uint32_t gid[SMALL_T];            // global primitive index of each local slot
	uint16_t idx[2][SMALL_T];         // ping-pong order of local slots
	uint16_t bid[SMALL_T];
	uint16_t posbl[SMALL_T];
	uint32_t fw[SMALL_T / 32];
	uint32_t bins[BIN_STRIDE];
	uint32_t st_tmp[12]; uint32_t st_rng[12]; uint32_t st_db[12]; // stack: tmp node, lo | n << 16, depth | buf << 16
};

__global__ void __launch_bounds__( SMALL_WARPS * 32 ) k_build_small( BuildArgs A, const uint32_t num_roots )
{
	// One warp builds a whole subtree of <= SMALL_T primitives: the reference's loop (:2347-2445) with the primitives
	// of the current node spread over the lanes.  The smaller child is continued, the larger pushed, so the stack
	// stays below log2(SMALL_T)+2 entries; order of work does not matter because numbering is fixed afterwards.
	__shared__ SmallSmem S_all[SMALL_WARPS];
	const uint32_t wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const uint32_t r = blockIdx.x * SMALL_WARPS + wid;
	if (r >= num_roots) return;
	SmallSmem& S = S_all[wid];
	const SmallRoot root = A.small[r];
	const uint32_t* src = A.idx[root.depth_buf >> 16];
	for (uint32_t k = lane; k < root.count; k += 32) S.gid[k] = src[root.first + k], S.idx[0][k] = (uint16_t)k;
	const float4 rmin = A.tmp_nodes[0], rmax = A.tmp_nodes[1];
	const float mdf = A.flavour ? 1e-7f : 1e-20f; // minDim (:2346 / :6555)
	const float3 min_dim = make_float3( __fmul_rn( __fsub_rn( rmax.x, rmin.x ), mdf ), __fmul_rn( __fsub_rn( rmax.y, rmin.y ), mdf ), __fmul_rn( __fsub_rn( rmax.z, rmin.z ), mdf ) );
	uint32_t sp = 0, local_max_depth = 0;
	uint32_t tmp = root.tmp, lo = 0, n = root.count, depth = root.depth_buf & 0xffffu, buf = 0;
	__syncwarp();
	while (true)
	{
		// ---- bin the node's primitives (:2357-2376)
		for (uint32_t k = lane; k < BIN_STRIDE; k += 32) S.bins[k] = bin_init_word( k );
		__syncwarp();
		const float4 nmin = A.tmp_nodes[(size_t)tmp * 2], nmax = A.tmp_nodes[(size_t)tmp * 2 + 1];
		const float ex_ = __fsub_rn( nmax.x, nmin.x ), ey_ = __fsub_rn( nmax.y, nmin.y ), ez_ = __fsub_rn( nmax.z, nmin.z );
		const float rpx = A.flavour ? rpd_avx( ex_ ) : __fdiv_rn( (float)BINS, ex_ ), rpy = A.flavour ? rpd_avx( ey_ ) : __fdiv_rn( (float)BINS, ey_ ), rpz = A.flavour ? rpd_avx( ez_ ) : __fdiv_rn( (float)BINS, ez_ );
		const float mx2 = __fmul_rn( nmin.x, 2.0f ), my2 = __fmul_rn( nmin.y, 2.0f ), mz2 = __fmul_rn( nmin.z, 2.0f );
		for (uint32_t k = lane; k < n; k += 32)
		{
			const uint32_t sl = S.idx[buf][lo + k];
			const float4 mn = __ldg( A.frag_min + S.gid[sl] ), mx = __ldg( A.frag_max + S.gid[sl] );
			uint32_t b3[3];
			if (A.flavour)
			{
				b3[0] = bin_of_avx( mn.x, mx.x, mx2, rpx ), b3[1] = bin_of_avx( mn.y, mx.y, my2, rpy ), b3[2] = bin_of_avx( mn.z, mx.z, mz2, rpz );
				const uint32_t p0 = bin_part_avx( mn.x, mx.x, mx2, rpx ), p1 = bin_part_avx( mn.y, mx.y, my2, rpy ), p2 = bin_part_avx( mn.z, mx.z, mz2, rpz );
				S.bid[lo + k] = (uint16_t)(p0 | (p1 << 3) | (p2 << 6));
				atomicAdd( S.bins + BIN_WORDS + p0, 1u ), atomicAdd( S.bins + BIN_WORDS + BINS + p1, 1u ), atomicAdd( S.bins + BIN_WORDS + 2 * BINS + p2, 1u );
			}
			else
			{
				b3[0] = bin_of( mn.x, mx.x, nmin.x, rpx ), b3[1] = bin_of( mn.y, mx.y, nmin.y, rpy ), b3[2] = bin_of( mn.z, mx.z, nmin.z, rpz );
				S.bid[lo + k] = (uint16_t)(b3[0] | (b3[1] << 3) | (b3[2] << 6));
			}
			const uint32_t kmn[3] = { f2key( mn.x ), f2key( mn.y ), f2key( mn.z ) }, kmx[3] = { f2key( mx.x ), f2key( mx.y ), f2key( mx.z ) };
			#pragma unroll
			for (int a = 0; a < 3; a++)
			{
				uint32_t* w = S.bins + (a * BINS + b3[a]) * 7;
				atomicMin( w + 0, kmn[0] ), atomicMin( w + 1, kmn[1] ), atomicMin( w + 2, kmn[2] );
				atomicMax( w + 3, kmx[0] ), atomicMax( w + 4, kmx[1] ), atomicMax( w + 5, kmx[2] );
				atomicAdd( w + 6, 1u );
			}
		}
		__syncwarp();
		const SweepResult R = sweep_node( S.bins, nmin, nmax, n, min_dim, A.c_trav, A.c_int, A.flavour );
		bool pop = false;
		if (!R.split)
		{
			for (uint32_t k = lane; k < n; k += 32) A.idx_final[root.first + lo + k] = S.gid[S.idx[buf][lo + k]];
			pop = true;
		}
		else
		{
			// ---- partition into the other buffer (:2414-2422 as a permutation, see partition_dest)
			const uint32_t L = R.lN, batches = (n + 31) >> 5;
			for (uint32_t bch = 0; bch < batches; bch++)
			{
				const uint32_t k = bch * 32 + lane;
				const bool fl = k < n && ((((uint32_t)S.bid[lo + k]) >> (3 * R.axis)) & 7u) <= R.pos;
				const uint32_t wv = __ballot_sync( 0xffffffffu, fl );
				if (lane == 0) S.fw[bch] = wv;
			}
			__syncwarp();
			// lefts in F = popcount of flag bits below L
			uint32_t lefts_in_F = 0;
			for (uint32_t bch = 0; bch * 32 < L; bch++)
			{
				const uint32_t wv = S.fw[bch], hi = L - bch * 32;
				lefts_in_F += __popc( hi >= 32 ? wv : (wv & ((1u << hi) - 1u)) );
			}
			const uint32_t m = L - lefts_in_F;
			const bool extra = L < n && !((S.fw[L >> 5] >> (L & 31)) & 1u);
			// BL_k table: back-lefts, k = number of lefts behind them
			uint32_t run = 0; // lefts before the current batch
			for (uint32_t bch = 0; bch < batches; bch++)
			{
				const uint32_t k = bch * 32 + lane, wv = S.fw[bch];
				const uint32_t before = run + __popc( wv & ((1u << lane) - 1u) );
				if (k < n && k >= L && ((wv >> lane) & 1u)) S.posbl[L - before - 1] = (uint16_t)k;
				run += __popc( wv );
			}
			__syncwarp();
			run = 0;
			const uint32_t ob = buf ^ 1u;
			for (uint32_t bch = 0; bch < batches; bch++)
			{
				const uint32_t k = bch * 32 + lane, wv = S.fw[bch];
				const uint32_t before = run + __popc( wv & ((1u << lane) - 1u) );
				if (k < n)
				{
					uint32_t pull, dest;
					{
						// partition_dest with the 16-bit shared table
						const bool is_left = (wv >> lane) & 1u;
						pull = 0xffffffffu;
						if (k < L)
						{
							if (is_left) dest = k;
							else { const uint32_t q = k - before; pull = S.posbl[q]; dest = q == 0 ? n - 1 : (uint32_t)S.posbl[q - 1] - 1; }
						}
						else if (is_left) dest = 0xffffffffu;
						else if (k == L) dest = m == 0 ? n - 1 : (uint32_t)S.posbl[m - 1] - 1;
						else { const uint32_t l = L - before, mx = m + (extra ? 1u : 0u); dest = n - 1 - (min( l + 1, mx ) + (n - 1 - k) - l); }
					}
					if (dest != 0xffffffffu) S.idx[ob][lo + dest] = S.idx[buf][lo + k];
					if (pull != 0xffffffffu) S.idx[ob][lo + k] = S.idx[buf][lo + pull];
				}
				run += __popc( wv );
			}
			__syncwarp();
			// ---- emit the children (:2426-2432)
			uint32_t cn = 0;
			if (lane == 0)
			{
				cn = atomicAdd( &A.ctr->tmp_nodes, 2u );
				const uint32_t gf = root.first + lo, d = depth + 1;
				A.tmp_nodes[(size_t)cn * 2] = make_float4( R.l1[0], R.l1[1], R.l1[2], __uint_as_float( gf ) );
				A.tmp_nodes[(size_t)cn * 2 + 1] = make_float4( R.l2[0], R.l2[1], R.l2[2], __uint_as_float( L ) );
				A.tmp_nodes[(size_t)cn * 2 + 2] = make_float4( R.r1[0], R.r1[1], R.r1[2], __uint_as_float( gf + L ) );
				A.tmp_nodes[(size_t)cn * 2 + 3] = make_float4( R.r2[0], R.r2[1], R.r2[2], __uint_as_float( n - L ) );
				A.node_first[cn] = gf, A.node_first[cn + 1] = gf + L, A.node_depth[cn] = d, A.node_depth[cn + 1] = d;
				A.tmp_nodes[(size_t)tmp * 2].w = __uint_as_float( cn ), A.tmp_nodes[(size_t)tmp * 2 + 1].w = __uint_as_float( 0u );
			}
			cn = __shfl_sync( 0xffffffffu, cn, 0 );
			__syncwarp(); // child records are re-read by this warp below: make lane 0's global writes visible to the warp
			depth++;
			local_max_depth = max( local_max_depth, depth );
			// continue with the smaller child, push the larger
			const bool left_small = L <= n - L;
			const uint32_t big_tmp = left_small ? cn + 1 : cn, big_lo = left_small ? lo + L : lo, big_n = left_small ? n - L : L;
			if (lane == 0) S.st_tmp[sp] = big_tmp, S.st_rng[sp] = big_lo | (big_n << 16), S.st_db[sp] = depth | (ob << 16);
			sp++;
			tmp = left_small ? cn : cn + 1, lo = left_small ? lo : lo + L, n = left_small ? L : n - L, buf = ob;
			__syncwarp();
		}
		if (pop)
		{
			if (sp == 0) break;
			sp--;
			__syncwarp();
			tmp = S.st_tmp[sp], lo = S.st_rng[sp] & 0xffffu, n = S.st_rng[sp] >> 16, depth = S.st_db[sp] & 0xffffu, buf = S.st_db[sp] >> 16;
			__syncwarp();
		}
	}
	if (lane == 0) atomicMax( &A.ctr->max_depth, local_max_depth );
}

// ---------------------------------------------------------------------------------------------- relayout

// per interior node: count nodes starting at `first`, and the smallest depth among them (head of the left-spine chain)
__global__ void k_rank_count( BuildArgs A, const uint32_t tmp_count, uint32_t* __restrict__ cnt, uint32_t* __restrict__ min_depth )
{
	const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
	if (x >= tmp_count || x == 1) return;
	if (__float_as_uint( A.tmp_nodes[(size_t)x * 2 + 1].w ) != 0) return; // leaf
	const uint32_t f = A.node_first[x];
	atomicAdd( cnt + f, 1u );
	atomicMin( min_depth + f, A.node_depth[x] );
}

// final index of the child pair of interior node x: 2 + 2 * (DFS-preorder rank among interior nodes)
__device__ __forceinline__ uint32_t final_pair( const BuildArgs& A, const uint32_t x, const uint32_t* __restrict__ prefix, const uint32_t* __restrict__ min_depth )
{
	const uint32_t f = A.node_first[x];
	return 2u + 2u * (prefix[f] + A.node_depth[x] - min_depth[f]);
}

__global__ void k_relayout( BuildArgs A, const uint32_t tmp_count, const uint32_t* __restrict__ prefix, const uint32_t* __restrict__ min_depth, float4* __restrict__ out )
{
	const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x;
	if (x >= tmp_count || x == 1) return;
	float4 a = A.tmp_nodes[(size_t)x * 2], b = A.tmp_nodes[(size_t)x * 2 + 1];
	const bool interior = __float_as_uint( b.w ) == 0;
	if (x == 0)
	{
		if (interior) a.w = __uint_as_float( final_pair( A, 0, prefix, min_depth ) );
		out[0] = a, out[1] = b, out[2] = make_float4( 0, 0, 0, 0 ), out[3] = make_float4( 0, 0, 0, 0 );
	}
	if (!interior) return;
	// copy this node's two children to their final pair, re-pointing interior children at their own final pairs
	const uint32_t c = __float_as_uint( A.tmp_nodes[(size_t)x * 2].w ), dst = final_pair( A, x, prefix, min_depth );
	for (uint32_t s = 0; s < 2; s++)
	{
		float4 ca = A.tmp_nodes[(size_t)(c + s) * 2], cb = A.tmp_nodes[(size_t)(c + s) * 2 + 1];
		if (__float_as_uint( cb.w ) == 0) ca.w = __uint_as_float( final_pair( A, c + s, prefix, min_depth ) );
		out[(size_t)(dst + s) * 2] = ca, out[(size_t)(dst + s) * 2 + 1] = cb;
	}
}

// ---------------------------------------------------------------------------------------------- host driver

int exclusive_scan( const uint32_t* in, uint32_t* out, uint32_t* tile_sum, uint32_t n, cudaStream_t s )
{
	const uint32_t tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
	k_scan_tiles<<<tiles, 256, 0, s>>>( in, tile_sum, n );
	LAUNCHED();
	k_scan_spine<<<1, 1024, 0, s>>>( tile_sum, tiles );
	LAUNCHED();
	k_scan_apply<<<tiles, 256, 0, s>>>( in, tile_sum, out, n );
	LAUNCHED();
	return TBVH_OK;
}

#define DEV_ALLOC( ptr, bytes ) do { CUDA_TRY( cudaMalloc( (void**)&(ptr), (bytes) ) ); scratch.push_back( (void*)(ptr) ); } while (0)

int build_sah_launch( tbvh_bvh b, float c_trav, float c_int, int flavour )
{
	const uint32_t n = b->info.prim_count;
	cudaStream_t s = b->ctx->stream;
	std::vector<void*> scratch;
	BuildArgs A = {};
	A.verts = b->d_verts, A.aabbs = b->d_aabbs, A.n = n, A.c_trav = c_trav, A.c_int = c_int, A.flavour = (uint32_t)flavour;
	{
		const int t = b->ctx->small_t; // measured on B200: 128 beats 64 and 256 (profiles/README.md)
		A.small_t = (uint32_t)(t < 8 ? 8 : t > SMALL_T ? SMALL_T : t);
	}
	const size_t max_nodes = (size_t)2 * n + 2, max_large = n / A.small_t + 2;
	int rc = TBVH_OK;
	uint32_t* tile_sum = 0;
	Counters* h_ctr = 0;
	cudaEvent_t e0 = 0, e1 = 0;
	// outputs (kept by the handle)
	CUDA_TRY( cudaMalloc( &b->d_nodes, max_nodes * 32 ) );
	CUDA_TRY( cudaMalloc( &b->d_prim_idx, (size_t)n * 4 ) );
	A.idx_final = b->d_prim_idx;
	auto body = [&]() -> int
	{
		DEV_ALLOC( A.frag_min, (size_t)n * 16 ); DEV_ALLOC( A.frag_max, (size_t)n * 16 );
		DEV_ALLOC( A.idx[0], (size_t)n * 4 ); DEV_ALLOC( A.idx[1], (size_t)n * 4 );
		DEV_ALLOC( A.bin_ids, (size_t)n * 2 );
		// chunk space: at most n / CHUNK + (#large nodes) chunks per level
		const size_t flag_words = (size_t)n + (size_t)CHUNK * (max_large + 1) + 1;
		DEV_ALLOC( A.flags, flag_words * 4 ); DEV_ALLOC( A.scan, flag_words * 4 ); DEV_ALLOC( A.pos_bl, ((size_t)n + 1) * 4 );
		DEV_ALLOC( A.tmp_nodes, max_nodes * 32 ); DEV_ALLOC( A.node_first, max_nodes * 4 ); DEV_ALLOC( A.node_depth, max_nodes * 4 );
		DEV_ALLOC( A.lvl[0], max_large * sizeof( LargeNode ) ); DEV_ALLOC( A.lvl[1], max_large * sizeof( LargeNode ) );
		DEV_ALLOC( A.chunk_start, (max_large + 1) * 4 ); DEV_ALLOC( A.chunk_start_next, (max_large + 1) * 4 ); DEV_ALLOC( A.bins, max_large * BIN_STRIDE * 4 ); DEV_ALLOC( A.split, max_large * sizeof( SplitInfo ) );
		DEV_ALLOC( A.chunk_pre, (flag_words / CHUNK + 2) * 4 );
		DEV_ALLOC( A.small, ((size_t)n + 1) * sizeof( SmallRoot ) );
		DEV_ALLOC( A.ctr, sizeof( Counters ) );
		DEV_ALLOC( tile_sum, (flag_words / SCAN_TILE + 2) * 4 );
		CUDA_TRY( cudaMallocHost( &h_ctr, sizeof( Counters ) ) );
		CUDA_TRY( cudaEventCreate( &e0 ) ); CUDA_TRY( cudaEventCreate( &e1 ) );
		CUDA_TRY( cudaEventRecord( e0, s ) );
		k_init_counters<<<1, 1, 0, s>>>( A ); LAUNCHED();
		k_fragments<<<(n + 255) / 256, 256, 0, s>>>( A ); LAUNCHED();
		k_init_root<<<1, 256, 0, s>>>( A ); LAUNCHED();
		uint32_t num = n > A.small_t ? 1 : 0, chunks = (n + CHUNK - 1) / CHUNK, level = 0;
		// Large phase.  The first levels of a big scene are bandwidth work over all primitives: one launch per stage, every CTA the
		// device can hold.  Once a level is down to a few chunks per SM the stages are launch-latency sized, and the rest of the
		// phase runs inside ONE persistent cooperative launch (k_large_phase) without further host round trips.
		int per_sm = 0;
		uint32_t pgrid = 0;
		if (num && b->ctx->build_mode == 0)
		{
			CUDA_TRY( cudaOccupancyMaxActiveBlocksPerMultiprocessor( &per_sm, k_large_phase, CHUNK, 0 ) );
			if (per_sm > BUILD_CTAS_PER_SM) per_sm = BUILD_CTAS_PER_SM;
			pgrid = (uint32_t)(per_sm > 0 ? per_sm * b->ctx->sm_count : 0);
		}
		const uint32_t persist_chunks = pgrid * 3;
		while (num)
		{
			if (pgrid && chunks <= persist_chunks)
			{
				const uint32_t state[2] = { num, chunks };
				CUDA_TRY( cudaMemcpyAsync( &A.ctr->lvl_num[0], &state[0], 4, cudaMemcpyHostToDevice, s ) );
				CUDA_TRY( cudaMemcpyAsync( &A.ctr->lvl_chunks[0], &state[1], 4, cudaMemcpyHostToDevice, s ) );
				A.level0 = level;
				void* params[] = { (void*)&A };
				const cudaError_t ce = cudaLaunchCooperativeKernel( (const void*)k_large_phase, dim3( pgrid ), dim3( CHUNK ), params, 0, s );
				if (ce == cudaErrorCooperativeLaunchTooLarge || ce == cudaErrorNotSupported || ce == cudaErrorLaunchOutOfResources)
				{
					// this device (or partition of it) cannot keep the persistent grid resident: the launch-per-stage path serves every level
					cudaGetLastError();
					pgrid = 0;
					continue;
				}
				CUDA_TRY( ce );
				g_tbvh_launches++;
				CUDA_TRY( cudaStreamSynchronize( s ) ); // `state` is on this frame
				break;
			}
			const LargeNode* cur = A.lvl[level & 1];
			LargeNode* next = A.lvl[(level + 1) & 1];
			const uint32_t* idx_in = A.idx[level & 1];
			uint32_t* idx_out = A.idx[(level + 1) & 1];
			k_bin<<<chunks, CHUNK, 0, s>>>( A, cur, num, idx_in ); LAUNCHED();
			k_sweep<<<(num * 32 + 255) / 256, 256, 0, s>>>( A, cur, next, num, idx_in, (level + 1) & 1 ); LAUNCHED();
			k_flags<<<chunks, CHUNK, 0, s>>>( A, cur, num ); LAUNCHED();
			{ const int r = exclusive_scan( A.flags, A.scan, tile_sum, chunks * CHUNK, s ); if (r != TBVH_OK) return r; }
			k_posbl<<<chunks, CHUNK, 0, s>>>( A, cur, num ); LAUNCHED();
			k_scatter<<<chunks, CHUNK, 0, s>>>( A, cur, num, idx_in, idx_out ); LAUNCHED();
			k_prepare_level<<<1, 1024, 0, s>>>( A, next ); LAUNCHED();
			CUDA_TRY( cudaMemcpyAsync( h_ctr, A.ctr, sizeof( Counters ), cudaMemcpyDeviceToHost, s ) );
			CUDA_TRY( cudaStreamSynchronize( s ) );
			num = h_ctr->next_large, chunks = h_ctr->total_chunks;
			if (num > max_large) { tbvh_set_error( "build: level list overflow (%u > %zu)", num, max_large ); return TBVH_E_LIMIT; }
			if (num)
			{
				k_bins_init<<<(num * BIN_STRIDE + 255) / 256, 256, 0, s>>>( A.bins, num * BIN_STRIDE ); LAUNCHED();
				CUDA_TRY( cudaMemsetAsync( &A.ctr->next_large, 0, 4, s ) );
			}
			level++;
			if (level > 4096) { tbvh_set_error( "build: runaway level count" ); return TBVH_E_LIMIT; }
		}
		CUDA_TRY( cudaMemcpyAsync( h_ctr, A.ctr, sizeof( Counters ), cudaMemcpyDeviceToHost, s ) );
		CUDA_TRY( cudaStreamSynchronize( s ) );
		const uint32_t roots = h_ctr->small_roots;
		if (roots)
		{
			k_build_small<<<(roots + SMALL_WARPS - 1) / SMALL_WARPS, SMALL_WARPS * 32, 0, s>>>( A, roots );
			LAUNCHED();
		}
		CUDA_TRY( cudaMemcpyAsync( h_ctr, A.ctr, sizeof( Counters ), cudaMemcpyDeviceToHost, s ) );
		CUDA_TRY( cudaStreamSynchronize( s ) );
		const uint32_t tmp_count = h_ctr->tmp_nodes;
		if (tmp_count > max_nodes) { tbvh_set_error( "build: node pool overflow" ); return TBVH_E_LIMIT; }
		// relayout into the reference's numbering: cnt -> flags, prefix -> scan, min depth -> pos_bl
		CUDA_TRY( cudaMemsetAsync( A.flags, 0, ((size_t)n + 1) * 4, s ) );
		CUDA_TRY( cudaMemsetAsync( A.pos_bl, 0xff, ((size_t)n + 1) * 4, s ) );
		k_rank_count<<<(tmp_count + 255) / 256, 256, 0, s>>>( A, tmp_count, A.flags, A.pos_bl ); LAUNCHED();
		{ const int r = exclusive_scan( A.flags, A.scan, tile_sum, n, s ); if (r != TBVH_OK) return r; }
		k_relayout<<<(tmp_count + 255) / 256, 256, 0, s>>>( A, tmp_count, A.scan, A.pos_bl, b->d_nodes ); LAUNCHED();
		CUDA_TRY( cudaEventRecord( e1, s ) );
		CUDA_TRY( cudaStreamSynchronize( s ) );
		float ms = 0;
		CUDA_TRY( cudaEventElapsedTime( &ms, e0, e1 ) );
		b->info.build_ms = ms;
		b->info.used_nodes = tmp_count, b->info.idx_count = n, b->info.max_depth = h_ctr->max_depth;
		uint32_t rootw[8];
		CUDA_TRY( cudaMemcpy( rootw, b->d_nodes, 32, cudaMemcpyDeviceToHost ) );
		memcpy( b->info.aabb_min, rootw, 12 ), memcpy( b->info.aabb_max, rootw + 4, 12 );
		b->root_ref = rootw[3], b->root_count = rootw[7];
		b->d_trav = b->d_nodes;
		return b->d_aabbs ? TBVH_OK : make_leaf_tris( b, s ); // a TLAS has no triangles of its own
	};
	rc = body();
	cudaStreamSynchronize( s );
	for (void* p : scratch) cudaFree( p );
	if (h_ctr) cudaFreeHost( h_ctr );
	if (e0) cudaEventDestroy( e0 );
	if (e1) cudaEventDestroy( e1 );
	return rc;
}
